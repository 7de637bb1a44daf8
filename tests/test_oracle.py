"""CPU tests that pin the oracle (no reference goldens exist, SURVEY.md 8c): closed forms vs the reference's
numerical differences, manifold round trips, an independent sparse solve (scipy splu), noise-free recovery of the
ground truth, chi2 monotonicity, the frozen goldens, and the reference's own ISAM/data/sphere400.txt and sphere2500.txt
datasets (committed under tests/golden by tools/make_sphere_golden.py)."""
import json
import os
import sys

import numpy as np
import pytest
import scipy.sparse.linalg as spl

import oracle_api as O
from oracle_api import OracleAPI
from pop_up_slam_b200 import geometry as geo, graphgen as gg

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = json.load(open(os.path.join(HERE, "golden", "oracle_configs_1_2.json")))


def test_standard_rad_and_round_trips():
    lib = O.oracle_lib()
    for t in np.linspace(-20, 20, 401):
        r = lib.orc_standard_rad(float(t))
        assert -np.pi - 1e-12 <= r <= np.pi + 1e-12
        assert abs(np.sin(r) - np.sin(t)) < 1e-9 and abs(np.cos(r) - np.cos(t)) < 1e-9
    rng = np.random.default_rng(0)
    for _ in range(200):
        v = np.concatenate([rng.uniform(-5, 5, 3), [rng.uniform(-3.1, 3.1), rng.uniform(-1.4, 1.4), rng.uniform(-3.1, 3.1)]])
        p = O.pose_from_xyzypr(v)
        assert np.allclose(O.pose_vector(p), v, atol=1e-12)                 # euler -> quat -> euler
        T = O.pose_wTo(p)
        assert np.allclose(T @ O.pose_oTw(p), np.eye(4), atol=1e-12)
        q = O.pose_from_mat4(T)
        assert np.allclose(O.pose_wTo(q), T, atol=1e-12)                    # matrix -> quat -> matrix
        d = rng.normal(0, 0.3, 6)
        p2 = O.pose_exmap(p, d)
        assert np.allclose(p2[:3], p[:3] + d[:3])
        rel = O.pose_ominus(p2, p)                                           # right-multiplied rotation vector
        ang = geo.quat_angle(rel[3:], np.array([1.0, 0, 0, 0]))
        assert abs(ang - np.linalg.norm(d[3:])) < 1e-10
        pl = geo.plane_normalize(rng.normal(size=4))
        d3 = rng.normal(0, 0.2, 3)
        pl2 = O.plane_exmap(pl, d3)
        assert abs(np.linalg.norm(pl2) - 1) < 1e-14
        # log(exmap(pl, d), pl) = d : the pose-plane residual is the inverse of the plane update
        assert np.allclose(O.plane_log_error(pl2, pl), d3, atol=1e-10)
        assert np.allclose(O.plane_exmap(pl, np.zeros(3)), pl, atol=1e-15)


def test_plane_transform_is_consistent_with_points():
    rng = np.random.default_rng(1)
    for _ in range(50):
        p = O.pose_from_xyzypr(np.concatenate([rng.uniform(-3, 3, 3), rng.uniform(-1, 1, 3)]))
        T = O.pose_wTo(p)
        pl = geo.plane_normalize(np.append(rng.normal(size=3), rng.uniform(-4, 4)))
        local = O.plane_transform(T, pl)
        back = O.plane_transform(O.pose_oTw(p), local)
        assert geo.plane_distance(back, pl) < 1e-12
        x_local = rng.normal(size=3)
        x_local -= (local[:3] @ x_local + local[3]) / (local[:3] @ local[:3]) * local[:3]   # a point on the local plane
        x_world = T[:3, :3] @ x_local + T[:3, 3]
        assert abs(pl[:3] @ x_world + pl[3]) < 1e-10


@pytest.mark.parametrize("cfg", [1, 2])
def test_numeric_and_analytic_jacobians_agree_on_graphs(cfg):
    g = gg.make_config(cfg, seed=5)
    api = OracleAPI()
    ids = gg.build_interleaved(api, g)
    for fid in list(ids["pp_fids"][::7]) + list(ids["odo_fids"][::5]) + [ids["prior_fid"], ids["ground_fid"]]:
        Hn, rn = api.factor_jacobian(int(fid), 0)
        Ha, ra = api.factor_jacobian(int(fid), 1)
        # (numericalDiff restores the linearisation point through an Euler round trip: rounding-level shift)
        assert np.allclose(rn, ra, atol=1e-9 * max(1, np.abs(ra).max()))
        assert np.abs(Hn - Ha).max() <= 1e-5 * max(1.0, np.abs(Ha).max())   # eps = 1e-4 truncation (SURVEY A.3)


@pytest.mark.parametrize("lam", [0.0, 1e-6, 1e-2])
def test_direct_solve_matches_scipy_splu(lam):
    g = gg.make_config(2, seed=1)
    api = OracleAPI()
    api.set_jacobian_mode(1)
    gg.build_interleaved(api, g)
    A, b = api.normal_equations(lam)
    ref = spl.splu(A.tocsc()).solve(b)
    got = api.solve_step(lam)
    assert np.linalg.norm(got - ref) / np.linalg.norm(ref) < 1e-10
    # ordering re-use gives the same answer
    api.set_reuse_ordering(1)
    assert np.allclose(api.solve_step(lam), got, rtol=1e-12, atol=1e-14)
    assert np.allclose(api.solve_step(lam), got, rtol=1e-12, atol=1e-14)


def test_noise_free_graph_recovers_truth():
    g = gg.make_corridor(seed=3, n_poses=60, n_planes=14, obs_per_pose=6, plane_noise=0.0, odo_noise=(0.0, 0.0), aisle=8.0,
                         radius=1.5, max_iterations=30, sigma_mode="reference")
    # start away from the truth
    rng = np.random.default_rng(0)
    g.poses_init = np.array([O.pose_exmap(p, np.concatenate([rng.normal(0, 0.05, 3), rng.normal(0, 0.02, 3)])) for p in g.poses_truth])
    g.poses_init[0] = g.poses_truth[0]
    g.pp_sqrtinf[:] = gg.diag_ut([100] * 3)
    g.odo_sqrtinf[:] = gg.diag_ut([100] * 6)
    g.prior_sqrtinf = gg.diag_ut([100] * 6)
    for jac in (0, 1):
        api = OracleAPI()
        api.set_jacobian_mode(jac)
        ids = gg.build_bulk(api, g)
        gg.configure(api, g, epsilon2=1e-9, epsilon_abs=1e-18, epsilon_rel=1e-12)
        api.batch_optimize()
        tr = api.trace()
        acc = tr["accepted"] == 1
        assert np.all(tr["chi2_new"][acc] < tr["chi2_before"][acc])          # accepted steps decrease chi2
        assert api.chi2() < 1e-10
        P = api.get_poses(ids["pose_ids"])
        assert np.abs(P[:, :3] - g.poses_truth[:, :3]).max() < 1e-5
        L = api.get_planes(ids["plane_ids"])
        assert max(geo.plane_distance(a, b) for a, b in zip(L, g.planes_truth)) < 1e-5


@pytest.mark.parametrize("key", sorted(GOLDEN))
def test_oracle_matches_frozen_goldens(key):
    gold = GOLDEN[key]
    g = gg.make_config(gold["config"], seed=gold["seed"])
    api = OracleAPI()
    api.set_jacobian_mode(0)
    ids = gg.build_interleaved(api, g)
    gg.configure(api, g)
    assert ids["pose_ids"].tolist() == gold["pose_ids"] and ids["plane_ids"].tolist() == gold["plane_ids"]
    assert [api.node_start(int(i)) for i in list(ids["pose_ids"][:8]) + list(ids["plane_ids"][:8])] == gold["node_starts"]
    assert [api.factor_row(int(f)) for f in ids["pp_fids"][:16]] == gold["factor_rows"]
    assert abs(api.chi2() - gold["chi2_initial"]) <= 1e-9 * gold["chi2_initial"]
    assert api.batch_optimize() == gold["iterations"]
    tr = api.trace()
    assert tr["accepted"].tolist() == gold["accepted"]
    assert np.allclose(tr["chi2_new"], gold["chi2_trace"], rtol=1e-7)
    assert abs(api.chi2() - gold["chi2_final"]) <= 1e-7 * gold["chi2_final"]
    assert np.allclose(api.get_poses(ids["pose_ids"]), np.array(gold["poses"]), atol=1e-7)
    assert np.allclose(api.get_planes(ids["plane_ids"]), np.array(gold["planes"]), atol=1e-7)


def test_huber_cost_is_applied_per_component():
    g = gg.make_config(2, seed=0, n_poses=30, n_planes=8)
    api = OracleAPI()
    ids = gg.build_bulk(api, g)
    fid = int(ids["pp_fids"][3])
    r0 = api.factor_error(fid)
    api.set_robust(1, 0.5)
    r1 = api.factor_error(fid)
    exp = np.where(np.abs(r0) < 0.5, r0, np.sign(r0) * np.sqrt(2 * 0.5 * np.abs(r0) - 0.25))
    assert np.allclose(r1, exp, atol=1e-14)


def test_sphere400_reference_dataset():
    """The reference's own odometry-only dataset through the Loader's conventions (ISAM/isam/Loader.cpp:316-365):
    EDGE3 i j x y z roll pitch yaw + 21 sqrt-information entries; prior sqrt-information 100*I on pose 0.  The edges come
    from tests/golden/sphere400.json, which holds them already in those conventions (measurement x y z yaw pitch roll, the
    rotational block of the sqrt-information re-ordered to yaw, pitch, roll as Loader.cpp:333-345 does)."""
    fx = json.load(open(os.path.join(HERE, "golden", "sphere400.json")))
    api = OracleAPI()
    api.set_jacobian_mode(1)
    api.set_properties(**dict(gg.PPS_PROPERTIES, method=0, max_iterations=10))
    ids = {}
    n_edges = 0
    for e in fx["edges"]:
        i, j = int(e[0]), int(e[1])
        meas, sqrtinf = np.array(e[2:8]), np.array(e[8:29])
        if not ids:
            ids[min(i, j)] = api.add_pose(None)
            api.add_pose_prior(ids[min(i, j)], np.zeros(6), gg.diag_ut([100.0] * 6))
        assert i < j
        for k in (i, j):
            if k not in ids:
                ids[k] = api.add_pose(None)
        api.add_odometry(ids[i], ids[j], meas, sqrtinf)
        n_edges += 1
    assert len(ids) == 400 and n_edges == 779
    c0 = api.chi2()
    api.batch_optimize()
    c1 = api.chi2()
    assert c1 < 1e-2 * c0
    assert c1 / (6 * n_edges + 6 - 6 * 400) < 5.0      # normalised chi2 of a converged sphere400 is O(1)


def test_measurement_refresh_and_projection_geometry():
    """the oracle's restatement of Mapper_mono::update_plane_measurement / reproj_to_newplane (Mapping.cpp:590-632)
    against independent numpy geometry: the ground row of a frame is normalize(wTo^T (0,0,-1,0)); a wall row contains
    the two ground points its segment pops up from; projected points lie on the plane and move along its normal."""
    g = gg.make_config(2, seed=3, n_poses=30, n_planes=10)
    o = OracleAPI()
    ids = gg.build_bulk(o, g)
    rng = np.random.default_rng(2)
    K = np.array([[535.4, 0, 320.1], [0, 539.2, 247.6], [0, 0, 1.0]])
    invK = np.linalg.inv(K)
    order = np.argsort(g.pp_pose, kind="stable")
    e0, e1 = int(order[0]), int(order[1])          # two factors of pose 0
    f = int(g.pp_pose[e0])
    segs = np.array([[100.0, 400.0, 500.0, 380.0]], dtype=np.float32)
    new = o.refresh_plane_measurements([ids["pose_ids"][f]], [0, 1], segs, invK, ids["pp_fids"][[e0, e1]], [0, 0], [0, 1])
    T = geo.pose7_to_T(o.get_pose(int(ids["pose_ids"][f])))
    ground = T.T @ np.array([0, 0, -1.0, 0])
    assert np.allclose(new[0], ground / np.linalg.norm(ground), atol=1e-6)
    # wall plane (sensor frame) contains the back-projected ground points of both segment ends
    gs = ground
    for px, py in ((100.0, 400.0), (500.0, 380.0)):
        ray = invK @ np.array([px, py, 1.0])
        P = -gs[3] / (gs[:3] @ ray) * ray
        assert abs(new[1][:3] @ P + new[1][3]) <= 1e-4
    assert np.allclose(o.get_measurement(int(ids["pp_fids"][e1])), new[1])
    pts = rng.uniform(-3, 3, size=(50, 3)).astype(np.float32)
    pl = ids["plane_ids"][np.arange(50) % g.n_planes]
    pr = o.project_to_planes(pl, pts)
    for i in range(50):
        v = o.get_plane(int(pl[i]))
        n = v[:3] / np.linalg.norm(v[:3])
        assert abs(n @ pr[i] + v[3] / np.linalg.norm(v[:3])) <= 1e-5
        assert np.linalg.norm(np.cross(pr[i] - pts[i], n)) <= 1e-5


SPHERE2500 = os.path.join(HERE, "golden", "sphere2500.txt.xz")
SPHERE2500_GT = os.path.join(HERE, "golden", "sphere2500_groundtruth.txt.xz")


def test_sphere2500_ground_truth_pins_the_pose_graph_path():
    """Known answers held by the reference itself (ISAM/data/sphere2500.txt and data/groundtruth/, committed whole under
    tests/golden):
    (1) chaining the ground-truth file's sequential edges through the factors' initialize() path (oplus) must make
        ALL of its 4 949 edges consistent, the 2 450 loop closures included: chi2 of the ground-truth graph ~ 0
        (6-digit text rounding).  Any wrong convention in Pose3d (Euler order, oplus / ominus direction, the Loader's
        roll-pitch-yaw swap) breaks this.
    (2) Gauss-Newton on the noisy dataset must reach a normalised chi2 of 1 (the noise was drawn from the stated
        sqrt-information) and land within 2 % of the sphere radius of the ground-truth trajectory."""
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from make_sphere_golden import build, load_edge3
    gt, noisy = load_edge3(SPHERE2500_GT), load_edge3(SPHERE2500)
    assert len(gt) == len(noisy) == 4949
    a = OracleAPI()
    a.set_jacobian_mode(1)
    ida = build(a, gt)
    assert len(ida) == 2500
    assert a.chi2() < 1e-2                                    # 29 700 weighted residual rows, weights 10 / 100 / 25
    P_gt = a.get_poses(np.array([ida[k] for k in sorted(ida)]))
    b = OracleAPI()
    b.set_jacobian_mode(1)
    b.set_properties(**dict(gg.PPS_PROPERTIES, method=0, max_iterations=20, epsilon_abs=1e-6, epsilon_rel=1e-8))
    idb = build(b, noisy)
    c0 = b.chi2()
    b.batch_optimize()
    c1 = b.chi2()
    dof = 6 * len(noisy) + 6 - 6 * len(idb)
    assert c1 < 1e-3 * c0
    assert 0.95 < c1 / dof < 1.05
    P = b.get_poses(np.array([idb[k] for k in sorted(idb)]))
    err = np.linalg.norm(P[:, :3] - P_gt[:, :3], axis=1)
    assert err.mean() < 0.02 * np.abs(P_gt[:, :3]).max()


def test_oracle_matches_sphere400_fixture():
    """the committed fixture of the reference's sphere400 dataset (tools/make_sphere_golden.py): the oracle still
    produces the frozen Gauss-Newton result (numeric Jacobians as upstream)."""
    import json
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from make_sphere_golden import build
    fx = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "sphere400.json")))
    edges = [(int(e[0]), int(e[1]), e[2:8], e[8:29]) for e in fx["edges"]]
    api = OracleAPI()
    api.set_jacobian_mode(0)
    api.set_properties(**fx["properties"])
    ids = build(api, edges)
    assert abs(api.chi2() - fx["oracle"]["chi2_initial"]) <= 1e-9 * fx["oracle"]["chi2_initial"]
    assert api.batch_optimize() == fx["oracle"]["iterations"]
    assert abs(api.chi2() - fx["oracle"]["chi2_final"]) <= 1e-8 * fx["oracle"]["chi2_final"]
    P = api.get_poses(np.array([ids[k] for k in fx["oracle"]["pose_index"]]))
    assert np.abs(P - np.array(fx["oracle"]["poses"])).max() <= 1e-8
