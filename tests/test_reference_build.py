"""CPU tests against oracle/_ref: the UNMODIFIED reference sources of the hot path (isam::Slam + Optimizer + Cholesky +
numericalDiff, slam3d.h, pop_planar_slam/src/isam_plane3d.{h,cpp}) compiled against the API shims of oracle/ref_shim.

They pin (a) the oracle restatement (oracle/) and (b) the product's host/device math header (csrc/pus_math.cuh compiled for
the host) to what the reference's own code computes: value types and exmaps, every factor's error() and numericalDiff
Jacobian, and whole Levenberg-Marquardt / Gauss-Newton / update() runs including the accept / reject sequence.

The reference side of every comparison, for every case, is stored in tests/golden/reference_build_*.npz (written by
tools/make_ref_build_golden.py, which runs the same seeded inputs through oracle/_ref), so the tests need neither the
reference checkout nor the _ref library at run time."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle_api as O
from oracle_api import OracleAPI
from pop_up_slam_b200 import geometry as geo, graphgen as gg
from pop_up_slam_b200.capi import _dp

HERE = os.path.dirname(os.path.abspath(__file__))
GOLDEN = [os.path.join(HERE, "golden", "reference_build_%s.npz" % part) for part in ("values", "factors", "runs")]
_G = None


def gold(key):
    global _G
    if _G is None:
        _G = {}
        for path in GOLDEN:
            with np.load(path) as z:
                _G.update(z)
    return _G[key]


def rand_pose(rng, scale=5.0):
    v = np.concatenate([rng.uniform(-scale, scale, 3), [rng.uniform(-3, 3), rng.uniform(-1.2, 1.2), rng.uniform(-3, 3)]])
    return O.pose_from_xyzypr(v)


def rand_plane(rng):
    n = rng.normal(size=3)
    n /= np.linalg.norm(n)
    return geo.plane_normalize(np.append(n, -rng.uniform(0.5, 8.0)))


def ut(rng, n):
    A = np.triu(rng.uniform(0.5, 2.0, size=(n, n)))
    A[np.diag_indices(n)] = rng.uniform(1.0, 30.0, n)
    return A[np.triu_indices(n)]


def value_type_inputs():
    """the 500 random cases of the value-type test: (v = x y z yaw pitch roll, pose tangent d, pose q, plane, plane tangent)"""
    rng = np.random.default_rng(0)
    for _ in range(500):
        v = np.concatenate([rng.uniform(-5, 5, 3), [rng.uniform(-3.1, 3.1), rng.uniform(-1.4, 1.4), rng.uniform(-3.1, 3.1)]])
        d = rng.normal(0, 0.3, 6) * (1e-5 if rng.random() < 0.2 else 1.0)      # also the small-angle branch
        q = rand_pose(rng)
        pl = rand_plane(rng)
        d3 = rng.normal(0, 0.2, 3) * (1e-6 if rng.random() < 0.2 else 1.0)
        yield v, d, q, pl, d3


def test_value_types_and_exmaps_match_the_reference_classes():
    """Pose3d / Rot3d / Point3d (Pose3d.h:131-235, Rot3d.h:100-136,229-233) and Plane3d (isam_plane3d.h:27-193)."""
    for t, r in zip(np.linspace(-20, 20, 201), gold("values/standard_rad")):
        assert r == O.oracle_lib().orc_standard_rad(float(t))
    n = 0
    for k, (v, d, q, pl, d3) in enumerate(value_type_inputs()):
        p = gold("values/pose")[k]
        assert np.allclose(p, O.pose_from_xyzypr(v), atol=1e-15)
        assert np.allclose(gold("values/vector")[k], O.pose_vector(p), atol=1e-13)
        assert np.allclose(gold("values/exmap")[k], O.pose_exmap(p, d), atol=1e-14)
        for name, fo in (("oplus", O.pose_oplus), ("ominus", O.pose_ominus)):
            a, b = gold("values/" + name)[k], fo(p, q)
            # Pose3d(Matrix4d) keeps Eigen's raw quaternion upstream; the oracle renormalises it (DESIGN.md section 3): same
            # rotation, |q| within rounding of 1
            assert np.allclose(a[:3], b[:3], atol=1e-12)
            assert min(np.abs(a[3:] - b[3:]).max(), np.abs(a[3:] + b[3:]).max()) < 1e-12
        assert np.allclose(gold("values/wTo")[k], O.pose_wTo(p), atol=1e-14)
        assert np.allclose(gold("values/oTw")[k], O.pose_oTw(p), atol=1e-13)
        T = O.pose_wTo(q)
        a, b = gold("values/from_mat4")[k], O.pose_from_mat4(T)
        assert np.allclose(a[:3], b[:3], atol=1e-13) and min(np.abs(a[3:] - b[3:]).max(), np.abs(a[3:] + b[3:]).max()) < 1e-12
        assert np.allclose(gold("values/plane_exmap")[k], O.plane_exmap(pl, d3), atol=1e-15)          # exmap_3dof :101-127, boost sinc_pi
        assert np.allclose(gold("values/plane_transform")[k], O.plane_transform(T, pl), atol=1e-14)  # transform_to / _from :180-188
        n += 1
    assert n == len(gold("values/pose")) == 500


FACTOR_KINDS = ("pose_plane", "odometry", "pose_prior", "plane_prior")


def _random_factor_graph(api, rng, n=120, robust=None):
    """poses, planes and one factor of every kind per pose (random sqrt-information incl. off-diagonal terms)."""
    poses = [rand_pose(rng) for _ in range(n)]
    planes = [rand_plane(rng) for _ in range(n)]
    pid = api.add_poses(np.array(poses))
    lid = api.add_planes(np.array(planes))
    fids = []
    for i in range(n):
        T = O.pose_wTo(poses[i])
        meas = O.plane_exmap(O.plane_transform(T, planes[i]), rng.normal(0, 0.3, 3))
        fids.append(("pose_plane", api.add_pose_plane(pid[i], lid[i], meas, ut(rng, 3))))
        j = (i + 1) % n
        m = O.pose_vector(O.pose_ominus(poses[j], poses[i])) + rng.normal(0, 0.05, 6)
        fids.append(("odometry", api.add_odometry(pid[i], pid[j], m, ut(rng, 6))))
        fids.append(("pose_prior", api.add_pose_prior(pid[i], O.pose_vector(poses[i]) + rng.normal(0, 0.05, 6), ut(rng, 6))))
        fids.append(("plane_prior", api.add_plane_prior(lid[i], O.plane_exmap(planes[i], rng.normal(0, 0.2, 3)), ut(rng, 3))))
    if robust:
        api.set_robust(*robust)
    return fids


def robust_tag(robust):
    return "none" if robust is None else "kind%d_b%g" % robust


@pytest.mark.parametrize("robust", [None, (1, 0.8), (2, 0.5)])
def test_factor_errors_and_numerical_jacobians_match_the_reference(robust):
    """Factor::error (Factor.h:67-77: sqrtinf * basic_error, per-component robust cost) and Factor::jacobian ->
    numericalDiff (numericalDiff.cpp:41-87) of Pose3d_Plane3d_Factor (isam_plane3d.h:271-304), Pose3d_Pose3d_Factor /
    Pose3d_Factor (slam3d.h:82-88,174-191) and Plane3d_Factor (isam_plane3d.h:450-473): 480 random factors.
    oracle numeric mode == reference to rounding; oracle closed forms == reference to its truncation error."""
    orc = OracleAPI()
    fo = _random_factor_graph(orc, np.random.default_rng(5), robust=robust)
    key = "factors/" + robust_tag(robust)
    worst = dict(err=0.0, num=0.0, ana=0.0)
    n = 0
    for k, (kind, b) in enumerate(fo):
        i = k // len(FACTOR_KINDS)
        er, Jr, rr = (gold("%s/%s/%s" % (key, kind, f))[i] for f in ("error", "jacobian", "residual"))
        eo = orc.factor_error(b)
        assert er.shape == eo.shape
        worst["err"] = max(worst["err"], np.abs(er - eo).max() / max(1.0, np.abs(eo).max()))
        Jn, rn = orc.factor_jacobian(b, 0)
        Ja, _ = orc.factor_jacobian(b, 1)
        assert Jr.shape == Jn.shape == Ja.shape, kind
        scale = max(1.0, np.abs(Jr).max())
        worst["num"] = max(worst["num"], np.abs(Jr - Jn).max() / scale)
        worst["ana"] = max(worst["ana"], np.abs(Jr - Ja).max() / scale)
        assert np.allclose(rr, rn, atol=1e-11 * max(1.0, np.abs(rn).max()))
        n += 1
    assert n == sum(len(gold("%s/%s/error" % (key, kind))) for kind in FACTOR_KINDS) == 480
    assert worst["err"] < 1e-12, worst
    assert worst["num"] < 1e-8, worst        # same central differences: only rounding amplified by 1 / (2 eps)
    # closed forms vs the reference's eps = 1e-4 central differences: its truncation error (SURVEY appendix A.3); with a
    # robust cost the differenced function sign * sqrt(rho) is only C1 at |r| = b and strongly curved beyond it for the
    # large sqrt-information values drawn here, so the reference's own differences are cruder there
    assert worst["ana"] < (2e-5 if robust is None else 5e-3), worst


@pytest.fixture(scope="module")
def hm():
    src = os.path.join(HERE, "hostmath_shim.cpp")
    out = os.path.join(HERE, "libhostmath.so")
    hdr = os.path.join(HERE, "..", "pop_up_slam_b200", "csrc", "pus_math.cuh")
    if not os.path.exists(out) or max(os.path.getmtime(src), os.path.getmtime(hdr)) > os.path.getmtime(out):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", out, src])
    lib = C.CDLL(out)
    P = C.POINTER(C.c_double)
    lib.hm_pose_plane_linearize.argtypes = [P, P, P, P, C.c_int, C.c_double, P, P, P]
    lib.hm_pose_factor_linearize.argtypes = [P, P, P, P, C.c_int, C.c_double, P, P, P]
    lib.hm_pose_plane_numeric.argtypes = [P, P, P, P, C.c_int, C.c_double, P, P, P]
    lib.hm_pose_factor_numeric.argtypes = [P, P, P, P, C.c_int, C.c_double, P, P, P]
    return lib


def math_header_cases(seed, n, with_prior=False):
    """random poses / planes and, per pose i, a pose-plane factor (meas, si), an odometry factor to pose i+1 (m, si6) and,
    with_prior, a pose prior measurement (sharing si6)"""
    rng = np.random.default_rng(seed)
    poses = [rand_pose(rng) for _ in range(n)]
    planes = [rand_plane(rng) for _ in range(n)]
    cases = []
    for i in range(n):
        meas = O.plane_exmap(O.plane_transform(O.pose_wTo(poses[i]), planes[i]), rng.normal(0, 0.3, 3))
        si = ut(rng, 3)
        j = (i + 1) % n
        m = O.pose_vector(O.pose_ominus(poses[j], poses[i])) + rng.normal(0, 0.05, 6)
        si6 = ut(rng, 6)
        prior = O.pose_vector(poses[i]) + rng.normal(0, 0.05, 6) if with_prior else None
        cases.append((meas, si, m, si6, prior))
    return poses, planes, cases


@pytest.mark.parametrize("robust", [0, 1])
def test_product_math_header_matches_the_reference(hm, robust):
    """pus_math.cuh (the __host__ __device__ header the kernels run, compiled for the host) against the reference's
    error() and numericalDiff Jacobians directly: residuals to rounding, closed-form Jacobians to the reference's
    eps = 1e-4 truncation error (2e-5 relative without a robust cost; with Huber the reference's own central
    differences are cruder around the C1 point |r| = b, see the previous test)."""
    poses, planes, cases = math_header_cases(11, 150)
    key = "header/robust%d/" % robust
    n = len(poses)
    worst_r = worst_j = 0.0
    for i, (meas, si, m, si6, _) in enumerate(cases):
        Jr, rr = gold(key + "pose_plane_jacobian")[i], gold(key + "pose_plane_residual")[i]
        r, Jp, Jl = np.zeros(3), np.zeros(18), np.zeros(9)
        hm.hm_pose_plane_linearize(_dp(poses[i]), _dp(planes[i]), _dp(np.ascontiguousarray(meas)), _dp(si), robust, 0.8, _dp(r), _dp(Jp), _dp(Jl))
        J = np.hstack([Jp.reshape(3, 6), Jl.reshape(3, 3)])
        worst_r = max(worst_r, np.abs(r - rr).max() / max(1.0, np.abs(rr).max()))
        worst_j = max(worst_j, np.abs(J - Jr).max() / max(1.0, np.abs(Jr).max()))
        j = (i + 1) % n
        Jr, rr = gold(key + "odometry_jacobian")[i], gold(key + "odometry_residual")[i]
        r6, J1, J2 = np.zeros(6), np.zeros(36), np.zeros(36)
        hm.hm_pose_factor_linearize(_dp(poses[i]), _dp(poses[j]), _dp(np.ascontiguousarray(m)), _dp(si6), robust, 0.8, _dp(r6), _dp(J1), _dp(J2))
        J = np.hstack([J1.reshape(6, 6), J2.reshape(6, 6)])
        worst_r = max(worst_r, np.abs(r6 - rr).max() / max(1.0, np.abs(rr).max()))
        worst_j = max(worst_j, np.abs(J - Jr).max() / max(1.0, np.abs(Jr).max()))
    assert worst_r < 1e-12, worst_r
    assert worst_j < (2e-2 if robust else 2e-5), worst_j


@pytest.mark.parametrize("robust", [0, 1])
def test_product_reference_jacobian_mode_matches_numericaldiff(hm, robust):
    """pus_set_jacobian_mode(h, 1): pose_plane_numeric / pose_factor_numeric of pus_math.cuh (what the kernels run in that
    mode) reproduce the reference's numericalDiff blocks (numericalDiff.cpp:41-87) to the rounding of the differences."""
    poses, planes, cases = math_header_cases(12, 100, with_prior=True)
    key = "numeric/robust%d/" % robust
    n = len(poses)
    worst_r = worst_j = 0.0
    for i, (meas, si, m, si6, _) in enumerate(cases):
        Jr, rr = gold(key + "pose_plane_jacobian")[i], gold(key + "pose_plane_residual")[i]
        r, Jp, Jl = np.zeros(3), np.zeros(18), np.zeros(9)
        hm.hm_pose_plane_numeric(_dp(poses[i]), _dp(planes[i]), _dp(np.ascontiguousarray(meas)), _dp(si), robust, 0.8, _dp(r), _dp(Jp), _dp(Jl))
        J = np.hstack([Jp.reshape(3, 6), Jl.reshape(3, 3)])
        worst_r = max(worst_r, np.abs(r - rr).max() / max(1.0, np.abs(rr).max()))
        worst_j = max(worst_j, np.abs(J - Jr).max() / max(1.0, np.abs(Jr).max()))
        j = (i + 1) % n
        Jr, rr = gold(key + "odometry_jacobian")[i], gold(key + "odometry_residual")[i]
        r6, J1, J2 = np.zeros(6), np.zeros(36), np.zeros(36)
        hm.hm_pose_factor_numeric(_dp(poses[i]), _dp(poses[j]), _dp(np.ascontiguousarray(m)), _dp(si6), robust, 0.8, _dp(r6), _dp(J1), _dp(J2))
        J = np.hstack([J1.reshape(6, 6), J2.reshape(6, 6)])
        worst_r = max(worst_r, np.abs(r6 - rr).max() / max(1.0, np.abs(rr).max()))
        worst_j = max(worst_j, np.abs(J - Jr).max() / max(1.0, np.abs(Jr).max()))
        # the pose prior with the measurement as the reference stores it
        Jr, rr, mm = (gold(key + f)[i] for f in ("pose_prior_jacobian", "pose_prior_residual", "pose_prior_measurement"))
        hm.hm_pose_factor_numeric(_dp(poses[i]), None, _dp(np.ascontiguousarray(mm)), _dp(si6), robust, 0.8, _dp(r6), _dp(J1), _dp(J2))
        worst_r = max(worst_r, np.abs(r6 - rr).max() / max(1.0, np.abs(rr).max()))
        worst_j = max(worst_j, np.abs(J1.reshape(6, 6) - Jr).max() / max(1.0, np.abs(Jr).max()))
    assert worst_r < 1e-12, worst_r
    assert worst_j < 1e-8, worst_j


def _compare_estimates(api, ids, key, tol):
    """estimates of `api` against the reference's stored under `key`"""
    Po, Lo = api.get_poses(ids["pose_ids"]), api.get_planes(ids["plane_ids"])
    Pr, Lr = gold(key + "/poses"), gold(key + "/planes")
    assert Po.shape == Pr.shape and Lo.shape == Lr.shape
    assert np.abs(Pr[:, :3] - Po[:, :3]).max() < tol
    sq = np.sign(np.sum(Pr[:, 3:] * Po[:, 3:], axis=1))[:, None]
    assert np.abs(Pr[:, 3:] * sq - Po[:, 3:]).max() < tol
    assert np.abs(Lr - Lo).max() < tol


def lm_key(cfg, kw, builder):
    return "lm/config%d%s_%s" % (cfg, "".join("_%s%s" % kv for kv in sorted(kw.items())), builder)


BUILDERS = {"interleaved": gg.build_interleaved, "bulk": gg.build_bulk}


@pytest.mark.parametrize("cfg,kw,builder", [(1, {}, "interleaved"), (2, {}, "interleaved"), (2, dict(seed=3), "bulk"),
                                            (3, dict(n_poses=600, n_planes=60), "bulk")])
def test_levenberg_marquardt_runs_match_the_reference_optimiser(cfg, kw, builder):
    """Whole batch_optimization() runs (Slam.cpp:198-210 -> Optimizer.cpp:371-467 -> Cholesky.cpp:68-147) of the reference
    code against the oracle in its reference mode (numeric Jacobians): the insertion order of Mapper_mono::processFrame
    with the factors' initialize() paths (configs 1, 2), and a Huber corridor with outliers whose 20 trial steps include
    rejected ones (config 3, reduced).  Same iteration count and accept / reject sequence, chi2 to 1e-10, estimates 1e-8."""
    key = lm_key(cfg, kw, builder)
    kw = dict(kw)
    g = gg.make_config(cfg, seed=kw.pop("seed", 0), **kw)
    orc = OracleAPI()
    orc.set_jacobian_mode(0)
    io = BUILDERS[builder](orc, g)
    gg.configure(orc, g)
    assert abs(gold(key + "/chi2_initial") - orc.chi2()) <= 1e-11 * orc.chi2()
    assert orc.batch_optimize() == gold(key + "/iterations")
    to = orc.trace()
    assert np.array_equal(gold(key + "/accepted"), to["accepted"])
    assert np.allclose(gold(key + "/lam"), to["lam"], rtol=1e-12)
    acc = gold(key + "/accepted") == 1
    assert np.allclose(gold(key + "/chi2_new")[acc], to["chi2_new"][acc], rtol=1e-10)
    assert abs(gold(key + "/chi2") - orc.chi2()) <= 1e-10 * orc.chi2()
    _compare_estimates(orc, io, key, 1e-8)
    # graph bookkeeping (G1): column offsets of every node as Slam::update_starts assigns them
    nodes = list(io["pose_ids"])[:50] + list(io["plane_ids"])[:20]
    assert [orc.node_start(b) for b in nodes] == gold(key + "/node_start").tolist()
    assert (orc.num_nodes(), orc.num_factors()) == tuple(gold(key + "/num_nodes_factors"))


def test_gauss_newton_update_and_graph_edits_match_the_reference():
    """Optimizer::gauss_newton (Optimizer.cpp:286-366), Slam::update with mod_batch = 1 (Slam.cpp:157-196 ->
    Optimizer::relinearize :114-185), and remove_factor / remove_node + re-solve (Mapping.cpp:659-700)."""
    g = gg.make_config(2, seed=1, n_poses=150, n_planes=30)
    orc = OracleAPI()
    orc.set_jacobian_mode(0)
    io = gg.build_bulk(orc, g)
    gg.configure(orc, g, method=0, max_iterations=10)
    assert abs(gold("gn/chi2_initial") - orc.chi2()) <= 1e-11 * orc.chi2()
    assert orc.batch_optimize() == gold("gn/iterations")
    assert abs(gold("gn/chi2") - orc.chi2()) <= 1e-9 * orc.chi2()
    _compare_estimates(orc, io, "gn", 1e-8)
    # update(): one relinearise + Gauss-Newton step per call
    orc = OracleAPI()
    orc.set_jacobian_mode(0)
    io = gg.build_bulk(orc, g)
    gg.configure(orc, g, mod_batch=1)
    orc.update()
    orc.update()
    assert abs(gold("update/chi2") - orc.chi2()) <= 1e-9 * orc.chi2()
    _compare_estimates(orc, io, "update", 1e-8)
    # loop-closure style edits: drop some factors and one plane (with its factors), solve again
    for f in io["pp_fids"][5:40:7]:
        orc.remove_factor(int(f))
    orc.remove_node(int(io["plane_ids"][7]))
    gg.configure(orc, g)
    orc.batch_optimize()
    assert (orc.num_nodes(), orc.num_factors()) == tuple(gold("edits/num_nodes_factors"))
    assert abs(gold("edits/chi2") - orc.chi2()) <= 1e-9 * orc.chi2()
    keep = [i for i in range(len(io["plane_ids"])) if i != 7]
    assert np.abs(gold("edits/planes") - orc.get_planes(io["plane_ids"][keep])).max() < 1e-8


def build_factor2_graph(api, g):
    """config-2 graph whose wall observations are Pose3d_Plane3d_Factor2 (measured plane re-popped from two ground-edge rays)"""
    pose_ids, plane_ids = api.add_poses(g.poses_init), api.add_planes(g.planes_init)
    api.add_pose_prior(pose_ids[g.prior_pose], g.prior_meas, g.prior_sqrtinf)
    api.add_odometry_bulk(pose_ids[g.odo_i], pose_ids[g.odo_j], g.odo_meas, g.odo_sqrtinf)
    api.add_plane_prior(plane_ids[g.ground_plane], g.ground_meas, g.ground_sqrtinf)
    n2 = 0
    for e in range(g.n_pose_plane):
        p, k = int(g.pp_pose[e]), int(g.pp_plane[e])
        rays = gg.rays_from_measurement(geo.pose7_to_T(g.poses_truth[p]), g.pp_meas[e])
        ok = k != g.ground_plane and abs(rays[2]) > 0.05 and abs(rays[5]) > 0.05   # (a ray is a direction: any non-zero scale gives the same ground hit)
        if ok:   # rays as precompute_edge_ray forms them from float32 pixels: (x, y, 1), float32-representable
            rays = np.concatenate([rays[:3] / rays[2], rays[3:] / rays[5]])
            rays = rays.astype(np.float32).astype(np.float64)
            api.add_pose_plane2(pose_ids[p], plane_ids[k], g.pp_meas[e], rays, g.pp_sqrtinf[e])
            n2 += 1
        else:
            api.add_pose_plane(pose_ids[p], plane_ids[k], g.pp_meas[e], g.pp_sqrtinf[e])
    assert n2 > 100
    return dict(pose_ids=pose_ids, plane_ids=plane_ids)


def test_pose_plane_factor2_matches_the_reference():
    """Pose3d_Plane3d_Factor2 (isam_plane3d.h:314-424): the measured plane is re-popped from two precomputed ground-edge
    rays with the current pose (get_wall_plane_equation, isam_plane3d.cpp:20-55) inside every error evaluation."""
    g = gg.make_config(2, seed=6, n_poses=60, n_planes=20)
    orc = OracleAPI()
    orc.set_jacobian_mode(0)
    io = build_factor2_graph(orc, g)
    gg.configure(orc, g)
    c0o = orc.chi2()
    assert abs(gold("factor2/chi2_initial") - c0o) <= 1e-10 * c0o
    assert orc.batch_optimize() == gold("factor2/iterations")
    assert np.array_equal(gold("factor2/accepted"), orc.trace()["accepted"])
    assert abs(gold("factor2/chi2") - orc.chi2()) <= 1e-9 * orc.chi2()
    _compare_estimates(orc, io, "factor2", 1e-7)


def popup_inputs():
    """40 camera frames (looking forward and slightly down) with 6 random ground segments each: (invK, Ts, segs, ns)"""
    rng = np.random.default_rng(2)
    K = np.array([[535.4, 0, 320.1], [0, 539.2, 247.6], [0, 0, 1.0]])
    invK = np.linalg.inv(K)
    nf, ns = 40, 6
    Ts, segs = [], []
    for _ in range(nf):
        v = np.array([rng.uniform(-3, 3), rng.uniform(-3, 3), rng.uniform(0.8, 1.6), rng.uniform(-3, 3), 0.0, 0.0])
        # camera looking forward and slightly down: x right, y down, z forward in the sensor frame
        Rw = geo.pose7_to_T(O.pose_from_xyzypr(v))[:3, :3] @ np.array([[0, 0, 1.0], [-1, 0, 0], [0, -1, 0]]) @ \
            geo.pose7_to_T(O.pose_from_xyzypr(np.array([0, 0, 0, 0, 0, rng.uniform(0.1, 0.4)])))[:3, :3]
        T = np.eye(4); T[:3, :3] = Rw; T[:3, 3] = v[:3]
        Ts.append(T)
        segs.append(np.stack([rng.uniform(20, 620, ns), rng.uniform(330, 470, ns), rng.uniform(20, 620, ns), rng.uniform(330, 470, ns)], axis=1))
    return invK, np.array(Ts), np.array(segs).reshape(-1, 4), ns


def test_popup_fit_arithmetic_against_the_reference_double_copy():
    """P1: the wall-plane arithmetic of popup_plane::update_plane_equation_from_seg (PUW/libs/popup_plane.cpp:654-749) --
    ground hit of the two edge rays, wall normal = segment x ground normal, sensor-frame plane -- against the reference's
    own double-precision copy get_wall_plane_equation (PPS/src/isam_plane3d.cpp:20-55; "copied from pop_up_wall").  The
    float32 original cannot be compiled here (its header pulls OpenCV / PCL / ROS / boost.python); the oracle's float32
    restatement must agree with the double copy to float32 rounding, up to the plane's scale."""
    from pop_up_slam_b200.capi import popup_fit_frames
    invK, Ts, segs, ns = popup_inputs()
    nf = len(Ts)
    seg_ptr = np.arange(nf + 1) * ns
    pw, ps, dist, good = popup_fit_frames(O.oracle_lib(), seg_ptr, segs, invK, Ts, prefix="orc_")
    ref_ptr = np.concatenate([[0], np.cumsum(gold("popup/count"))])
    worst = 0.0
    for f in range(nf):
        planes = gold("popup/planes")[ref_ptr[f]:ref_ptr[f + 1]]
        mine = ps[f * (ns + 1) + 1:(f + 1) * (ns + 1)].astype(np.float64)
        for a, b in zip(planes, mine):
            worst = max(worst, np.abs(a / np.linalg.norm(a) - b / np.linalg.norm(b)).max())
    assert ref_ptr[-1] > 0
    assert worst < 2e-4, worst


@pytest.mark.gpu
@pytest.mark.parametrize("cfg,seed", [(1, 5), (2, 7)])
def test_gpu_against_the_reference_library_directly(cfg, seed):
    """The CUDA path and the reference's own optimiser on a graph that is in no other fixture: same iterations / accept
    sequence, chi2 and estimates within BASELINE's 1e-4."""
    from pop_up_slam_b200.capi import GpuGraphAPI
    key = "gpu_direct/config%d_seed%d" % (cfg, seed)
    g = gg.make_config(cfg, seed=seed)
    gpu = GpuGraphAPI()
    ig = gg.build_interleaved(gpu, g)
    gg.configure(gpu, g)
    assert abs(gpu.chi2() - gold(key + "/chi2_initial")) <= 1e-10 * gold(key + "/chi2_initial")
    assert gpu.batch_optimize() == gold(key + "/iterations")
    assert np.array_equal(gpu.trace()["accepted"], gold(key + "/accepted"))
    assert abs(gpu.chi2() - gold(key + "/chi2")) <= 1e-4 * gold(key + "/chi2")
    _compare_estimates(gpu, ig, key, 1e-4)


def _loopclose_scenario(api, g, n_dup=4):
    """A graph in which `n_dup` walls were re-detected as NEW landmarks in the second half of the trajectory (what happens
    before a loop closure), built in processFrame's order; returns the ids and, per duplicate, its factor ids."""
    rng = np.random.default_rng(7)
    n, m = g.n_poses, g.n_planes
    counts = np.bincount(g.pp_plane, minlength=m)
    cand = [k for k in np.argsort(-counts) if k != g.ground_plane][:n_dup]
    pose_ids = api.add_poses(g.poses_init)
    plane_ids = api.add_planes(g.planes_init)
    dup_ids = {int(k): api.add_plane(g.planes_init[k] + 0) for k in cand}
    api.add_pose_prior(pose_ids[g.prior_pose], g.prior_meas, g.prior_sqrtinf)
    api.add_odometry_bulk(pose_ids[g.odo_i], pose_ids[g.odo_j], g.odo_meas, g.odo_sqrtinf)
    api.add_plane_prior(plane_ids[g.ground_plane], g.ground_meas, g.ground_sqrtinf)
    dup_facs = {k: [] for k in dup_ids}
    late = set()     # the later half of each candidate wall's observations go to its duplicate
    for k in dup_ids:
        es = np.nonzero(g.pp_plane == k)[0]
        es = es[np.argsort(g.pp_pose[es], kind="stable")]
        late.update(int(e) for e in es[len(es) // 2:])
    fids = []
    for e in range(g.n_pose_plane):
        p, k = int(g.pp_pose[e]), int(g.pp_plane[e])
        target = dup_ids[k] if e in late else plane_ids[k]
        f = api.add_pose_plane(pose_ids[p], target, g.pp_meas[e], g.pp_sqrtinf[e])
        fids.append(f)
        if e in late:
            dup_facs[k].append((f, e))
    assert all(len(v) > 5 for v in dup_facs.values())
    return dict(pose_ids=pose_ids, plane_ids=plane_ids, dup_ids=dup_ids, dup_facs=dup_facs)


def _loopclose_merge(api, g, ids):
    """Mapper_mono::loopclose_merge (Mapping.cpp:659-700), call for call: for every factor of the duplicate landmark a new
    Pose3d_Plane3d_Factor on the matched landmark with the old measurement and noise is added, then the old one removed;
    afterwards the duplicate plane vertex is removed; processFrame then runs batch_optimization() (loop_success)."""
    for k, dup in ids["dup_ids"].items():
        for f, e in ids["dup_facs"][k]:
            api.add_pose_plane(ids["pose_ids"][int(g.pp_pose[e])], ids["plane_ids"][k], api.get_measurement(f, 4), g.pp_sqrtinf[e])
            api.remove_factor(f)
    for k, dup in ids["dup_ids"].items():
        api.remove_node(dup)
    return api.batch_optimize()


def loopclose_run(api):
    """optimise with duplicated landmarks, merge, optimise again: (ids, iterations before, chi2 before, iterations after)"""
    g = gg.make_config(2, seed=5, n_poses=160, n_planes=30)
    ids = _loopclose_scenario(api, g)
    gg.configure(api, g)
    it0 = api.batch_optimize()
    c0 = api.chi2()
    return ids, it0, c0, _loopclose_merge(api, g, ids)


def test_loopclose_merge_replay_matches_the_reference():
    """SURVEY 8(f).2: the exact edit sequence of Mapper_mono::loopclose_merge replayed on the reference optimiser and on
    the oracle: optimise with duplicated landmarks, merge, optimise again."""
    orc = OracleAPI()
    orc.set_jacobian_mode(0)
    io, b0, c0o, b1 = loopclose_run(orc)
    assert (b0, b1, orc.num_nodes(), orc.num_factors()) == tuple(gold("loopclose/iterations_nodes_factors"))
    c0r, c1r = gold("loopclose/chi2")
    assert abs(c0r - c0o) <= 1e-9 * c0o and abs(c1r - orc.chi2()) <= 1e-9 * orc.chi2()
    _compare_estimates(orc, io, "loopclose", 1e-8)


def test_frame_by_frame_replay_matches_the_reference():
    """The reference's real loop (Mapper_mono::processFrame, Mapping.cpp:464-554): per key-frame one pose + odometry + newly
    seen planes + its pose-plane factors, node values initialised by the factors' own initialize() paths, then Slam::update()
    (batch_optimization() every 5th frame) -- replayed call for call on the reference optimiser and on the oracle."""
    import sys
    sys.path.insert(0, os.path.dirname(HERE))
    from bench import replay_frames
    g = gg.make_config(2, seed=9, n_poses=45, n_planes=12)
    orc = OracleAPI()
    orc.set_jacobian_mode(0)
    gg.configure(orc, g, mod_batch=1)
    replay_frames(orc, g)
    assert (orc.num_nodes(), orc.num_factors()) == tuple(gold("replay/num_nodes_factors"))
    cr, co = float(gold("replay/chi2")), orc.chi2()
    assert abs(cr - co) <= 1e-8 * cr, (cr, co)
    assert gold("replay/node_start").tolist() == [orc.node_start(i) for i in range(orc.num_nodes())]
    # ids are insertion-ordered and identical on both sides: compare every node through its kind (a wrong kind raises)
    is_plane, values = gold("replay/is_plane"), gold("replay/values")
    for nid in range(orc.num_nodes()):
        if is_plane[nid]:
            a, b = values[nid, :4], orc.get_plane(nid)
            if np.dot(a, b) < 0:
                b = -b
        else:
            a, b = values[nid], orc.get_pose(nid)
        assert np.abs(np.asarray(a) - np.asarray(b)).max() < 1e-7, (nid, a, b)


@pytest.mark.gpu
def test_gpu_loopclose_merge_replay_matches_the_reference():
    """the same replay through the C-ABI of the CUDA library against the reference optimiser (tombstoned factors / node,
    layout recompiled on the next solve, ids stable)."""
    from pop_up_slam_b200.capi import GpuGraphAPI
    gpu = GpuGraphAPI()
    ig, a0, c0g, a1 = loopclose_run(gpu)
    assert (a0, a1, gpu.num_nodes(), gpu.num_factors()) == tuple(gold("loopclose/iterations_nodes_factors"))
    c0r, c1r = gold("loopclose/chi2")
    assert abs(c0g - c0r) <= 1e-4 * c0r and abs(gpu.chi2() - c1r) <= 1e-4 * c1r
    _compare_estimates(gpu, ig, "loopclose", 1e-4)
