"""Generate tests/golden/reference_build_{values,factors,runs}.npz: the reference side of every comparison in
tests/test_reference_build.py,
computed by oracle/_ref -- the UNMODIFIED reference sources of the hot path compiled against the API shims of oracle/ref_shim
(`make -C oracle ref REF=<reference checkout>`).

The inputs are drawn by the test module's own seeded helpers, so the tests regenerate exactly the cases stored here.  The
outputs are split over three files so that each stays below 1 MB.
Regenerate with:  python tools/make_ref_build_golden.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import oracle_api as O  # noqa: E402
import ref_api as R  # noqa: E402
import test_reference_build as T  # noqa: E402
from bench import replay_frames  # noqa: E402
from pop_up_slam_b200 import graphgen as gg  # noqa: E402

out = {}


def put_estimates(key, api, ids):
    out[key + "/poses"] = api.get_poses(ids["pose_ids"])
    out[key + "/planes"] = api.get_planes(ids["plane_ids"])


# ---- value types ----
lib = R.ref_lib()
out["values/standard_rad"] = np.array([lib.ref_standard_rad(float(t)) for t in np.linspace(-20, 20, 201)])
rows = {k: [] for k in ("pose", "vector", "exmap", "oplus", "ominus", "wTo", "oTw", "from_mat4", "plane_exmap", "plane_transform")}
for v, d, q, pl, d3 in T.value_type_inputs():
    p = R.pose_from_xyzypr(v)
    Tq = O.pose_wTo(q)
    for k, val in (("pose", p), ("vector", R.pose_vector(p)), ("exmap", R.pose_exmap(p, d)), ("oplus", R.pose_oplus(p, q)),
                   ("ominus", R.pose_ominus(p, q)), ("wTo", R.pose_wTo(p)), ("oTw", R.pose_oTw(p)), ("from_mat4", R.pose_from_mat4(Tq)),
                   ("plane_exmap", R.plane_exmap(pl, d3)), ("plane_transform", R.plane_transform(Tq, pl))):
        rows[k].append(val)
out.update({"values/" + k: np.array(v) for k, v in rows.items()})

# ---- per-factor error() / numericalDiff Jacobians ----
for robust in (None, (1, 0.8), (2, 0.5)):
    ref = R.RefAPI()
    fr = T._random_factor_graph(ref, np.random.default_rng(5), robust=robust)
    rows = {(kind, f): [] for kind in T.FACTOR_KINDS for f in ("error", "jacobian", "residual")}
    for kind, a in fr:
        J, r = ref.factor_jacobian(a)
        rows[kind, "error"].append(ref.factor_error(a))
        rows[kind, "jacobian"].append(J)
        rows[kind, "residual"].append(r)
    out.update({"factors/%s/%s/%s" % (T.robust_tag(robust), kind, f): np.array(v) for (kind, f), v in rows.items()})

# ---- the product's math header: the reference's Jacobians of the same factors ----
for name, seed, n, with_prior in (("header", 11, 150, False), ("numeric", 12, 100, True)):
    for robust in (0, 1):
        poses, planes, cases = T.math_header_cases(seed, n, with_prior)
        ref = R.RefAPI()
        if robust:
            ref.set_robust(1, 0.8)
        pid, lid = ref.add_poses(np.array(poses)), ref.add_planes(np.array(planes))
        rows = {}
        for i, (meas, si, m, si6, prior) in enumerate(cases):
            facs = [("pose_plane", ref.add_pose_plane(pid[i], lid[i], meas, si)), ("odometry", ref.add_odometry(pid[i], pid[(i + 1) % n], m, si6))]
            if with_prior:
                facs.append(("pose_prior", ref.add_pose_prior(pid[i], prior, si6)))
            for kind, f in facs:
                J, r = ref.factor_jacobian(f)
                rows.setdefault(kind + "_jacobian", []).append(J)
                rows.setdefault(kind + "_residual", []).append(r)
                if kind == "pose_prior":
                    rows.setdefault(kind + "_measurement", []).append(ref.get_measurement(f, 6))
        out.update({"%s/robust%d/%s" % (name, robust, k): np.array(v) for k, v in rows.items()})

# ---- whole Levenberg-Marquardt runs ----
for cfg, kw, builder in [(1, {}, "interleaved"), (2, {}, "interleaved"), (2, dict(seed=3), "bulk"), (3, dict(n_poses=600, n_planes=60), "bulk")]:
    key = T.lm_key(cfg, kw, builder)
    kw = dict(kw)
    g = gg.make_config(cfg, seed=kw.pop("seed", 0), **kw)
    ref = R.RefAPI()
    ir = T.BUILDERS[builder](ref, g)
    gg.configure(ref, g)
    out[key + "/chi2_initial"] = np.array(ref.chi2())
    out[key + "/iterations"] = np.array(ref.batch_optimize())
    tr = ref.trace()
    out[key + "/accepted"], out[key + "/lam"], out[key + "/chi2_new"] = tr["accepted"], tr["lam"], tr["chi2_new"]
    out[key + "/chi2"] = np.array(ref.chi2())
    put_estimates(key, ref, ir)
    out[key + "/node_start"] = np.array([ref.node_start(a) for a in list(ir["pose_ids"])[:50] + list(ir["plane_ids"])[:20]])
    out[key + "/num_nodes_factors"] = np.array([ref.num_nodes(), ref.num_factors()])

# ---- Gauss-Newton, update(), graph edits ----
g = gg.make_config(2, seed=1, n_poses=150, n_planes=30)
ref = R.RefAPI()
ir = gg.build_bulk(ref, g)
gg.configure(ref, g, method=0, max_iterations=10)
out["gn/chi2_initial"] = np.array(ref.chi2())
out["gn/iterations"] = np.array(ref.batch_optimize())
out["gn/chi2"] = np.array(ref.chi2())
put_estimates("gn", ref, ir)
ref = R.RefAPI()
ir = gg.build_bulk(ref, g)
gg.configure(ref, g, mod_batch=1)
ref.update()
ref.update()
out["update/chi2"] = np.array(ref.chi2())
put_estimates("update", ref, ir)
for f in ir["pp_fids"][5:40:7]:
    ref.remove_factor(int(f))
ref.remove_node(int(ir["plane_ids"][7]))
gg.configure(ref, g)
ref.batch_optimize()
out["edits/num_nodes_factors"] = np.array([ref.num_nodes(), ref.num_factors()])
out["edits/chi2"] = np.array(ref.chi2())
out["edits/planes"] = ref.get_planes(ir["plane_ids"][[i for i in range(len(ir["plane_ids"])) if i != 7]])

# ---- Pose3d_Plane3d_Factor2 ----
g = gg.make_config(2, seed=6, n_poses=60, n_planes=20)
ref = R.RefAPI()
ir = T.build_factor2_graph(ref, g)
gg.configure(ref, g)
out["factor2/chi2_initial"] = np.array(ref.chi2())
out["factor2/iterations"] = np.array(ref.batch_optimize())
out["factor2/accepted"] = ref.trace()["accepted"]
out["factor2/chi2"] = np.array(ref.chi2())
put_estimates("factor2", ref, ir)

# ---- get_wall_plane_equation (the reference's double copy of the pop-up arithmetic) ----
invK, Ts, segs, ns = T.popup_inputs()
planes, count = [], []
for f in range(len(Ts)):
    Tf = Ts[f].astype(np.float32).astype(np.float64)
    s = segs[f * ns:(f + 1) * ns].astype(np.float32).astype(np.float64)
    pts = np.concatenate([np.c_[s[:, 0], s[:, 1], np.ones(ns)], np.c_[s[:, 2], s[:, 3], np.ones(ns)]], axis=1).reshape(-1, 3)
    p = R.wall_plane_equation(pts @ invK.astype(np.float32).astype(np.float64).T, Tf)
    planes.append(p)
    count.append(len(p))
out["popup/planes"], out["popup/count"] = np.concatenate(planes), np.array(count)

# ---- graphs the CUDA path is compared on ----
for cfg, seed in ((1, 5), (2, 7)):
    key = "gpu_direct/config%d_seed%d" % (cfg, seed)
    g = gg.make_config(cfg, seed=seed)
    ref = R.RefAPI()
    ir = gg.build_interleaved(ref, g)
    gg.configure(ref, g)
    out[key + "/chi2_initial"] = np.array(ref.chi2())
    out[key + "/iterations"] = np.array(ref.batch_optimize())
    out[key + "/accepted"] = ref.trace()["accepted"]
    out[key + "/chi2"] = np.array(ref.chi2())
    put_estimates(key, ref, ir)

# ---- loop-closure merge replay ----
ref = R.RefAPI()
ir, it0, c0, it1 = T.loopclose_run(ref)
out["loopclose/iterations_nodes_factors"] = np.array([it0, it1, ref.num_nodes(), ref.num_factors()])
out["loopclose/chi2"] = np.array([c0, ref.chi2()])
put_estimates("loopclose", ref, ir)

# ---- frame-by-frame replay ----
g = gg.make_config(2, seed=9, n_poses=45, n_planes=12)
ref = R.RefAPI()
gg.configure(ref, g, mod_batch=1)
replay_frames(ref, g)
out["replay/num_nodes_factors"] = np.array([ref.num_nodes(), ref.num_factors()])
out["replay/chi2"] = np.array(ref.chi2())
out["replay/node_start"] = np.array([ref.node_start(i) for i in range(ref.num_nodes())])
is_plane, values = [], np.full((ref.num_nodes(), 7), np.nan)
for nid in range(ref.num_nodes()):
    try:
        values[nid] = ref.get_pose(nid)
        is_plane.append(0)
    except Exception:
        values[nid, :4] = ref.get_plane(nid)
        is_plane.append(1)
out["replay/is_plane"] = np.array(is_plane, dtype=np.int8)
out["replay/values"] = values

# three files, each below 1 MB: the math-header cases ride with the value types, the numeric-mode ones with the factors
PART_OF_SECTION = {"values": "values", "header": "values", "factors": "factors", "numeric": "factors"}
for part in ("values", "factors", "runs"):
    keys = [k for k in out if PART_OF_SECTION.get(k.split("/")[0], "runs") == part]
    path = os.path.join(ROOT, "tests", "golden", "reference_build_%s.npz" % part)
    np.savez_compressed(path, **{k: out[k] for k in keys})
    print("wrote", path, os.path.getsize(path), "bytes,", sum(out[k].size for k in keys), "values")
