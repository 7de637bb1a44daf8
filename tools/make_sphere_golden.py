"""Fixtures from the reference's own iSAM datasets (read from /root/reference, which only exists in the build
container; the committed JSON travels to the GPU box):

  tests/golden/sphere400.json  -- ISAM/data/sphere400.txt parsed with the Loader's conventions
      (ISAM/isam/Loader.cpp:316-365: EDGE3 i j x y z roll pitch yaw + 21 sqrt-information entries, rotational block
      re-ordered to yaw, pitch, roll; prior sqrt-information 100*I on the first pose) together with the oracle's
      Gauss-Newton result on it (numeric Jacobians as upstream): chi2 before / after, iterations, every 8th pose.
  tests/golden/sphere2500.txt.xz, tests/golden/sphere2500_groundtruth.txt.xz  -- ISAM/data/sphere2500.txt and
      data/groundtruth/sphere2500_groundtruth.txt, byte for byte, xz-compressed.

Regenerate with:  python tools/make_sphere_golden.py
"""
import json
import lzma
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle_api import OracleAPI  # noqa: E402
from pop_up_slam_b200 import graphgen as gg  # noqa: E402

DATA = "/root/reference/pop_planar_slam/Thirdparty/isam/data"


def load_edge3(path):
    """[(i, j, meas[x y z yaw pitch roll], sqrtinf packed upper-triangular 21)] in file order (.xz files are decompressed)"""
    edges = []
    for line in (lzma.open(path, "rt") if path.endswith(".xz") else open(path)):
        tok = line.split()
        if not tok or tok[0] != "EDGE3":
            continue
        i, j = int(tok[1]), int(tok[2])
        x, y, z, roll, pitch, yaw = map(float, tok[3:9])
        S = np.zeros((6, 6))
        S[np.triu_indices(6)] = list(map(float, tok[9:30]))
        S2 = S.copy()                                   # Loader.cpp:333-345
        S2[3:, 3:] = [[S[5, 5], S[4, 5], S[3, 5]], [0, S[4, 4], S[3, 4]], [0, 0, S[3, 3]]]
        edges.append((i, j, [x, y, z, yaw, pitch, roll], S2[np.triu_indices(6)].tolist()))
    return edges


def build(api, edges):
    ids = {}
    for (i, j, m, s) in edges:
        if not ids:
            ids[i] = api.add_pose(None)
            api.add_pose_prior(ids[i], np.zeros(6), gg.diag_ut([100.0] * 6))
        for k in (i, j):
            if k not in ids:
                ids[k] = api.add_pose(None)
        api.add_odometry(ids[i], ids[j], m, s)
    return ids


if __name__ == "__main__":
    edges = load_edge3(os.path.join(DATA, "sphere400.txt"))
    api = OracleAPI()
    api.set_jacobian_mode(0)
    api.set_properties(**dict(gg.PPS_PROPERTIES, method=0, max_iterations=10))
    ids = build(api, edges)
    c0 = api.chi2()
    it = api.batch_optimize()
    c1 = api.chi2()
    order = sorted(ids)
    P = api.get_poses(np.array([ids[k] for k in order]))
    out = dict(source="ISAM/data/sphere400.txt (Loader.cpp:316-365 conventions)", n_poses=len(ids), n_edges=len(edges),
               edges=[[i, j] + [float(v) for v in m] + [float(v) for v in s] for (i, j, m, s) in edges],
               properties=dict(gg.PPS_PROPERTIES, method=0, max_iterations=10),
               oracle=dict(chi2_initial=c0, chi2_final=c1, iterations=it, pose_index=order[::8], poses=P[::8].tolist()))
    path = os.path.join(ROOT, "tests", "golden", "sphere400.json")
    json.dump(out, open(path, "w"))
    print("sphere400:", len(ids), "poses", len(edges), "edges; chi2", c0, "->", c1, "in", it, "iterations; wrote", path, os.path.getsize(path), "bytes")

    for src in ("sphere2500.txt", "groundtruth/sphere2500_groundtruth.txt"):
        path = os.path.join(ROOT, "tests", "golden", os.path.basename(src) + ".xz")
        with lzma.open(path, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
            f.write(open(os.path.join(DATA, src), "rb").read())
        print("wrote", path, os.path.getsize(path), "bytes")
