"""Test-side binding of oracle/_ref/libisam_ref.so: the UNMODIFIED reference sources of the hot path (iSAM's Slam /
Optimizer / Cholesky / numericalDiff, slam3d.h, isam_plane3d.{h,cpp}) compiled against the API shims of oracle/ref_shim
(recipe: `make -C oracle ref`, needs the reference checkout; the built library travels to the GPU box).

Test infrastructure only -- never imported by the product or the tests.  The fixture generators tools/make_ref_golden.py
and tools/make_ref_build_golden.py run it to write tests/golden/reference_build.json and reference_build_*.npz, which
carry its outputs to the tests; bench.py --impl reference also times it when the library has been built."""
import ctypes as C
import os
import subprocess

import numpy as np

from pop_up_slam_b200.capi import GraphAPI, _dp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_LIB = os.path.join(ROOT, "oracle", "_ref", "libisam_ref.so")
REFERENCE = "/root/reference"

_lib = None


def available():
    if os.path.exists(REF_LIB):
        return True
    if os.path.isdir(os.path.join(REFERENCE, "pop_planar_slam")):
        try:
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref"])
        except Exception:
            return False
    return os.path.exists(REF_LIB)


def ref_lib():
    global _lib
    if _lib is None:
        if not available():
            raise RuntimeError("oracle/_ref/libisam_ref.so is not built (needs the reference checkout: make -C oracle ref)")
        _lib = C.CDLL(REF_LIB)
        _lib.ref_standard_rad.restype = C.c_double
        _lib.ref_standard_rad.argtypes = [C.c_double]
    return _lib


class RefAPI(GraphAPI):
    """isam::Slam of the reference behind the same Python surface as the CUDA library and the oracle."""

    def __init__(self):
        super().__init__(ref_lib(), "ref_", 0)

    def factor_jacobian(self, fid):
        """Factor::jacobian() of the reference (numericalDiff, eps = 1e-4) at the current estimate: (J, residual)."""
        Hm = np.zeros(6 * 12)
        r = np.zeros(6)
        ncols = self._chk(self.lib.ref_factor_jacobian(self.h, int(fid), 0, _dp(Hm), _dp(r)))
        dim = 3 if ncols in (3, 9) else 6
        return Hm[:dim * ncols].reshape(dim, ncols).copy(), r[:dim].copy()

    def factor_error(self, fid):
        r = np.zeros(6)
        d = self._chk(self.lib.ref_factor_error(self.h, int(fid), _dp(r)))
        return r[:d].copy()


def _call(fn, n_out, *args):
    out = np.zeros(n_out)
    fn(*[_dp(np.ascontiguousarray(a, dtype=np.float64)) for a in args], _dp(out))
    return out


def pose_from_xyzypr(v): return _call(ref_lib().ref_pose_from_xyzypr, 7, v)
def pose_vector(p7): return _call(ref_lib().ref_pose_vector, 6, p7)
def pose_exmap(p7, d6): return _call(ref_lib().ref_pose_exmap, 7, p7, d6)
def pose_oplus(a7, b7): return _call(ref_lib().ref_pose_oplus, 7, a7, b7)
def pose_ominus(a7, b7): return _call(ref_lib().ref_pose_ominus, 7, a7, b7)
def pose_wTo(p7): return _call(ref_lib().ref_pose_wTo, 16, p7).reshape(4, 4)
def pose_oTw(p7): return _call(ref_lib().ref_pose_oTw, 16, p7).reshape(4, 4)
def pose_from_mat4(T): return _call(ref_lib().ref_pose_from_mat4, 7, np.asarray(T).reshape(16))
def plane_exmap(p4, d3): return _call(ref_lib().ref_plane_exmap, 4, p4, d3)
def plane_transform(T, p4): return _call(ref_lib().ref_plane_transform, 4, np.asarray(T).reshape(16), p4)


def wall_plane_equation(rays, T):
    """get_wall_plane_equation (isam_plane3d.cpp:20-55): rays [2n][3] (pairs), T 4x4 -> [n][4] sensor-frame planes."""
    rays = np.ascontiguousarray(rays, dtype=np.float64)
    n = rays.shape[0] // 2
    out = np.zeros((n, 4))
    got = ref_lib().ref_wall_plane_equation(n, _dp(rays), _dp(np.ascontiguousarray(T, dtype=np.float64).reshape(16)), _dp(out))
    return out[:got]
