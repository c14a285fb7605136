"""ctypes binding of the loop-closing oracle (tests/cpp/loop_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

The oracle is compiled on demand into build/ with the flags of oracle/Makefile (no FMA contraction); it includes
tests/cpp/fuse_oracle.cpp and through it oracle/projection_oracle.cpp, so KeyFrame::GetFeaturesInArea and the grid are theirs."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.oracle_lib import KP_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRCS = [os.path.join(ROOT, "tests", "cpp", "loop_oracle.cpp"), os.path.join(ROOT, "tests", "cpp", "fuse_oracle.cpp"),
        os.path.join(ROOT, "oracle", "projection_oracle.cpp")]
SO = os.path.join(ROOT, "build", "libloop_oracle.so")

_vp = C.c_void_p


def _ptr(a):
    return a.ctypes.data_as(_vp)


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    tmp = SO + ".%d.tmp" % os.getpid()
    subprocess.check_call(["g++", "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", tmp, SRCS[0]])
    os.replace(tmp, SO)


class LoopOracle:
    def __init__(self, lib):
        self.lib = lib
        lib.orbo_search_by_projection_sim3.restype = C.c_int
        lib.orbo_search_by_projection_sim3.argtypes = [_vp, _vp, C.c_int, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, C.c_float]
        lib.orbo_fuse_sim3.restype = None
        lib.orbo_fuse_sim3.argtypes = [C.c_int, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.c_float, _vp, _vp]

    def search_by_projection_sim3(self, K, occupied, valid, u, v, level, pdesc, th, ratio=1.0):
        """K = key-frame dict (kp, desc, bg, scale); occupied[n] = vpMatched[idx] != NULL on entry.  Returns
        (match_f[n] = point index assigned by this call or -1, nmatches)."""
        kp = np.ascontiguousarray(K["kp"], KP_DTYPE)
        n = len(kp)
        desc = np.ascontiguousarray(np.asarray(K["desc"], np.uint8).reshape(n, 32))
        matched = np.where(np.asarray(occupied, bool), -2, -1).astype(np.int32) if n else np.zeros(1, np.int32)
        arrs = [np.ascontiguousarray(a, dt) for a, dt in ((valid, np.uint8), (u, np.float32), (v, np.float32), (level, np.int32))]
        pd = np.ascontiguousarray(pdesc, np.uint8).reshape(-1, 32)
        nm = self.lib.orbo_search_by_projection_sim3(_ptr(kp), _ptr(desc), n, _ptr(np.ascontiguousarray(K["bg"], np.float32)),
                                                     _ptr(np.ascontiguousarray(K["scale"], np.float32)), _ptr(matched), len(arrs[0]),
                                                     *[_ptr(a) for a in arrs], _ptr(pd), int(th), C.c_float(ratio))
        if nm < 0:
            raise ValueError("the reference would write vpMatched[-1]")
        return np.where(matched >= 0, matched, -1).astype(np.int32)[:n], nm

    def fuse_sim3(self, kfs, kf_offsets, point_desc, point, valid, u, v, level, th=4.0):
        """kfs = list of key-frame dicts (kp, desc, bg, scale).  Returns (match, n_fused)."""
        n_kf = len(kfs)
        feat_off = np.zeros(n_kf + 1, np.int32)
        feat_off[1:] = np.cumsum([len(k["kp"]) for k in kfs]) if n_kf else []
        cat = (lambda parts, dt, shape: np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(shape, dt), dt))
        kp = cat([k["kp"] for k in kfs], KP_DTYPE, (0,))
        desc = cat([np.asarray(k["desc"], np.uint8).reshape(-1, 32) for k in kfs], np.uint8, (0, 32))
        bg = cat([np.asarray(k["bg"], np.float32) for k in kfs], np.float32, (0,))
        nlev = len(kfs[0]["scale"]) if n_kf else 1
        scale = cat([np.asarray(k["scale"], np.float32) for k in kfs], np.float32, (0,))
        offs = np.ascontiguousarray(kf_offsets, np.int32)
        nq = int(offs[-1])
        pd = np.ascontiguousarray(point_desc, np.uint8).reshape(-1, 32)
        arrs = [np.ascontiguousarray(a, dt) for a, dt in ((point, np.int32), (valid, np.uint8), (u, np.float32), (v, np.float32),
                                                           (level, np.int32))]
        match = np.full(max(nq, 1), -1, np.int32)
        n_fused = np.zeros(max(n_kf, 1), np.int32)
        self.lib.orbo_fuse_sim3(n_kf, _ptr(feat_off), _ptr(kp), _ptr(desc), _ptr(bg), nlev, _ptr(scale), _ptr(offs), _ptr(pd),
                                *[_ptr(a) for a in arrs], C.c_float(th), _ptr(match), _ptr(n_fused))
        return match[:nq], n_fused[:n_kf]


_cached = None


def load():
    global _cached
    if _cached is None:
        if not os.path.exists(SO) or any(os.path.getmtime(f) > os.path.getmtime(SO) for f in SRCS):
            build()
        _cached = LoopOracle(C.CDLL(SO))
    return _cached
