"""ctypes binding of the Fuse oracle (tests/cpp/fuse_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

The oracle is compiled on demand into build/ with the flags of oracle/Makefile (no FMA contraction); it includes
oracle/projection_oracle.cpp, so the key frame's grid is the projection oracle's own."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.oracle_lib import KP_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRCS = [os.path.join(ROOT, "tests", "cpp", "fuse_oracle.cpp"), os.path.join(ROOT, "oracle", "projection_oracle.cpp")]
SO = os.path.join(ROOT, "build", "libfuse_oracle.so")

_vp = C.c_void_p


def _ptr(a):
    return a.ctypes.data_as(_vp)


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    tmp = SO + ".%d.tmp" % os.getpid()
    subprocess.check_call(["g++", "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", tmp, SRCS[0]])
    os.replace(tmp, SO)


class FuseOracle:
    def __init__(self, lib):
        self.lib = lib
        lib.orbo_kf_get_features_in_area.restype = C.c_int
        lib.orbo_kf_get_features_in_area.argtypes = [_vp, C.c_int, _vp, C.c_float, C.c_float, C.c_float, _vp]
        lib.orbo_fuse.restype = None
        lib.orbo_fuse.argtypes = [C.c_int, _vp, _vp, _vp, _vp, _vp, C.c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  C.c_float, _vp, _vp]

    def kf_get_features_in_area(self, kp, bounds_grid, x, y, r):
        kp = np.ascontiguousarray(kp, KP_DTYPE)
        out = np.zeros(max(len(kp), 1), np.int32)
        n = self.lib.orbo_kf_get_features_in_area(_ptr(kp), len(kp), _ptr(np.ascontiguousarray(bounds_grid, np.float32)), x, y, r, _ptr(out))
        return out[:n]

    def fuse(self, kfs, kf_offsets, point_desc, point, valid, u, v, invz, level, th=3.0):
        """kfs = list of dicts (tests/fuse_synth.py: kp, desc, ur or None, bg, scale, inv_sigma2, bf).  Returns (match, n_fused)."""
        n_kf = len(kfs)
        feat_off = np.zeros(n_kf + 1, np.int32)
        feat_off[1:] = np.cumsum([len(k["kp"]) for k in kfs]) if n_kf else []
        cat = (lambda parts, dt, shape: np.ascontiguousarray(np.concatenate(parts) if parts else np.zeros(shape, dt), dt))
        kp = cat([k["kp"] for k in kfs], KP_DTYPE, (0,))
        desc = cat([np.asarray(k["desc"], np.uint8).reshape(-1, 32) for k in kfs], np.uint8, (0, 32))
        ur = cat([np.full(len(k["kp"]), -1, np.float32) if k["ur"] is None else np.asarray(k["ur"], np.float32) for k in kfs], np.float32, (0,))
        bg = cat([np.asarray(k["bg"], np.float32) for k in kfs], np.float32, (0,))
        nlev = len(kfs[0]["scale"]) if n_kf else 1
        scale = cat([np.asarray(k["scale"], np.float32) for k in kfs], np.float32, (0,))
        inv = cat([np.asarray(k["inv_sigma2"], np.float32) for k in kfs], np.float32, (0,))
        bf = np.array([k["bf"] for k in kfs] or [0], np.float32)
        offs = np.ascontiguousarray(kf_offsets, np.int32)
        nq = int(offs[-1])
        pd = np.ascontiguousarray(point_desc, np.uint8).reshape(-1, 32)
        arrs = [np.ascontiguousarray(a, dt) for a, dt in ((point, np.int32), (valid, np.uint8), (u, np.float32), (v, np.float32),
                                                           (invz, np.float32), (level, np.int32))]
        match = np.full(max(nq, 1), -1, np.int32)
        n_fused = np.zeros(max(n_kf, 1), np.int32)
        self.lib.orbo_fuse(n_kf, _ptr(feat_off), _ptr(kp), _ptr(desc), _ptr(ur), _ptr(bg), nlev, _ptr(scale), _ptr(inv), _ptr(bf), _ptr(offs),
                           _ptr(pd), *[_ptr(a) for a in arrs], C.c_float(th), _ptr(match), _ptr(n_fused))
        return match[:nq], n_fused[:n_kf]


_cached = None


def load():
    global _cached
    if _cached is None:
        if not os.path.exists(SO) or any(os.path.getmtime(f) > os.path.getmtime(SO) for f in SRCS):
            build()
        _cached = FuseOracle(C.CDLL(SO))
    return _cached
