"""ctypes binding of the SearchForInitialization oracle (tests/cpp/init_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

The oracle is compiled on demand into build/ with the flags of oracle/Makefile (no FMA contraction); it includes
oracle/projection_oracle.cpp, so the frame grid and GetFeaturesInArea it searches are the projection oracle's own."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.oracle_lib import KP_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRCS = [os.path.join(ROOT, "tests", "cpp", "init_oracle.cpp"), os.path.join(ROOT, "oracle", "projection_oracle.cpp")]
SO = os.path.join(ROOT, "build", "libinit_oracle.so")

_vp = C.c_void_p


def _ptr(a):
    return a.ctypes.data_as(_vp)


def build():
    os.makedirs(os.path.dirname(SO), exist_ok=True)
    tmp = SO + ".%d.tmp" % os.getpid()
    subprocess.check_call(["g++", "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", tmp, SRCS[0]])
    os.replace(tmp, SO)


class InitOracle:
    def __init__(self, lib):
        self.lib = lib
        lib.orbo_search_for_initialization.restype = C.c_int
        lib.orbo_search_for_initialization.argtypes = [_vp, _vp, C.c_int, _vp, _vp, C.c_int, _vp, _vp, C.c_int, C.c_float, C.c_int, _vp]

    def search_for_initialization(self, kp1, desc1, kp2, desc2, bounds_grid, prev_matched, window_size=100, nnratio=0.9,
                                  check_orientation=True):
        """Returns (vnMatches12, nmatches, vbPrevMatched after the call); the input array is left as it is."""
        kp1 = np.ascontiguousarray(kp1, KP_DTYPE); kp2 = np.ascontiguousarray(kp2, KP_DTYPE)
        d1 = np.ascontiguousarray(desc1, np.uint8).reshape(len(kp1), 32); d2 = np.ascontiguousarray(desc2, np.uint8).reshape(len(kp2), 32)
        bg = np.ascontiguousarray(bounds_grid, np.float32)
        prev = np.array(prev_matched, np.float32, copy=True).reshape(len(kp1), 2)
        out = np.full(max(len(kp1), 1), -1, np.int32)
        nm = self.lib.orbo_search_for_initialization(_ptr(kp1), _ptr(d1), len(kp1), _ptr(kp2), _ptr(d2), len(kp2), _ptr(bg), _ptr(prev),
                                                     int(window_size), C.c_float(nnratio), int(check_orientation), _ptr(out))
        if nm < 0:
            raise ValueError("keypoint angles out of range (the reference asserts)")
        return out[:len(kp1)], nm, prev


_cached = None


def load():
    global _cached
    if _cached is None:
        if not os.path.exists(SO) or any(os.path.getmtime(f) > os.path.getmtime(SO) for f in SRCS):
            build()
        _cached = InitOracle(C.CDLL(SO))
    return _cached
