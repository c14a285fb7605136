"""ctypes binding of the RGB-D depth oracle (tests/cpp/rgbd_oracle.cpp).  TEST INFRASTRUCTURE ONLY.

The oracle is compiled on demand into build/ with the flags of oracle/Makefile (no FMA contraction)."""
import ctypes as C
import os
import subprocess

import numpy as np

from tests.oracle_lib import KP_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "rgbd_oracle.cpp")
SO = os.path.join(ROOT, "build", "librgbd_oracle.so")
DEPTH_TYPES = {np.dtype(np.uint16): 0, np.dtype(np.float32): 1}

_vp = C.c_void_p
_lib = None


def _ptr(a):
    return a.ctypes.data_as(_vp)


def _load():
    global _lib
    if _lib is None:
        os.makedirs(os.path.dirname(SO), exist_ok=True)
        tmp = SO + ".%d.tmp" % os.getpid()
        subprocess.check_call(["g++", "-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-shared", "-o", tmp, SRC])
        os.replace(tmp, SO)
        L = C.CDLL(SO)
        L.orbo_grab_depth.restype = C.c_int
        L.orbo_grab_depth.argtypes = [_vp, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_float, _vp]
        L.orbo_compute_stereo_from_rgbd.restype = None
        L.orbo_compute_stereo_from_rgbd.argtypes = [_vp, C.c_int, C.c_int, _vp, _vp, C.c_int, C.c_float, _vp, _vp]
        L.orbo_rgbd_depth.restype = None
        L.orbo_rgbd_depth.argtypes = [_vp, C.c_int, C.c_size_t, C.c_int, C.c_int, C.c_float, _vp, _vp, C.c_int, C.c_float, _vp, _vp]
        _lib = L
    return _lib


def grab_depth(depth, depth_factor):
    """Tracking::GrabImageRGBD's depth conversion: returns (float32 map, converted?)."""
    depth = np.ascontiguousarray(depth)
    rows, cols = depth.shape
    out = np.empty((rows, cols), np.float32)
    conv = _load().orbo_grab_depth(_ptr(depth), DEPTH_TYPES[depth.dtype], depth.strides[0], rows, cols, float(depth_factor), _ptr(out))
    return out, bool(conv)


def compute_stereo_from_rgbd(depth_f32, keys, keys_un, bf):
    """Frame::ComputeStereoFromRGBD on a converted map: returns (mvuRight, mvDepth)."""
    depth_f32 = np.ascontiguousarray(depth_f32, np.float32)
    keys = np.ascontiguousarray(keys, KP_DTYPE); keys_un = np.ascontiguousarray(keys_un, KP_DTYPE)
    n = len(keys)
    u = np.empty(max(n, 1), np.float32); d = np.empty(max(n, 1), np.float32)
    _load().orbo_compute_stereo_from_rgbd(_ptr(depth_f32), depth_f32.shape[0], depth_f32.shape[1], _ptr(keys), _ptr(keys_un), n, float(bf),
                                          _ptr(u), _ptr(d))
    return u[:n], d[:n]


def rgbd_depth(depth, depth_factor, keys, keys_un, bf):
    """The raw map through GrabImageRGBD, then ComputeStereoFromRGBD: returns (mvuRight, mvDepth)."""
    depth = np.ascontiguousarray(depth)
    keys = np.ascontiguousarray(keys, KP_DTYPE); keys_un = np.ascontiguousarray(keys_un, KP_DTYPE)
    n = len(keys)
    u = np.empty(max(n, 1), np.float32); d = np.empty(max(n, 1), np.float32)
    _load().orbo_rgbd_depth(_ptr(depth), DEPTH_TYPES[depth.dtype], depth.strides[0], depth.shape[0], depth.shape[1], float(depth_factor),
                            _ptr(keys), _ptr(keys_un), n, float(bf), _ptr(u), _ptr(d))
    return u[:n], d[:n]
