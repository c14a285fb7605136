"""CPU side of the RGB-D frames: the depth oracle (tests/cpp/rgbd_oracle.cpp) pinned to cv2's convertTo and to an independent numpy
restatement of ComputeStereoFromRGBD, the GrabImageRGBD predicate at its edge, and the INTEGRATION.md snippet compiling."""
import os
import subprocess

import numpy as np
import pytest

from tests import rgbd_oracle
from tests.oracle_lib import KP_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SNIPPET = os.path.join(ROOT, "tests", "cpp", "rgbd_frame_test.cpp")
SNIPPET_EXE = os.path.join(ROOT, "build", "rgbd_frame_test")
FACTORS = [1 / 5000, 1 / 1000, 1 / 5208, 1 / 3.7, 1.0]

cv2 = pytest.importorskip("cv2")


def cv2_convert(src, f):
    """convertTo(CV_32F, f) through cv2: normalize(NORM_INF) scales by alpha / max|src| and converts with that factor."""
    m = float(np.nanmax(np.abs(src[np.isfinite(src)]))) if src.dtype == np.float32 else float(np.abs(src).max())
    return cv2.normalize(src, None, alpha=float(np.float32(f)) * m, norm_type=cv2.NORM_INF, dtype=cv2.CV_32F)


def build_snippet():
    os.makedirs(os.path.dirname(SNIPPET_EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "tests", "cpp", "cv_stub"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200", "csrc", "adapter"), "-o", SNIPPET_EXE, SNIPPET,
                           "-L" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200"), "-lorbx",
                           "-Wl,-rpath," + os.path.join(ROOT, "wut_cuda_orb_slam3_b200")])


@pytest.mark.parametrize("f", FACTORS)
def test_u16_conversion_equals_cv2_for_every_value(f):
    src = np.arange(65536, dtype=np.uint16).reshape(256, 256)
    got, converted = rgbd_oracle.grab_depth(src, f)
    assert converted                                   # a CV_16U map is always converted
    want = cv2_convert(src, f)
    assert got.tobytes() == want.tobytes()
    assert got.tobytes() == (src.astype(np.float32) * np.float32(f)).tobytes()


@pytest.mark.parametrize("f", FACTORS[:-1])
def test_f32_conversion_equals_cv2_on_special_values(f):
    rng = np.random.default_rng(3)
    vals = np.concatenate([rng.uniform(-10, 10, 4000).astype(np.float32), rng.uniform(0, 65535, 4000).astype(np.float32),
                           np.array([0.0, -0.0, -1.0, -5.5, 1e-45, 3e-39, -1e-40, 1.1754942e-38, np.inf, np.nan, 65536.0], np.float32)])
    src = np.resize(vals, 64 * 128).reshape(64, 128).astype(np.float32)
    got, converted = rgbd_oracle.grab_depth(src, f)
    assert converted
    want = src * np.float32(f) + np.float32(0)       # cvt_32f adds beta = 0: a -0 product becomes +0
    assert got.tobytes() == want.tobytes()
    # cv2 on the finite part (normalize's max would be inf / NaN otherwise); max |src| = 2^16, so normalize's scale is exactly f
    fin = np.where(np.isfinite(src), src, np.float32(0))
    assert rgbd_oracle.grab_depth(fin, f)[0].tobytes() == cv2_convert(fin, f).tobytes()


def edge_factors():
    """The adjacent floats either side of |f - 1| = 1e-5, above and below 1 (f - 1 is exact in float there)."""
    out = []
    for direction in (2.0, 0.0):
        f = np.float32(1.0)
        while not abs(float(np.float32(f - np.float32(1.0)))) > 1e-5:
            inside, f = f, np.nextafter(f, np.float32(direction))
        out.append((inside, f))
    return out


EDGE = edge_factors()


def test_predicate_at_its_edge():
    """GrabImageRGBD: the float just inside leaves a CV_32F map alone, the one just outside converts it; a CV_16U map is converted
    at either."""
    assert [(float(a), float(b)) for a, b in EDGE] == [(1 + 83 * 2 ** -23, 1 + 84 * 2 ** -23), (1 - 167 * 2 ** -24, 1 - 168 * 2 ** -24)]
    src = np.array([[3.0, 7.0, 1e-40, 4097.3]], np.float32)
    u16 = np.array([[3, 7, 65535, 4097]], np.uint16)
    for inside, outside in EDGE:
        m_in, c_in = rgbd_oracle.grab_depth(src, inside)
        m_out, c_out = rgbd_oracle.grab_depth(src, outside)
        assert not c_in and m_in.tobytes() == src.tobytes()
        assert c_out and m_out.tobytes() == (src * outside + np.float32(0)).tobytes() != src.tobytes()
        for f in (inside, outside):
            m, c = rgbd_oracle.grab_depth(u16, f)
            assert c and m.tobytes() == (u16.astype(np.float32) * f).tobytes()
    assert not rgbd_oracle.grab_depth(src, 1.0)[1]


def numpy_compute_stereo_from_rgbd(depth, keys, keys_un, bf):
    u = np.full(len(keys), -1, np.float32)
    d = np.full(len(keys), -1, np.float32)
    z = depth[keys["y"].astype(np.int32), keys["x"].astype(np.int32)]
    ok = z > 0
    d[ok] = z[ok]
    with np.errstate(over="ignore"):                   # bf / denormal = inf, as in float arithmetic
        u[ok] = keys_un["x"][ok] - np.float32(bf) / z[ok]
    return u, d


def test_compute_stereo_from_rgbd_matches_numpy():
    rng = np.random.default_rng(9)
    rows, cols = 480, 640
    depth = rng.uniform(-1, 8, (rows, cols)).astype(np.float32)
    depth[rng.random((rows, cols)) < 0.1] = 0
    depth[rng.random((rows, cols)) < 0.02] = np.nan
    depth[rng.random((rows, cols)) < 0.01] = np.inf
    depth[rng.random((rows, cols)) < 0.01] = np.float32(1e-42)
    n = 3000
    keys = np.zeros(n, KP_DTYPE)
    keys["x"] = rng.uniform(16, cols - 17, n).astype(np.float32); keys["y"] = rng.uniform(16, rows - 17, n).astype(np.float32)
    keys_un = keys.copy()
    keys_un["x"] += rng.uniform(-3, 3, n).astype(np.float32)
    u, d = rgbd_oracle.compute_stereo_from_rgbd(depth, keys, keys_un, 40.0)
    wu, wd = numpy_compute_stereo_from_rgbd(depth, keys, keys_un, 40.0)
    assert u.tobytes() == wu.tobytes() and d.tobytes() == wd.tobytes()
    z = depth[keys["y"].astype(np.int32), keys["x"].astype(np.int32)]
    assert (d[np.isinf(z)] == np.inf).all() and (u[np.isinf(z)] == keys_un["x"][np.isinf(z)]).all()
    assert (d[~(z > 0)] == -1).all()
    # the composite (raw map -> GrabImageRGBD -> ComputeStereoFromRGBD) on a u16 map
    raw = rng.integers(0, 40000, (rows, cols)).astype(np.uint16)
    cu, cd = rgbd_oracle.rgbd_depth(raw, 1 / 5000, keys, keys_un, 40.0)
    wu, wd = numpy_compute_stereo_from_rgbd(raw.astype(np.float32) * np.float32(1 / 5000), keys, keys_un, 40.0)
    assert cu.tobytes() == wu.tobytes() and cd.tobytes() == wd.tobytes()


def test_snippet_compiles_and_links():
    """The RGB-D Frame body of INTEGRATION.md builds against the cv stub and the library (run on the GPU in test_gpu_rgbd.py)."""
    build_snippet()
    assert os.path.exists(SNIPPET_EXE)
