"""RGB-D frames (orbx_extract_rgbd, orbx_extract_rgbd_batch, orbx_extract_rgbd_batch_device): the one call equals the pieces it
replaces (orbx_extract / orbx_extract_color with vLappingArea (0, 0), orbx_undistort_keypoints) byte for byte, mvuRight / mvDepth
equal the CPU oracle of GrabImageRGBD + ComputeStereoFromRGBD on the same raw map, and every batch frame equals the single call."""
import ctypes as C
import os
import subprocess
import threading

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import rgbd_oracle
from tests.test_rgbd_cpu import EDGE, SNIPPET_EXE, build_snippet
from wut_cuda_orb_slam3_b200 import capi, synth
from wut_cuda_orb_slam3_b200.capi import KP_DTYPE, lib, ptr
from wut_cuda_orb_slam3_b200.prep import rgbd_calib

pytestmark = pytest.mark.gpu

SHAPES = [(640, 480, 1000), (752, 480, 1200)]          # TUM RGB-D, and a EuRoC-size frame
K = np.array([517.306408, 516.469215, 318.643040, 255.313989], np.float32)
TUM1 = [0.262383, -0.953104, -0.005358, 0.002628, 1.163314]
DIST_SETS = {"none": [], "zero_first": [0.0, 0.1, 0.01, -0.01, 0.2], "four": TUM1[:4], "tum1": TUM1,
             "eight": TUM1 + [0.01, -0.02, 0.003], "twelve": TUM1 + [0.01, -0.02, 0.003, 1e-3, -2e-3, 5e-4, 1e-4]}
BF = 40.0
TUM_FACTOR = 1.0 / 5000.0


def coded_u16(rows, cols, seed=0):
    """Raw u16 depth whose value follows (row, col), with holes (0)."""
    y, x = np.mgrid[0:rows, 0:cols]
    d = (1000 + y * 97 + x * 3 + seed).astype(np.uint16)
    d[(x + y + seed) % 7 == 0] = 0
    return d


def coded_f32(rows, cols, seed=0):
    """f32 depth whose value is 1 + row * 1024 + col (unique per pixel), with holes, NaN, negatives, +inf and denormals."""
    y, x = np.mgrid[0:rows, 0:cols]
    d = (1 + y * 1024 + x).astype(np.float32)
    k = (x * 7 + y * 3 + seed) % 13
    d[k == 0] = 0; d[k == 1] = np.nan; d[k == 2] = -d[k == 2]; d[k == 3] = np.inf; d[k == 4] = np.float32(3e-41); d[k == 5] = -0.0
    return d


def color_of(seed, cols, rows, ch):
    planes = [synth.image(seed + c, cols, rows) for c in range(ch)]
    return np.ascontiguousarray(np.stack(planes, axis=2))


def assert_in_bounds(kp, rows, cols):
    assert ((kp["x"] >= 0) & (kp["x"].astype(np.int32) < cols) & (kp["y"] >= 0) & (kp["y"].astype(np.int32) < rows)).all()


def oracle_depth(raw, factor, kp, kp_un):
    return rgbd_oracle.rgbd_depth(raw, factor, kp, kp_un, BF)


@pytest.mark.parametrize("cols,rows,nfeatures", SHAPES)
@pytest.mark.parametrize("dist", sorted(DIST_SETS))
def test_single_frame_equals_pieces_and_oracle(oracle, cols, rows, nfeatures, dist):
    img = synth.image(7, cols, rows)
    raw = coded_u16(rows, cols)
    ex = orbx.ORBextractor(nfeatures, 1.2, 8, 20, 7)
    kp, kp_un, desc, u, d = orbx.extract_rgbd(ex, img, raw, K, DIST_SETS[dist], BF, TUM_FACTOR)
    nm, wkp, wdesc = orbx.ORBextractor(nfeatures, 1.2, 8, 20, 7)(img, None, (0, 0))
    assert nm == len(kp) and kp.tobytes() == wkp.tobytes() and np.array_equal(desc, wdesc)
    assert kp_un.tobytes() == orbx.undistort_keypoints(kp, K, DIST_SETS[dist]).tobytes()
    assert_in_bounds(kp, rows, cols)
    ou, od = oracle_depth(raw, TUM_FACTOR, kp, kp_un)
    assert u.tobytes() == ou.tobytes() and d.tobytes() == od.tobytes()
    assert (d > 0).sum() > 0.7 * len(d) and (d == -1).sum() > 0
    # the handle keeps frame 0 inspectable, as after orbx_extract
    assert np.array_equal(ex.pyramid_level(0), img)
    if dist == "tum1" and cols == 640:
        # the whole chain against the oracle's own extraction and undistortion
        okp, _, _ = oracle.extractor(nfeatures, 1.2, 8, 20, 7).extract(img, (0, 0))
        assert len(okp) == len(kp)
        for f in ("x", "y", "octave", "response"):
            assert np.array_equal(okp[f], kp[f]), f
        okp_un = oracle.undistort_keypoints(okp, K, np.float32(TUM1), K)
        assert np.array_equal(okp_un["x"], kp_un["x"]) and np.array_equal(okp_un["y"], kp_un["y"])
        ou2, od2 = oracle_depth(raw, TUM_FACTOR, okp, okp_un)
        assert u.tobytes() == ou2.tobytes() and d.tobytes() == od2.tobytes()


@pytest.mark.parametrize("ch", [3, 4])
@pytest.mark.parametrize("rgb", [True, False])
def test_color_input(ch, rgb):
    cols, rows, nf = SHAPES[0]
    im = color_of(30, cols, rows, ch)
    raw = coded_u16(rows, cols, seed=2)
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    ex.set_pyramid_mirror(True)
    kp, kp_un, desc, u, d = orbx.extract_rgbd(ex, im, raw, K, TUM1, BF, TUM_FACTOR, rgb=rgb)
    nm, wkp, wdesc = orbx.ORBextractor(nf, 1.2, 8, 20, 7).extract_color(im, rgb, (0, 0))
    assert nm == len(kp) > 100 and kp.tobytes() == wkp.tobytes() and np.array_equal(desc, wdesc)
    assert kp_un.tobytes() == orbx.undistort_keypoints(kp, K, TUM1).tobytes()
    ou, od = oracle_depth(raw, TUM_FACTOR, kp, kp_un)
    assert u.tobytes() == ou.tobytes() and d.tobytes() == od.tobytes()
    assert ex.pyramid_mirror(0).shape == (rows, cols)        # the mirror was filled


DEPTH_CASES = [("u16", TUM_FACTOR), ("u16", 1.0), ("f32", 1.0), ("f32", 1.0 / 1000), ("f32", float(EDGE[0][0])), ("f32", float(EDGE[0][1])),
               ("f32", float(EDGE[1][0])), ("f32", float(EDGE[1][1]))]


@pytest.mark.parametrize("kind,factor", DEPTH_CASES)
def test_depth_semantics(kind, factor):
    cols, rows, nf = SHAPES[0]
    img = synth.image(11, cols, rows)
    raw = coded_u16(rows, cols, seed=3) if kind == "u16" else coded_f32(rows, cols)
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    kp, kp_un, _, u, d = orbx.extract_rgbd(ex, img, raw, K, TUM1, BF, np.float32(factor))
    assert_in_bounds(kp, rows, cols)
    ou, od = oracle_depth(raw, np.float32(factor), kp, kp_un)
    assert u.tobytes() == ou.tobytes() and d.tobytes() == od.tobytes()
    yi, xi = kp["y"].astype(np.int32), kp["x"].astype(np.int32)
    if kind == "f32" and factor == 1.0:
        # the unique code shows the sample's (row, col) exactly: truncation of the DISTORTED keypoint
        ok = d > 0
        coded = np.isfinite(d) & (d >= 1)                   # samples that kept their code (not +inf or a denormal)
        assert coded.sum() > 100 and np.array_equal(d[coded], (1 + yi * 1024 + xi)[coded].astype(np.float32))
        assert np.isinf(d).any() and np.array_equal(u[np.isinf(d)], kp_un["x"][np.isinf(d)])
        assert ((d > 0) & (d < 1e-38)).any()                # denormal samples are depths, as on the CPU
        assert (d[~ok] == -1).all() and (u[~ok] == -1).all()
    # a depth map with a row step wider than the row gives the same bytes
    wide = np.zeros((rows, cols + 5), raw.dtype)
    wide[:, :cols] = raw
    r2 = orbx.extract_rgbd(ex, img, wide[:, :cols], K, TUM1, BF, np.float32(factor))
    assert r2[3].tobytes() == u.tobytes() and r2[4].tobytes() == d.tobytes()


def pinned(shape, dtype):
    import torch
    tdt = {np.uint8: torch.uint8, np.uint16: torch.int16, np.float32: torch.float32}[dtype]
    return torch.empty(shape, dtype=tdt, pin_memory=True).numpy().view(dtype)


def make_frames(n, cols, rows, seed0, depth="u16", pin=False):
    imgs = pinned((n, rows, cols), np.uint8) if pin else np.empty((n, rows, cols), np.uint8)
    dt = np.uint16 if depth == "u16" else np.float32
    deps = pinned((n, rows, cols), dt) if pin else np.empty((n, rows, cols), dt)
    for i in range(n):
        imgs[i] = synth.image(seed0 + i, cols, rows)
        deps[i] = coded_u16(rows, cols, seed=i) if depth == "u16" else coded_f32(rows, cols, seed=i)
    return imgs, deps


def single_reference(nf, imgs, deps, dist, factor):
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    return [orbx.extract_rgbd(ex, imgs[i], deps[i], K, dist, BF, factor) for i in range(len(imgs))]


def assert_frame(got, want, i):
    n, kp, kp_un, desc, u, d = got
    a = n[i]
    assert a == len(want[0]), (i, a, len(want[0]))
    for g, w in zip((kp[i, :a], kp_un[i, :a], desc[i, :a], u[i, :a], d[i, :a]), want):
        assert g.tobytes() == w.tobytes(), i


def chunk_schedule(n, chunk):
    """api.cu chunk_schedule: (first frame, frames) per chunk of the host call."""
    sched, f0 = [], 0
    ramp = (max(chunk // 4, 1), max(chunk // 2, 1))
    for r in range(2):
        if n - f0 > 2 * chunk:
            sched.append((f0, ramp[r])); f0 += ramp[r]
    tail = ramp[0] + ramp[1] if n - f0 > 3 * chunk else 0
    while f0 < n - tail:
        nf = min(chunk, n - tail - f0); sched.append((f0, nf)); f0 += nf
    if tail:
        sched += [(f0, ramp[1]), (f0 + ramp[1], ramp[0])]
    return sched


# (frames, max_batch, pinned, depth type): default chunking is 64 frames on the slot streams: 1 and 3 frames are one chunk,
# 70 frames two chunks, 250 frames ramp up, ramp down and reuse slots; max_batch = 256: one 256-frame chunk + a 44-frame one on the
# serial three-stream pipeline; max_batch = 128: 700 frames ramp up, ramp down and reuse slots on the serial pipeline.
HOST_CASES = [(1, 0, False, "u16"), (3, 0, True, "f32"), (70, 0, False, "u16"), (250, 0, True, "u16"), (300, 256, True, "f32"),
              (700, 128, True, "u16")]


def test_host_cases_reach_every_branch():
    slots = 6
    seen = set()
    for n, max_batch, _, _ in HOST_CASES:
        chunk = min(max_batch, n) if max_batch else min(n, 64)
        s = chunk_schedule(n, chunk)
        assert sum(p for _, p in s) == n and all(0 < p <= chunk for _, p in s)
        serial = chunk >= 128
        ramp_down = len(s) >= 2 and s[-1][1] < s[-2][1] < chunk
        seen.add((serial, "reuse" if len(s) > slots else "no-reuse", "ramp" if ramp_down else "no-ramp"))
    assert (False, "reuse", "ramp") in seen and (True, "reuse", "ramp") in seen and (True, "no-reuse", "no-ramp") in seen
    assert (False, "no-reuse", "no-ramp") in seen


@pytest.mark.parametrize("n,max_batch,pin,depth", HOST_CASES)
def test_host_batch_equals_single_frames(n, max_batch, pin, depth):
    cols, rows, nf = SHAPES[0] if n > 100 or n == 3 else SHAPES[1]
    imgs, deps = make_frames(n, cols, rows, seed0=100 + n, depth=depth, pin=pin)
    factor = TUM_FACTOR if depth == "u16" else 1.0
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7, max_batch=max_batch)
    got = ex.extract_rgbd_batch(imgs, deps, K, TUM1, BF, factor)
    want = single_reference(nf, imgs, deps, TUM1, factor)
    for i in range(n):
        assert_frame(got, want[i], i)
    with pytest.raises(capi.OrbxError):          # the batch's pyramids are not kept for inspection
        ex.pyramid_level(0, frame=0)


@pytest.mark.parametrize("n,max_batch", [(21, 16), (3, 0)])
def test_device_batch_on_caller_stream_with_color(n, max_batch):
    import torch
    cols, rows, nf = SHAPES[0]
    colors = np.stack([color_of(500 + 3 * i, cols, rows, 3) for i in range(n)])
    deps = np.stack([coded_u16(rows, cols, seed=i) for i in range(n)])
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7, max_batch=max_batch)
    cap = ex.max_keypoints(rows, cols)
    ref = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    want = [orbx.extract_rgbd(ref, colors[i], deps[i], K, TUM1, BF, TUM_FACTOR, rgb=True) for i in range(n)]
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    sentinel = -7.5
    d_kp = torch.zeros((n, cap * KP_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    d_kpu = torch.full((n, cap * KP_DTYPE.itemsize), 0xA5, dtype=torch.uint8, device=dev)
    d_desc = torch.zeros((n, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(n, dtype=torch.int32, device=dev)
    d_u = torch.full((n, cap), sentinel, dtype=torch.float32, device=dev); d_d = torch.full_like(d_u, sentinel)
    d_gray = torch.empty((n, rows, cols), dtype=torch.uint8, device=dev)
    with torch.cuda.stream(stream):
        big = torch.randn(4096, 4096, device=dev)            # the inputs are written behind a long busy kernel
        for _ in range(4):
            big = big @ big.T / 4096.0
        d_col = torch.from_numpy(colors).to(dev, non_blocking=False)
        d_dep = torch.from_numpy(deps.view(np.int16)).to(dev, non_blocking=False)
        capi.check(lib().orbx_cvt_gray_device(0, ptr(d_col), cols * 3, rows * cols * 3, 3, 1, n, rows, cols, ptr(d_gray), cols, rows * cols,
                                              ptr(stream.cuda_stream)))
        ex.extract_rgbd_batch_device(d_gray, d_dep, n, rows, cols, cols, rows * cols, 0, cols * 2, rows * cols * 2, K, TUM1, BF, TUM_FACTOR,
                                     d_kp, d_kpu, d_desc, cap, d_n, d_u, d_d, stream=stream.cuda_stream)
    # the next extraction on the handle waits for the batch on the caller's stream (no orbx_sync)
    img = synth.image(5, cols, rows)
    nm, k1, _ = ex(img, None, (0, 0))
    fnm, fk1, _ = orbx.ORBextractor(nf, 1.2, 8, 20, 7)(img, None, (0, 0))
    assert nm == fnm and k1.tobytes() == fk1.tobytes()
    cnt = d_n.cpu().numpy()
    kp = d_kp.cpu().numpy().view(KP_DTYPE).reshape(n, cap); kpu = d_kpu.cpu().numpy()
    desc = d_desc.cpu().numpy(); u = d_u.cpu().numpy(); d = d_d.cpu().numpy()
    for i in range(n):
        a = cnt[i]
        assert a == len(want[i][0])
        assert kp[i, :a].tobytes() == want[i][0].tobytes() and np.array_equal(desc[i, :a], want[i][2])
        assert kpu[i].view(KP_DTYPE)[:a].tobytes() == want[i][1].tobytes()
        assert u[i, :a].tobytes() == want[i][3].tobytes() and d[i, :a].tobytes() == want[i][4].tobytes()
        assert (u[i, a:] == sentinel).all() and (d[i, a:] == sentinel).all() and (kpu[i, a * KP_DTYPE.itemsize:] == 0xA5).all()


def _raw_batch(ex, imgs, deps, cap, guard=64, depth_type=0, calib=None):
    n, rows, cols = imgs.shape
    kp = np.full(n * cap * 28 + guard, 0xA5, np.uint8); kpu = kp.copy()
    desc = np.full(n * cap * 32 + guard, 0xA5, np.uint8)
    u = np.full(n * cap * 4 + guard, 0xA5, np.uint8); d = u.copy()
    cnt = np.full(n + guard // 4, -3, np.int32)
    pi = (C.c_void_p * max(n, 1))(*[imgs.ctypes.data + i * imgs.strides[0] for i in range(n)])
    pd = (C.c_void_p * max(n, 1))(*[deps.ctypes.data + i * deps.strides[0] for i in range(n)])
    c, _keep = calib if calib else rgbd_calib(K, TUM1, BF, TUM_FACTOR)
    rc = lib().orbx_extract_rgbd_batch(ex._h, pi, pd, n, rows, cols, cols, depth_type, deps.strides[1], C.byref(c), ptr(kp), ptr(kpu),
                                       ptr(desc), cap, ptr(cnt), ptr(u), ptr(d))
    intact = all((a[-guard:] == 0xA5).all() for a in (kp, kpu, desc, u, d)) and (cnt[n:] == -3).all()
    return rc, cnt[:n], intact


def test_capacity_overflow_keeps_guards():
    cols, rows, nf = SHAPES[0]
    imgs, deps = make_frames(5, cols, rows, seed0=40)
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    rc, cnt, intact = _raw_batch(ex, imgs, deps, 200)
    assert rc == capi.ORBX_ERR_CAPACITY and intact and (cnt > 200).any()
    rc, _, intact = _raw_batch(ex, imgs, deps, ex.max_keypoints(rows, cols))
    assert rc == capi.ORBX_OK and intact
    # the single-frame call
    c, _keep = rgbd_calib(K, TUM1, BF, TUM_FACTOR)
    guard = 64
    kp = np.full(200 * 28 + guard, 0xA5, np.uint8); kpu = kp.copy(); desc = np.full(200 * 32 + guard, 0xA5, np.uint8)
    u = np.full(200 * 4 + guard, 0xA5, np.uint8); d = u.copy()
    n = C.c_int(0)
    rc = lib().orbx_extract_rgbd(ex._h, ptr(imgs[0]), rows, cols, cols, 1, 0, ptr(deps[0]), 0, cols * 2, C.byref(c), ptr(kp), ptr(kpu), ptr(desc),
                                 200, C.byref(n), ptr(u), ptr(d))
    assert rc == capi.ORBX_ERR_CAPACITY and n.value > 200
    assert all((a[-guard:] == 0xA5).all() for a in (kp, kpu, desc, u, d))


def test_bad_arguments_and_zero_frames():
    cols, rows, nf = 320, 240, 500
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    img = synth.image(1, cols, rows)
    dep = coded_u16(rows, cols)
    cap = ex.max_keypoints(rows, cols)
    kp = np.zeros(cap, KP_DTYPE); kpu = kp.copy(); de = np.zeros((cap, 32), np.uint8); fl = np.zeros(cap, np.float32); fl2 = fl.copy()
    n = C.c_int(0)
    good, _k1 = rgbd_calib(K, TUM1, BF, TUM_FACTOR)
    bad_nd, _k2 = rgbd_calib(K, TUM1[:3], BF, TUM_FACTOR)
    null_dist, _k3 = rgbd_calib(K, TUM1, BF, TUM_FACTOR)
    null_dist.dist = None

    def single(h=ex._h, im=img, r=rows, c=cols, step=cols, ch=1, depth=dep, dt=0, dstep=cols * 2, calib=good, capacity=cap):
        return lib().orbx_extract_rgbd(h, ptr(im) if im is not None else None, r, c, step, ch, 0, ptr(depth) if depth is not None else None, dt,
                                       dstep, C.byref(calib) if calib is not None else None, ptr(kp), ptr(kpu), ptr(de), capacity, C.byref(n),
                                       ptr(fl), ptr(fl2))

    assert single() == capi.ORBX_OK
    assert single(h=None) == capi.ORBX_ERR_INVALID_ARG
    assert single(im=None) == capi.ORBX_ERR_EMPTY_IMAGE
    assert single(r=0) == capi.ORBX_ERR_EMPTY_IMAGE
    assert single(c=0) == capi.ORBX_ERR_EMPTY_IMAGE
    assert single(depth=None) == capi.ORBX_ERR_INVALID_ARG
    assert single(dt=2) == capi.ORBX_ERR_INVALID_ARG
    assert single(dt=-1) == capi.ORBX_ERR_INVALID_ARG
    assert single(dstep=cols * 2 - 1) == capi.ORBX_ERR_INVALID_ARG
    assert single(dt=1, dstep=cols * 2) == capi.ORBX_ERR_INVALID_ARG       # f32 rows need cols * 4 bytes
    assert single(calib=None) == capi.ORBX_ERR_INVALID_ARG
    assert single(calib=bad_nd) == capi.ORBX_ERR_INVALID_ARG
    assert single(calib=null_dist) == capi.ORBX_ERR_INVALID_ARG
    assert single(ch=2) == capi.ORBX_ERR_INVALID_ARG
    assert single(ch=3) == capi.ORBX_ERR_INVALID_ARG                      # step < cols * 3
    assert single(capacity=0) == capi.ORBX_ERR_INVALID_ARG
    assert single(step=cols - 1) == capi.ORBX_ERR_INVALID_ARG
    # the batch calls: n_frames == 0 does nothing, every argument is checked first
    one_i = (C.c_void_p * 1)(img.ctypes.data); one_d = (C.c_void_p * 1)(dep.ctypes.data); null1 = (C.c_void_p * 1)(None)
    B = lib().orbx_extract_rgbd_batch

    def batch(h=ex._h, ims=one_i, deps=one_d, nfr=1, dt=0, dstep=cols * 2, calib=good, outs=True):
        o = [ptr(kp), ptr(kpu), ptr(de)] if outs else [None] * 3
        return B(h, ims, deps, nfr, rows, cols, cols, dt, dstep, C.byref(calib) if calib is not None else None, *o, cap, ptr(np.zeros(1, np.int32)),
                 ptr(fl), ptr(fl2))

    assert batch(nfr=0, ims=None, deps=None, outs=False) == capi.ORBX_OK
    assert batch() == capi.ORBX_OK
    assert batch(nfr=-1) == capi.ORBX_ERR_INVALID_ARG
    assert batch(h=None) == capi.ORBX_ERR_INVALID_ARG
    assert batch(ims=null1) == capi.ORBX_ERR_EMPTY_IMAGE
    assert batch(deps=None) == capi.ORBX_ERR_INVALID_ARG
    assert batch(deps=null1) == capi.ORBX_ERR_INVALID_ARG
    assert batch(dt=5) == capi.ORBX_ERR_INVALID_ARG
    assert batch(dstep=10) == capi.ORBX_ERR_INVALID_ARG
    assert batch(calib=None) == capi.ORBX_ERR_INVALID_ARG
    assert batch(calib=bad_nd) == capi.ORBX_ERR_INVALID_ARG
    assert batch(outs=False) == capi.ORBX_ERR_INVALID_ARG
    import torch
    dev = torch.device("cuda", 0)
    di = torch.zeros(rows * cols, dtype=torch.uint8, device=dev); dd = torch.zeros(rows * cols + 1, dtype=torch.int16, device=dev)
    dk = torch.zeros(cap * 28, dtype=torch.uint8, device=dev); dku = dk.clone(); dde = torch.zeros(cap * 32, dtype=torch.uint8, device=dev)
    dn = torch.zeros(1, dtype=torch.int32, device=dev); dfl = torch.zeros(cap, dtype=torch.float32, device=dev); dfl2 = dfl.clone()
    D = lib().orbx_extract_rgbd_batch_device

    def dcall(nfr=1, im=di, depth=ptr(dd), dpitch=cols * 2, dstride=rows * cols * 2, dt=0, calib=good):
        return D(ex._h, ptr(im) if im is not None else None, rows * cols, cols, depth, dstride, dpitch, dt, nfr, rows, cols,
                 C.byref(calib) if calib is not None else None, ptr(dk), ptr(dku), ptr(dde), cap, ptr(dn), ptr(dfl), ptr(dfl2), None)

    assert dcall(nfr=0) == capi.ORBX_OK
    assert dcall(nfr=-1) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(im=None) == capi.ORBX_ERR_EMPTY_IMAGE
    assert dcall(depth=None) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(depth=C.c_void_p(dd.data_ptr() + 1)) == capi.ORBX_ERR_INVALID_ARG      # misaligned u16 base
    assert dcall(dpitch=cols * 2 + 1) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(dpitch=cols) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(dt=3) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(calib=bad_nd) == capi.ORBX_ERR_INVALID_ARG
    assert dcall() == capi.ORBX_OK
    ex.sync()


def test_frame_without_keypoints():
    cols, rows, nf = SHAPES[0]
    flat = np.full((rows, cols), 128, np.uint8)
    dep = coded_u16(rows, cols)
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    kp, kp_un, desc, u, d = orbx.extract_rgbd(ex, flat, dep, K, TUM1, BF, TUM_FACTOR)
    assert len(kp) == len(kp_un) == len(desc) == len(u) == len(d) == 0
    imgs, deps = make_frames(3, cols, rows, seed0=70)
    imgs[1] = flat
    got = ex.extract_rgbd_batch(imgs, deps, K, TUM1, BF, TUM_FACTOR)
    assert got[0][1] == 0 and got[0][0] > 0 and got[0][2] > 0
    want = single_reference(nf, imgs, deps, TUM1, TUM_FACTOR)
    for i in range(3):
        assert_frame(got, want[i], i)


def test_two_handles_on_two_threads():
    cols, rows, nf = SHAPES[0]
    sets = [make_frames(12, cols, rows, seed0=s) for s in (200, 300)]
    want = [single_reference(nf, im, dp, TUM1, TUM_FACTOR) for im, dp in sets]
    got = [None, None]
    errors = []

    def run(k):
        try:
            ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
            for _ in range(2):
                got[k] = ex.extract_rgbd_batch(sets[k][0], sets[k][1], K, TUM1, BF, TUM_FACTOR)
                single = [orbx.extract_rgbd(ex, sets[k][0][i], sets[k][1][i], K, TUM1, BF, TUM_FACTOR) for i in (0, 11)]
                for i, s in zip((0, 11), single):
                    assert all(a.tobytes() == b.tobytes() for a, b in zip(s, want[k][i]))
        except Exception as e:       # surfaced below
            errors.append(e)

    ts = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
    for k in range(2):
        for i in range(12):
            assert_frame(got[k], want[k][i], i)


def test_snippet_on_the_gpu(tmp_path):
    """The INTEGRATION.md Frame body gives the Python call's bytes."""
    build_snippet()
    out = str(tmp_path / "rgbd.bin")
    subprocess.run([SNIPPET_EXE, "9", out], check=True, capture_output=True, text=True)
    raw = np.fromfile(out, np.uint8)
    n = int(raw[:4].view(np.int32)[0])
    cols, rows = 640, 480
    img = synth.image(9, cols, rows)
    y, x = np.mgrid[0:rows, 0:cols]
    dep = (1000 + y * 97 + x).astype(np.uint16)
    dep[(x + y) % 7 == 0] = 0
    want = orbx.extract_rgbd(orbx.ORBextractor(1000, 1.2, 8, 20, 7), img, dep, K, TUM1, BF, np.float32(1) / np.float32(5000))
    assert n == len(want[0]) > 100
    off = 4
    for w in want:
        b = w.tobytes()
        assert raw[off:off + len(b)].tobytes() == b
        off += len(b)
    assert off == len(raw)
    assert os.path.exists(SNIPPET_EXE)
