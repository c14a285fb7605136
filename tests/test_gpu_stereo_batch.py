"""Stereo batches (orbx_extract_stereo_batch / orbx_extract_stereo_batch_device): for every pair the batch returns exactly what
orbx_extract_stereo returns for that pair (keypoint bytes, descriptors, counts, mvuRight / mvDepth over the first nL rows), and
the first and last pair of a batch equal the CPU oracle's Frame::ComputeStereoMatches."""
import ctypes as C
import threading

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from wut_cuda_orb_slam3_b200 import capi, synth
from wut_cuda_orb_slam3_b200.capi import KP_DTYPE, lib, ptr

pytestmark = pytest.mark.gpu

BF = 47.9
MAX_D = 47.9 / 0.11
SHAPES = [(752, 480, 1200), (1241, 376, 2000)]       # EuRoC / KITTI stereo shapes of BASELINE.json


def make_pairs(n, cols, rows, seed0=500, pinned=False):
    if pinned:
        import torch
        left = torch.empty((n, rows, cols), dtype=torch.uint8, pin_memory=True).numpy()
        right = torch.empty((n, rows, cols), dtype=torch.uint8, pin_memory=True).numpy()
    else:
        left = np.empty((n, rows, cols), np.uint8); right = np.empty((n, rows, cols), np.uint8)
    for i in range(n):
        left[i] = synth.image(seed0 + i, cols, rows, view=0, max_disp=40)
        right[i] = synth.image(seed0 + i, cols, rows, view=1, max_disp=40)
    return left, right


def reference(nfeatures, left, right):
    """orbx_extract_stereo pair by pair on a fresh pair of handles."""
    exL = orbx.ORBextractor(nfeatures, 1.2, 8, 20, 7); exR = orbx.ORBextractor(nfeatures, 1.2, 8, 20, 7)
    return [orbx.extract_stereo(exL, exR, left[i], right[i], BF, MAX_D) for i in range(len(left))]


def assert_pair(got, want, i):
    nL, nR, kL, dL, kR, dR, u, d = got
    wkL, wdL, wkR, wdR, wu, wd = want
    a, b = nL[i], nR[i]
    assert a == len(wkL) and b == len(wkR), (i, a, b, len(wkL), len(wkR))
    assert kL[i, :a].tobytes() == wkL.tobytes() and kR[i, :b].tobytes() == wkR.tobytes(), i
    assert np.array_equal(dL[i, :a], wdL) and np.array_equal(dR[i, :b], wdR), i
    assert u[i, :a].tobytes() == wu.tobytes() and d[i, :a].tobytes() == wd.tobytes(), i


def assert_oracle(oracle, nfeatures, got, left, right, i):
    nL, nR, kL, dL, kR, dR, u, d = got
    oL = oracle.extractor(nfeatures, 1.2, 8, 20, 7); oR = oracle.extractor(nfeatures, 1.2, 8, 20, 7)
    okL, odL, _ = oL.extract(left[i], (0, 0)); okR, odR, _ = oR.extract(right[i], (0, 0))
    ou, od, kept = oracle.stereo_match(oL, oR, okL, odL, okR, odR, BF, MAX_D)
    a = nL[i]
    assert a == len(okL) and nR[i] == len(okR)
    assert np.array_equal(u[i, :a], ou) and np.array_equal(d[i, :a], od)
    assert kept > 20 and (u[i, :a] >= 0).sum() == kept


def chunk_schedule(n, chunk):
    """api.cu chunk_schedule: (first pair, pairs) per chunk of the host call."""
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


# Batch sizes reach every branch of the host scheduler (checked against the schedule in test_host_cases_reach_every_branch):
# - default chunking, 32 pairs (64 frames; slot streams): 1, 3 and 17 pairs are one chunk each (1 and 3 pairs run
#   fast_cells_kernel, total_cells x frames < 8192; 17 pairs fast_cells_warp_kernel); 40 pairs two chunks; 125 pairs ramp up,
#   ramp down and reuse slots;
# - max_batch = 256: 128-pair chunks (256 frames), the serial three-stream pipeline, 150 pairs = two chunks;
# - max_batch = 128: 64-pair chunks (128 frames), still serial; 300 pairs ramp up, ramp down and reuse slots, so the waits that
#   order a slot's next upload and compute behind its matcher and download run.
HOST_CASES = [(1, 0, False), (3, 0, True), (17, 0, False), (40, 0, True), (125, 0, False), (150, 256, True), (300, 128, True)]


def test_host_cases_reach_every_branch():
    slots = 6
    seen = set()
    for n, max_batch, _ in HOST_CASES:
        frames = min(max_batch, 2 * n) if max_batch else min(2 * n, 64)
        chunk = max(frames // 2, 1)
        s = chunk_schedule(n, chunk)
        assert sum(p for _, p in s) == n and all(0 < p <= chunk for _, p in s)
        serial = 2 * chunk >= 128
        ramp_down = len(s) >= 2 and s[-1][1] < s[-2][1] < chunk
        seen.add((serial, "reuse" if len(s) > slots else "no-reuse", "ramp" if ramp_down else "no-ramp"))
    assert (False, "reuse", "ramp") in seen and (True, "reuse", "ramp") in seen and (True, "no-reuse", "no-ramp") in seen


@pytest.mark.parametrize("cols,rows,nfeatures", SHAPES)
@pytest.mark.parametrize("n,max_batch,pinned", HOST_CASES)
def test_host_batch_matches_extract_stereo(oracle, cols, rows, nfeatures, n, max_batch, pinned):
    left, right = make_pairs(n, cols, rows, seed0=1000 + n, pinned=pinned)
    ex = orbx.ORBextractor(nfeatures, 1.2, 8, 20, 7, max_batch=max_batch)
    got = ex.extract_stereo_batch(left, right, BF, MAX_D)
    want = reference(nfeatures, left, right)
    for i in range(n):
        assert_pair(got, want[i], i)
    assert_oracle(oracle, nfeatures, got, left, right, 0)
    if n > 1:
        assert_oracle(oracle, nfeatures, got, left, right, n - 1)


# 21 pairs in 8-pair chunks: three chunks on the caller's stream, packed by pack_kernel (16 frames); 1 and 3 pairs: one chunk
# of 2 / 6 frames, packed inside orient_describe_kernel (fewer than 8 frames) through both sets of the caller's slabs
@pytest.mark.parametrize("cols,rows,nfeatures", SHAPES)
@pytest.mark.parametrize("n,max_batch", [(21, 16), (3, 0), (1, 0)])
def test_device_batch_on_caller_stream(cols, rows, nfeatures, n, max_batch):
    import torch
    left, right = make_pairs(n, cols, rows, seed0=3000 + n)
    ex = orbx.ORBextractor(nfeatures, 1.2, 8, 20, 7, max_batch=max_batch)
    want = ex.extract_stereo_batch(left, right, BF, MAX_D)
    cap = ex.max_keypoints(rows, cols)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    d_kL = torch.zeros((n, cap * KP_DTYPE.itemsize), dtype=torch.uint8, device=dev)
    d_kR = torch.zeros_like(d_kL)
    d_dL = torch.zeros((n, cap, 32), dtype=torch.uint8, device=dev); d_dR = torch.zeros_like(d_dL)
    d_nL = torch.zeros(n, dtype=torch.int32, device=dev); d_nR = torch.zeros_like(d_nL)
    sentinel = -7.5
    d_u = torch.full((n, cap), sentinel, dtype=torch.float32, device=dev); d_d = torch.full_like(d_u, sentinel)
    with torch.cuda.stream(stream):
        # the inputs are written on the caller's stream, behind a long busy kernel: the call must queue behind both
        big = torch.randn(4096, 4096, device=dev)
        for _ in range(4):
            big = big @ big.T / 4096.0
        d_left = torch.from_numpy(left).to(dev, non_blocking=False)
        d_right = torch.from_numpy(right).to(dev, non_blocking=False)
        ex.extract_stereo_batch_device(d_left, d_right, n, rows, cols, cols, rows * cols, BF, MAX_D, d_kL, d_dL, d_nL, d_kR, d_dR,
                                       d_nR, cap, d_u, d_d, stream=stream.cuda_stream)
    ex.sync()                                # orbx_sync covers the caller's stream
    got = (d_nL.cpu().numpy(), d_nR.cpu().numpy(), d_kL.cpu().numpy().view(KP_DTYPE).reshape(n, cap), d_dL.cpu().numpy(),
           d_kR.cpu().numpy().view(KP_DTYPE).reshape(n, cap), d_dR.cpu().numpy(), d_u.cpu().numpy(), d_d.cpu().numpy())
    nL, nR, kL, dL, kR, dR, u, d = got
    assert np.array_equal(nL, want[0]) and np.array_equal(nR, want[1])
    for i in range(n):
        a, b = nL[i], nR[i]
        assert kL[i, :a].tobytes() == want[2][i, :a].tobytes() and kR[i, :b].tobytes() == want[4][i, :b].tobytes()
        assert np.array_equal(dL[i, :a], want[3][i, :a]) and np.array_equal(dR[i, :b], want[5][i, :b])
        assert u[i, :a].tobytes() == want[6][i, :a].tobytes() and d[i, :a].tobytes() == want[7][i, :a].tobytes()
        assert (u[i, a:] == sentinel).all() and (d[i, a:] == sentinel).all()      # rows past *d_nL untouched
    # probes refuse every frame after a stereo batch (its pyramids are not kept for inspection)
    with pytest.raises(capi.OrbxError):
        ex.pyramid_level(0, frame=0)
    with pytest.raises(capi.OrbxError):
        ex.blurred_level(0, frame=0)
    # ... until the next extraction
    ex(left[0], None, (0, 0))
    assert ex.pyramid_level(0, frame=0).shape == (rows, cols)


def test_probes_refused_after_host_batch():
    cols, rows, nf = SHAPES[0]
    left, right = make_pairs(2, cols, rows, seed0=11)
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    ex.extract_stereo_batch(left, right, BF, MAX_D)
    for frame in (0, 1, 2, 3):
        with pytest.raises(capi.OrbxError):
            ex.pyramid_level(0, frame=frame)
        with pytest.raises(capi.OrbxError):
            ex.candidates(0, frame=frame)
        with pytest.raises(capi.OrbxError):
            ex.level_keypoints(0, frame=frame)


def _raw_call(ex, left, right, n, rows, cols, step, cap, guard=64):
    """orbx_extract_stereo_batch with guard bytes after every slab; returns (rc, outputs, guards intact)."""
    kL = np.full(n * cap * KP_DTYPE.itemsize + guard, 0xA5, np.uint8); kR = kL.copy()
    dL = np.full(n * cap * 32 + guard, 0xA5, np.uint8); dR = dL.copy()
    u = np.full(n * cap * 4 + guard, 0xA5, np.uint8); d = u.copy()
    nL = np.full(n + guard // 4, -3, np.int32); nR = nL.copy()
    pl = (C.c_void_p * max(n, 1))(*[left.ctypes.data + i * left.strides[0] for i in range(n)])
    pr = (C.c_void_p * max(n, 1))(*[right.ctypes.data + i * right.strides[0] for i in range(n)])
    rc = lib().orbx_extract_stereo_batch(ex._h, pl, pr, n, rows, cols, step, BF, MAX_D, ptr(kL), ptr(dL), ptr(nL), ptr(kR), ptr(dR),
                                         ptr(nR), cap, ptr(u), ptr(d))
    intact = all((a[-guard:] == 0xA5).all() for a in (kL, kR, dL, dR, u, d)) and (nL[n:] == -3).all() and (nR[n:] == -3).all()
    return rc, (nL[:n], nR[:n], u[:n * cap * 4].view(np.float32).reshape(n, cap), d[:n * cap * 4].view(np.float32).reshape(n, cap)), intact


def test_capacity_too_small_keeps_guards():
    cols, rows, nf = SHAPES[0]
    left, right = make_pairs(5, cols, rows, seed0=40)
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    rc, (nL, nR, _, _), intact = _raw_call(ex, left, right, 5, rows, cols, cols, 200)
    assert rc == capi.ORBX_ERR_CAPACITY and intact
    assert (np.maximum(nL, nR) > 200).any()
    # a capacity that fits leaves the guards intact too
    rc, _, intact = _raw_call(ex, left, right, 5, rows, cols, cols, ex.max_keypoints(rows, cols))
    assert rc == capi.ORBX_OK and intact


def test_featureless_right_and_identical_pair():
    cols, rows, nf = SHAPES[0]
    left, _ = make_pairs(2, cols, rows, seed0=60)
    right = np.stack([np.full((rows, cols), 128, np.uint8), left[1]])          # pair 0: no right keypoints; pair 1: L == R
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    got = ex.extract_stereo_batch(left, right, BF, MAX_D)
    nL, nR, _, _, _, _, u, d = got
    assert nR[0] == 0 and nL[0] > 0
    assert (u[0, :nL[0]] == -1).all() and (d[0, :nL[0]] == -1).all()
    # L == R: every keypoint finds itself at disparity ~0 with SAD 0, so the median SAD is 0 and the filter of
    # src/Frame.cc:1001-1009 (keep SAD < 1.5 * 1.4 * median) rejects every match, as in the reference.  The values the
    # disparity <= 0 branch writes are checked by test_zero_disparity_branch_values.
    assert nL[1] == nR[1] and (u[1, :nL[1]] == -1).all() and (d[1, :nL[1]] == -1).all()
    want = reference(nf, left, right)
    for i in range(2):
        assert_pair(got, want[i], i)


def test_zero_pairs_and_bad_arguments():
    cols, rows, nf = 320, 240, 500
    ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    img = synth.image(1, cols, rows)
    cap = ex.max_keypoints(rows, cols)
    one = (C.c_void_p * 1)(img.ctypes.data)
    null1 = (C.c_void_p * 1)(None)
    kp = np.zeros(cap, KP_DTYPE); de = np.zeros((cap, 32), np.uint8); n = np.zeros(1, np.int32); f = np.zeros(cap, np.float32)
    L = lib().orbx_extract_stereo_batch

    def call(h=ex._h, il=one, ir=one, np_=1, r=rows, c=cols, step=cols, outs=True, capacity=cap):
        o = [ptr(kp), ptr(de), ptr(n), ptr(kp), ptr(de), ptr(n)] if outs else [None] * 6
        return L(h, il, ir, np_, r, c, step, BF, MAX_D, *o, capacity, ptr(f) if outs else None, ptr(f) if outs else None)

    assert call(np_=0) == capi.ORBX_OK
    assert call(np_=0, il=None, ir=None, outs=False) == capi.ORBX_OK
    assert call() == capi.ORBX_OK
    assert call(h=None) == capi.ORBX_ERR_INVALID_ARG
    assert call(np_=-1) == capi.ORBX_ERR_INVALID_ARG
    assert call(il=None) == capi.ORBX_ERR_EMPTY_IMAGE
    assert call(ir=null1) == capi.ORBX_ERR_EMPTY_IMAGE
    assert call(r=0) == capi.ORBX_ERR_EMPTY_IMAGE
    assert call(c=0) == capi.ORBX_ERR_EMPTY_IMAGE
    assert call(outs=False) == capi.ORBX_ERR_INVALID_ARG
    assert call(step=cols - 1) == capi.ORBX_ERR_INVALID_ARG
    assert call(capacity=0) == capi.ORBX_ERR_INVALID_ARG
    assert call(capacity=1 << 20) == capi.ORBX_ERR_UNSUPPORTED
    D = lib().orbx_extract_stereo_batch_device
    import torch
    dev = torch.device("cuda", 0)
    di = torch.zeros(rows * cols, dtype=torch.uint8, device=dev)
    dk = torch.zeros(cap * KP_DTYPE.itemsize, dtype=torch.uint8, device=dev); dd = torch.zeros(cap * 32, dtype=torch.uint8, device=dev)
    dn = torch.zeros(1, dtype=torch.int32, device=dev); dfl = torch.zeros(cap, dtype=torch.float32, device=dev)

    def dcall(h=ex._h, il=di, ir=di, np_=1, pitch=cols, outs=True, capacity=cap):
        o = [ptr(dk), ptr(dd), ptr(dn), ptr(dk), ptr(dd), ptr(dn)] if outs else [None] * 6
        return D(h, ptr(il) if il is not None else None, ptr(ir) if ir is not None else None, rows * cols, np_, rows, cols, pitch, BF,
                 MAX_D, *o, capacity, ptr(dfl) if outs else None, ptr(dfl) if outs else None, None)

    assert dcall(np_=0) == capi.ORBX_OK
    assert dcall(h=None) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(np_=-2) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(il=None) == capi.ORBX_ERR_EMPTY_IMAGE
    assert dcall(outs=False) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(pitch=cols - 1) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(capacity=-1) == capi.ORBX_ERR_INVALID_ARG
    assert dcall(capacity=1 << 20) == capi.ORBX_ERR_UNSUPPORTED
    assert dcall() == capi.ORBX_OK
    ex.sync()


def test_handle_state_after_stereo_batch():
    """A stereo batch leaves the handle as good as new for orbx_extract, orbx_extract_batch and orbx_extract_stereo."""
    cols, rows, nf = SHAPES[0]
    left, right = make_pairs(9, cols, rows, seed0=90)
    used = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    other = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
    used.extract_stereo_batch(left, right, BF, MAX_D)
    img = synth.image(5, cols, rows)
    nm, k, dsc = used(img, None, (0, 0))
    fnm, fk, fd = orbx.ORBextractor(nf, 1.2, 8, 20, 7)(img, None, (0, 0))
    assert nm == fnm and k.tobytes() == fk.tobytes() and np.array_equal(dsc, fd)
    used.extract_stereo_batch(left, right, BF, MAX_D)
    b = used.extract_batch(left)
    fb = orbx.ORBextractor(nf, 1.2, 8, 20, 7).extract_batch(left)
    assert all(np.array_equal(x, y) for x, y in zip(b[:2], fb[:2]))
    for i in range(len(left)):
        assert b[2][i, :b[1][i]].tobytes() == fb[2][i, :fb[1][i]].tobytes() and np.array_equal(b[3][i, :b[1][i]], fb[3][i, :fb[1][i]])
    used.extract_stereo_batch(left, right, BF, MAX_D)
    s = orbx.extract_stereo(used, other, left[3], right[3], BF, MAX_D)
    fs = orbx.extract_stereo(orbx.ORBextractor(nf, 1.2, 8, 20, 7), orbx.ORBextractor(nf, 1.2, 8, 20, 7), left[3], right[3], BF, MAX_D)
    assert all(x.tobytes() == y.tobytes() for x, y in zip(s, fs))


def test_two_handles_on_two_threads():
    cols, rows, nf = SHAPES[1]
    sets = [make_pairs(12, cols, rows, seed0=s) for s in (200, 300)]
    want = [orbx.ORBextractor(nf, 1.2, 8, 20, 7).extract_stereo_batch(l, r, BF, MAX_D) for l, r in sets]
    got = [None, None]
    errors = []

    def run(k):
        try:
            ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
            for _ in range(3):
                got[k] = ex.extract_stereo_batch(sets[k][0], sets[k][1], BF, MAX_D)
        except Exception as e:       # surfaced below
            errors.append(e)

    ts = [threading.Thread(target=run, args=(k,)) for k in range(2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
    for k in range(2):
        nL, nR = want[k][0], want[k][1]
        assert np.array_equal(got[k][0], nL) and np.array_equal(got[k][1], nR)
        for i in range(12):
            a, b = nL[i], nR[i]
            assert got[k][2][i, :a].tobytes() == want[k][2][i, :a].tobytes()
            assert got[k][4][i, :b].tobytes() == want[k][4][i, :b].tobytes()
            assert got[k][6][i, :a].tobytes() == want[k][6][i, :a].tobytes()
            assert got[k][7][i, :a].tobytes() == want[k][7][i, :a].tobytes()


def test_zero_disparity_branch_values(oracle):
    """The disparity <= 0 branch of src/Frame.cc:983-986 (uR = uL - 0.01, depth = bf / 0.01) on matches that survive the median
    filter.  Each left keypoint sits on a column about which both images are mirror-symmetric in the SAD window, and the right
    image is the left one + 1: the SAD profile is symmetric (sub-pixel offset exactly 0) with its minimum, 121, at the keypoint's
    own column, so the disparity is exactly 0; every match has SAD 121, which the median filter keeps."""
    cols, rows = 752, 480
    rng = np.random.default_rng(77)
    left = rng.integers(10, 240, (rows, cols)).astype(np.uint8)
    pts = [(100 + 60 * k, 40 + 36 * k) for k in range(10)]
    for c, r in pts:
        for dx in range(1, 13):
            left[r - 6:r + 7, c + dx] = left[r - 6:r + 7, c - dx]
    right = left + 1
    exL = orbx.ORBextractor(1200, 1.2, 8, 20, 7); exR = orbx.ORBextractor(1200, 1.2, 8, 20, 7)
    exL(left, None, (0, 0)); exR(right, None, (0, 0))           # the matcher reads these pyramids
    kp = np.zeros(len(pts), KP_DTYPE)
    kp["x"] = [c for c, _ in pts]; kp["y"] = [r for _, r in pts]; kp["size"] = 31; kp["octave"] = 0; kp["class_id"] = -1
    desc = rng.integers(0, 256, (len(pts), 32)).astype(np.uint8)
    u, d = orbx.compute_stereo_matches(exL, exR, kp, desc, kp.copy(), desc.copy(), BF, MAX_D)
    assert np.array_equal(u, np.float32(kp["x"].astype(np.float64) - 0.01))
    assert np.array_equal(d, np.full(len(pts), np.float32(BF) / np.float32(0.01)))
    oL = oracle.extractor(1200, 1.2, 8, 20, 7); oR = oracle.extractor(1200, 1.2, 8, 20, 7)
    oL.extract(left, (0, 0)); oR.extract(right, (0, 0))
    ou, od, kept = oracle.stereo_match(oL, oR, kp, desc, kp.copy(), desc.copy(), BF, MAX_D)
    assert kept == len(pts) and np.array_equal(u, ou) and np.array_equal(d, od)
