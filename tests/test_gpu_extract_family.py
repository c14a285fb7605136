"""One handle through every kind of extraction call in turn.  Each call grows slot staging that a call of another kind used
before it, one of them while a device batch on a caller's stream may still be running.  Every result equals the same call on a
fresh handle, bit for bit: counts, and keypoints, descriptors, mvuRight, mvDepth and mvKeysUn over the rows each frame has."""
import ctypes as C

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from wut_cuda_orb_slam3_b200 import synth
from wut_cuda_orb_slam3_b200.capi import KP_DTYPE, check, lib, ptr

pytestmark = pytest.mark.gpu

NF, MAX_BATCH = 1000, 8
SMALL, BIG = (320, 240), (640, 480)                    # (cols, rows)
BF, MAX_D = 47.9, 47.9 / 0.11
K = np.array([517.306408, 516.469215, 318.643040, 255.313989], np.float32)
TUM1 = [0.262383, -0.953104, -0.005358, 0.002628, 1.163314]


def handle():
    return orbx.ORBextractor(NF, 1.2, 8, 20, 7, max_batch=MAX_BATCH)


def assert_same(got, want):
    """got / want: lists of (counts[F], slab[F, capacity, ...]); slab rows past a frame's count are not compared."""
    assert len(got) == len(want)
    for (gn, gs), (wn, ws) in zip(got, want):
        gn, wn = np.asarray(gn), np.asarray(wn)
        assert np.array_equal(gn, wn), (gn, wn)
        for i, a in enumerate(gn):
            assert gs[i, :a].tobytes() == ws[i, :a].tobytes(), i


def single(ex, img):
    _, kps, desc = ex(img) if img.ndim == 2 else ex.extract_color(img, rgb=True)
    n = [len(kps)]
    return [(n, kps[None]), (n, desc[None])]


def mono_host(ex, imgs):
    _, n, kps, desc = ex.extract_batch(imgs)
    return [(n, kps), (n, desc)]


def stereo_host(ex, left, right, cap):
    N, rows, cols = left.shape
    kL = np.zeros((N, cap), KP_DTYPE); kR = np.zeros((N, cap), KP_DTYPE)
    dL = np.zeros((N, cap, 32), np.uint8); dR = np.zeros((N, cap, 32), np.uint8)
    u = np.zeros((N, cap), np.float32); d = np.zeros((N, cap), np.float32)
    nL = np.zeros(N, np.int32); nR = np.zeros(N, np.int32)
    pl = (C.c_void_p * N)(*[left.ctypes.data + i * left.strides[0] for i in range(N)])
    pr = (C.c_void_p * N)(*[right.ctypes.data + i * right.strides[0] for i in range(N)])
    check(lib().orbx_extract_stereo_batch(ex._h, pl, pr, N, rows, cols, cols, BF, MAX_D, ptr(kL), ptr(dL), ptr(nL), ptr(kR), ptr(dR),
                                          ptr(nR), cap, ptr(u), ptr(d)))
    return [(nL, kL), (nL, dL), (nR, kR), (nR, dR), (nL, u), (nL, d)]


def rgbd_host(ex, imgs, deps):
    n, kp, kp_un, desc, u, d = ex.extract_rgbd_batch(imgs, deps, K, TUM1, BF, 1.0)
    return [(n, kp), (n, kp_un), (n, desc), (n, u), (n, d)]


class Device:
    """Output slabs of a device batch on the GPU, read back once the caller's stream is done.  They are zeroed on torch's current
    stream: a batch on no stream (the handle's own) must not start before that."""

    def __init__(self, torch, n, cap, names, stream):
        dev = torch.device("cuda", 0)
        self.t = {}
        for k in names:
            if k.startswith("n"):
                self.t[k] = torch.zeros(n, dtype=torch.int32, device=dev)
            elif k.startswith("kp"):
                self.t[k] = torch.zeros((n, cap * KP_DTYPE.itemsize), dtype=torch.uint8, device=dev)
            elif k.startswith("desc"):
                self.t[k] = torch.zeros((n, cap, 32), dtype=torch.uint8, device=dev)
            else:
                self.t[k] = torch.zeros((n, cap), dtype=torch.float32, device=dev)
        if stream is None:
            torch.cuda.synchronize()

    def read(self, pairs):
        h = {k: v.cpu().numpy() for k, v in self.t.items()}
        for k in h:
            if k.startswith("kp"):
                h[k] = h[k].view(KP_DTYPE).reshape(h[k].shape[0], -1)
        return [(h[c], h[s]) for c, s in pairs]


def mono_device(torch, ex, d_imgs, cap, stream):
    n, rows, cols = d_imgs.shape
    o = Device(torch, n, cap, ("n", "nm", "kp", "desc"), stream)
    ex.extract_batch_device(d_imgs, n, rows, cols, cols, rows * cols, o.t["kp"], o.t["desc"], cap, o.t["n"], o.t["nm"], stream=stream)
    return lambda: o.read([("n", "kp"), ("n", "desc")])


def stereo_device(torch, ex, d_left, d_right, cap, stream):
    n, rows, cols = d_left.shape
    o = Device(torch, n, cap, ("nL", "nR", "kpL", "kpR", "descL", "descR", "u", "d"), stream)
    t = o.t
    ex.extract_stereo_batch_device(d_left, d_right, n, rows, cols, cols, rows * cols, BF, MAX_D, t["kpL"], t["descL"], t["nL"], t["kpR"],
                                   t["descR"], t["nR"], cap, t["u"], t["d"], stream=stream)
    return lambda: o.read([("nL", "kpL"), ("nL", "descL"), ("nR", "kpR"), ("nR", "descR"), ("nL", "u"), ("nL", "d")])


def rgbd_device(torch, ex, d_imgs, d_deps, cap, stream):
    n, rows, cols = d_imgs.shape
    o = Device(torch, n, cap, ("n", "kp", "kp_un", "desc", "u", "d"), stream)
    t = o.t
    ex.extract_rgbd_batch_device(d_imgs, d_deps, n, rows, cols, cols, rows * cols, 0, cols * 2, rows * cols * 2, K, TUM1, BF, 1.0 / 5000,
                                 t["kp"], t["kp_un"], t["desc"], cap, t["n"], t["u"], t["d"], stream=stream)
    return lambda: o.read([("n", "kp"), ("n", "kp_un"), ("n", "desc"), ("n", "u"), ("n", "d")])


def grey(seed, cols, rows, n=None, view=0):
    if n is None:
        return synth.image(seed, cols, rows, view=view, max_disp=40)
    return np.stack([synth.image(seed + i, cols, rows, view=view, max_disp=40) for i in range(n)])


def color(seed, cols, rows, ch):
    return np.ascontiguousarray(np.stack([synth.image(seed + c, cols, rows) for c in range(ch)], axis=2))


def test_every_kind_of_call_on_one_handle():
    import torch
    dev = torch.device("cuda", 0)
    cols, rows = BIG
    ex = handle()
    cap = ex.max_keypoints(rows, cols)
    stream = torch.cuda.Stream(device=dev)
    got, want = [], []

    def step(call):                  # the same call on the shared handle and on a fresh one
        got.append(call(ex)); want.append(call(handle()))

    step(lambda h: single(h, grey(1, *SMALL)))
    step(lambda h: single(h, color(2, cols, rows, 3)))
    step(lambda h: mono_host(h, grey(10, cols, rows, n=20)))

    # a device batch on the caller's stream behind a long kernel, then at once a stereo host batch with more pairs and a larger
    # capacity: its staging grows while the device batch may still be running
    d_imgs = torch.from_numpy(grey(40, cols, rows, n=12)).to(dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        big = torch.randn(4096, 4096, device=dev)
        for _ in range(4):
            big = big @ big.T / 4096.0
        shared = mono_device(torch, ex, d_imgs, cap, stream.cuda_stream)
    left, right = grey(60, cols, rows, n=14), grey(60, cols, rows, n=14, view=1)
    step(lambda h: stereo_host(h, left, right, cap + 64))
    fresh = mono_device(torch, handle(), d_imgs, cap, None)
    torch.cuda.synchronize()
    got.append(shared()); want.append(fresh())

    d_left, d_right = torch.from_numpy(grey(80, cols, rows, n=6)).to(dev), torch.from_numpy(grey(80, cols, rows, n=6, view=1)).to(dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        shared = stereo_device(torch, ex, d_left, d_right, cap, stream.cuda_stream)
    fresh = stereo_device(torch, handle(), d_left, d_right, cap, None)
    rng = np.random.default_rng(5)
    deps = (rng.integers(0, 20000, (10, rows, cols)) / 5000.0).astype(np.float32)     # f32 maps: twice the bytes of u16
    step(lambda h: rgbd_host(h, grey(100, cols, rows, n=10), deps))
    torch.cuda.synchronize()
    got.append(shared()); want.append(fresh())

    d_imgs = torch.from_numpy(grey(120, cols, rows, n=9)).to(dev)
    d_deps = torch.from_numpy(rng.integers(0, 20000, (9, rows, cols)).astype(np.int16)).to(dev)
    torch.cuda.synchronize()
    with torch.cuda.stream(stream):
        shared = rgbd_device(torch, ex, d_imgs, d_deps, cap, stream.cuda_stream)
    fresh = rgbd_device(torch, handle(), d_imgs, d_deps, cap, None)
    step(lambda h: single(h, grey(3, cols, rows)))     # waits for the device batch on the caller's stream (no sync)
    torch.cuda.synchronize()
    got.append(shared()); want.append(fresh())

    for g, w in zip(got, want):
        assert_same(g, w)
    assert all(g[0][0][0] > 100 for g in got)          # every call found features in its first frame


def test_color_frames_of_growing_size():
    ex = handle()
    for cols, rows in (SMALL, BIG):
        for ch in (3, 4):                  # at one shape, a four-channel image replaces the colour staging of a three-channel one
            img = color(7 * ch + cols, cols, rows, ch)
            assert_same(single(ex, img), single(handle(), img))
