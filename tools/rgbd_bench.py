"""RGB-D frames on one GPU: orbx_extract_rgbd against the sequence it replaces, and the batches against the plain extraction
batches over the same frames.  Writes profiles/r09_rgbd.txt (or the path given with --out).

  * single frame, 640x480 / 1000 features, a colour (BGR) image and a raw u16 depth map (TUM, 5000 per metre), pageable and
    page-locked host buffers: orbx_extract_rgbd against orbx_extract_color + orbx_undistort_keypoints + the CPU convertTo of the
    whole map (numpy, one pass into a preallocated map) + the per-keypoint lookup of ComputeStereoFromRGBD.  Host clock around calls
    that end synchronised, median of --single-reps, the two alternated.
  * resident, per 512 frames: orbx_extract_rgbd_batch_device against orbx_extract_batch_device on the same device frames (CUDA
    events); rgbd_frame_kernel's own device time from torch.profiler in a separate pass.
  * host-fed, per 512 frames: orbx_extract_rgbd_batch against orbx_extract_batch from page-locked buffers, with H2D bytes per frame
    and the measured pinned H2D ceiling of the box.

Fails (exit 1) unless the batches equal the single-frame call on the first and last frame."""
import argparse
import ctypes as C
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import wut_cuda_orb_slam3_b200 as orbx  # noqa: E402
from wut_cuda_orb_slam3_b200 import synth  # noqa: E402
from wut_cuda_orb_slam3_b200.capi import KP_DTYPE, check, lib, ptr  # noqa: E402
from wut_cuda_orb_slam3_b200.prep import rgbd_calib  # noqa: E402

COLS, ROWS, NFEAT = 640, 480, 1000
K = np.array([517.306408, 516.469215, 318.643040, 255.313989], np.float32)
DIST = np.array([0.262383, -0.953104, -0.005358, 0.002628, 1.163314], np.float32)
BF, FACTOR = 40.0, np.float32(1) / np.float32(5000)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except Exception as e:       # reported, not fatal
        return "%s (nvidia-smi unavailable: %s)" % (torch.cuda.get_device_name(0), e)


def depth_map(seed):
    rng = np.random.default_rng(seed)
    d = rng.integers(2000, 20000, (ROWS, COLS)).astype(np.uint16)
    d[rng.random((ROWS, COLS)) < 0.1] = 0
    return d


def timed(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_rgbd.txt"))
    ap.add_argument("--single-reps", type=int, default=300)
    ap.add_argument("--frames", type=int, default=512)
    ap.add_argument("--reps", type=int, default=10)
    a = ap.parse_args()
    conv_buf = np.empty((ROWS, COLS), np.float32)

    def convert(d):                                         # convertTo(CV_32F, f): one pass, preallocated output
        return np.multiply(d, FACTOR, out=conv_buf, dtype=np.float32)
    conv_name = "numpy multiply into a preallocated float32 map, one pass"
    lines = ["# RGB-D frames (tools/rgbd_bench.py)", "GPU: " + gpu_info(), "torch %s, CUDA %s" % (torch.__version__, torch.version.cuda), ""]

    # ---- single frame -------------------------------------------------------------------------------------------------
    ex = orbx.ORBextractor(NFEAT, 1.2, 8, 20, 7)
    cap = ex.max_keypoints(ROWS, COLS)
    calib, _keep = rgbd_calib(K, DIST, BF, FACTOR)
    color = np.ascontiguousarray(np.stack([synth.image(s, COLS, ROWS) for s in (1, 2, 3)], axis=2))
    dep = depth_map(0)
    kp = np.zeros(cap, KP_DTYPE); kpu = kp.copy(); desc = np.zeros((cap, 32), np.uint8)
    u = np.zeros(cap, np.float32); z = u.copy()
    n = C.c_int(0); nm = C.c_int(0)
    kpu2 = kp.copy()

    def one_call(im, dp, kp, kpu, desc, u, z):
        check(lib().orbx_extract_rgbd(ex._h, ptr(im), ROWS, COLS, COLS * 3, 3, 0, ptr(dp), 0, COLS * 2, C.byref(calib), ptr(kp), ptr(kpu), ptr(desc),
                                      cap, C.byref(n), ptr(u), ptr(z)))

    def sequence(im, dp, kp, kpu, desc, u, z):
        check(lib().orbx_extract_color(ex._h, ptr(im), ROWS, COLS, COLS * 3, 3, 0, 0, 0, ptr(kp), ptr(desc), cap, C.byref(n), C.byref(nm)))
        N = n.value
        check(lib().orbx_undistort_keypoints(0, ptr(kp), N, ptr(K), ptr(DIST), len(DIST), ptr(K), ptr(kpu)))
        m = convert(dp)                                     # GrabImageRGBD's convertTo of the whole map
        k = kp[:N]
        d = m[k["y"].astype(np.int32), k["x"].astype(np.int32)]
        ok = d > 0
        z[:N] = np.where(ok, d, np.float32(-1))
        u[:N] = np.where(ok, kpu[:N]["x"] - np.float32(BF) / np.where(ok, d, np.float32(1)), np.float32(-1))

    def pinned_copy(x):
        t = torch.empty(x.nbytes, dtype=torch.uint8, pin_memory=True).numpy().view(x.dtype).reshape(x.shape)
        t[...] = x
        return t

    ok_all = True
    for label, mk in (("pageable", lambda x: x.copy()), ("pinned", pinned_copy)):
        im, dp = mk(color), mk(dep)
        outs1 = [mk(a) for a in (kp, kpu, desc, u, z)]
        outs2 = [mk(a) for a in (kp, kpu2, desc, u, z)]
        for _ in range(20):
            one_call(im, dp, *outs1); sequence(im, dp, *outs2)
        n1 = n.value
        one_call(im, dp, *outs1)
        sequence(im, dp, *outs2)
        same = all(outs1[j][:n1].tobytes() == outs2[j][:n1].tobytes() for j in range(5))
        ok_all &= same
        t1, t2 = [], []
        for _ in range(a.single_reps):
            s = time.perf_counter(); one_call(im, dp, *outs1); t1.append(time.perf_counter() - s)
            s = time.perf_counter(); sequence(im, dp, *outs2); t2.append(time.perf_counter() - s)
        m1, m2 = statistics.median(t1) * 1e3, statistics.median(t2) * 1e3
        lines.append("single frame %dx%d / %d, BGR + u16 depth, %s host buffers (%d keypoints, outputs equal: %s):" % (COLS, ROWS, NFEAT, label, n1, same))
        lines.append("  orbx_extract_rgbd                                         median %.3f ms  (p10 %.3f, p90 %.3f)" %
                     (m1, np.percentile(t1, 10) * 1e3, np.percentile(t1, 90) * 1e3))
        lines.append("  extract_color + undistort_keypoints + CPU convert + lookup  median %.3f ms  (p10 %.3f, p90 %.3f)" %
                     (m2, np.percentile(t2, 10) * 1e3, np.percentile(t2, 90) * 1e3))
        lines.append("  one call / sequence = %.3f" % (m1 / m2))
    lines.append("  (CPU conversion: %s)" % conv_name)
    lines.append("")

    # ---- resident batches -----------------------------------------------------------------------------------------------
    F = a.frames
    dev = torch.device("cuda", 0)
    d_img = torch.empty((F, ROWS, COLS), dtype=torch.uint8, device=dev)
    synth.images_device(d_img, 900, F, COLS, ROWS, COLS, ROWS * COLS)
    h_dep = np.stack([depth_map(i) for i in range(F)])
    d_dep = torch.from_numpy(h_dep.view(np.int16)).to(dev)
    bx = orbx.ORBextractor(NFEAT, 1.2, 8, 20, 7, max_batch=256)
    d_kp = torch.empty((F, cap * 28), dtype=torch.uint8, device=dev); d_kpu = torch.empty_like(d_kp)
    d_desc = torch.empty((F, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.empty(F, dtype=torch.int32, device=dev); d_nm = torch.empty_like(d_n)
    d_u = torch.empty((F, cap), dtype=torch.float32, device=dev); d_z = torch.empty_like(d_u)
    tst = torch.cuda.Stream(device=dev)                     # the calls and the events on one caller stream
    st = tst.cuda_stream

    def rgbd_dev():
        bx.extract_rgbd_batch_device(d_img, d_dep, F, ROWS, COLS, COLS, ROWS * COLS, 0, COLS * 2, ROWS * COLS * 2, K, DIST, BF, FACTOR, d_kp, d_kpu,
                                     d_desc, cap, d_n, d_u, d_z, stream=st)

    def mono_dev():
        bx.extract_batch_device(d_img, F, ROWS, COLS, COLS, ROWS * COLS, d_kp, d_desc, cap, d_n, d_nm, stream=st)

    tr, tm = [], []
    with torch.cuda.stream(tst):
        for _ in range(3):
            tr.append(timed(rgbd_dev, a.reps)); tm.append(timed(mono_dev, a.reps))
        rgbd_dev()
    torch.cuda.synchronize()
    cnt = d_n.cpu().numpy()
    r_ms, m_ms = min(tr), min(tm)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof, torch.cuda.stream(tst):
        for _ in range(5):
            rgbd_dev()
        torch.cuda.synchronize()
    kus = [e.device_time_total / e.count for e in prof.key_averages() if "rgbd_frame_kernel" in e.key]
    lines.append("resident, %d frames of %dx%d / %d (max_batch 256; %.0f keypoints per frame on average):" % (F, COLS, ROWS, NFEAT, cnt.mean()))
    lines.append("  orbx_extract_rgbd_batch_device   %.3f ms per call  (%.1f us per frame)" % (r_ms, r_ms * 1e3 / F))
    lines.append("  orbx_extract_batch_device        %.3f ms per call  (%.1f us per frame)" % (m_ms, m_ms * 1e3 / F))
    lines.append("  difference                       %.3f ms per call  (best of 3 x %d calls each, alternated)" % (r_ms - m_ms, a.reps))
    lines.append("  rgbd_frame_kernel (torch.profiler, separate pass)   %s us per call" % (", ".join("%.1f" % k for k in kus) or "not found"))
    # spot check: frames 0 and F - 1 against the single-frame call
    sx = orbx.ORBextractor(NFEAT, 1.2, 8, 20, 7)
    h_img = d_img.cpu().numpy()
    kpa = d_kp.cpu().numpy().view(KP_DTYPE).reshape(F, cap); ua = d_u.cpu().numpy(); za = d_z.cpu().numpy()
    for i in (0, F - 1):
        w = orbx.extract_rgbd(sx, h_img[i], h_dep[i], K, DIST, BF, FACTOR)
        ok_all &= bool(cnt[i] == len(w[0]) and kpa[i, :cnt[i]].tobytes() == w[0].tobytes() and ua[i, :cnt[i]].tobytes() == w[3].tobytes()
                       and za[i, :cnt[i]].tobytes() == w[4].tobytes())
    lines.append("")

    # ---- host-fed batches -------------------------------------------------------------------------------------------------
    p_img = torch.empty((F, ROWS, COLS), dtype=torch.uint8, pin_memory=True); p_img.copy_(torch.from_numpy(h_img))
    p_dep = torch.empty((F, ROWS, COLS), dtype=torch.int16, pin_memory=True); p_dep.copy_(torch.from_numpy(h_dep.view(np.int16)))
    imgs, deps = p_img.numpy(), p_dep.numpy().view(np.uint16)
    hk = torch.empty((F, cap * 28), dtype=torch.uint8, pin_memory=True).numpy(); hku = torch.empty((F, cap * 28), dtype=torch.uint8, pin_memory=True).numpy()
    hd = torch.empty((F, cap, 32), dtype=torch.uint8, pin_memory=True).numpy()
    hu = torch.empty((F, cap), dtype=torch.float32, pin_memory=True).numpy(); hz = torch.empty((F, cap), dtype=torch.float32, pin_memory=True).numpy()
    hn = np.zeros(F, np.int32); hnm = np.zeros(F, np.int32)
    pi = (C.c_void_p * F)(*[imgs.ctypes.data + i * imgs.strides[0] for i in range(F)])
    pd = (C.c_void_p * F)(*[deps.ctypes.data + i * deps.strides[0] for i in range(F)])
    hx = orbx.ORBextractor(NFEAT, 1.2, 8, 20, 7, max_batch=256)

    def rgbd_host():
        check(lib().orbx_extract_rgbd_batch(hx._h, pi, pd, F, ROWS, COLS, COLS, 0, COLS * 2, C.byref(calib), ptr(hk), ptr(hku), ptr(hd), cap, ptr(hn),
                                            ptr(hu), ptr(hz)))

    def mono_host():
        check(lib().orbx_extract_batch(hx._h, pi, F, ROWS, COLS, COLS, 0, 0, ptr(hk), ptr(hd), cap, ptr(hn), ptr(hnm)))

    th, tmh = [], []
    for _ in range(a.reps):
        s = time.perf_counter(); rgbd_host(); th.append(time.perf_counter() - s)
        s = time.perf_counter(); mono_host(); tmh.append(time.perf_counter() - s)
    rgbd_host()
    ok_all &= bool(np.array_equal(hn, cnt) and hu[0, :cnt[0]].tobytes() == ua[0, :cnt[0]].tobytes())
    # pinned H2D ceiling of the box: one large copy from page-locked memory
    big = torch.empty(1 << 30, dtype=torch.uint8, pin_memory=True)
    dbig = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    h2d = min(timed(lambda: dbig.copy_(big, non_blocking=True), 5) for _ in range(3))
    ceil = (1 << 30) / (h2d * 1e-3)
    rh, mh = statistics.median(th) * 1e3, statistics.median(tmh) * 1e3
    bpf_r, bpf_m = ROWS * COLS * 3, ROWS * COLS
    lines.append("host-fed, %d frames from page-locked buffers (max_batch 256, serial pipeline; median of %d, alternated):" % (F, a.reps))
    lines.append("  orbx_extract_rgbd_batch   %.3f ms  (%.0f frames/s; H2D %d bytes per frame -> %.1f GB/s of input)" %
                 (rh, F / rh * 1e3, bpf_r, bpf_r * F / (rh * 1e-3) / 1e9))
    lines.append("  orbx_extract_batch        %.3f ms  (%.0f frames/s; H2D %d bytes per frame -> %.1f GB/s of input)" %
                 (mh, F / mh * 1e3, bpf_m, bpf_m * F / (mh * 1e-3) / 1e9))
    lines.append("  pinned H2D ceiling (1 GiB copy, best of 3 x 5): %.1f GB/s -> %.3f ms for the RGB-D batch's %d input bytes" %
                 (ceil / 1e9, bpf_r * F / ceil * 1e3, bpf_r * F))
    lines.append("")
    lines.append("batches equal the single-frame call: %s" % ok_all)
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(text)
    print(text)
    return 0 if ok_all else 1


if __name__ == "__main__":
    sys.exit(main())
