"""Stereo batch throughput: orbx_extract_stereo_batch(_device) against a loop of orbx_extract_stereo, at the EuRoC and KITTI
stereo shapes, on one GPU.  Writes profiles/r06_stereo_batch.txt (or the path given with --out).

  * resident: device-generated pairs (orbx_synth_images_device, views 0 and 1), orbx_extract_stereo_batch_device, 64 / 256 / 512 pairs
  * end to end: the same pairs from page-locked host buffers through orbx_extract_stereo_batch
  * loop: the same pairs through orbx_extract_stereo, one call per pair (two handles), into page-locked slabs of the same layout
  * end to end, serial: the same with max_batch = 256 (128-pair chunks: the serial three-stream pipeline)
  * stereo share: the resident stereo batch against orbx_extract_batch_device over the same 2N frames (left images, then right
    images: the same chunks of the same frames), both timed with CUDA events; the difference is the stereo kernels' time
  * kernel split: stereo_match_kernel and stereo_median_kernel device time per resident call, from torch.profiler (a separate
    pass after the timed ones)

Fails (exit 1) unless the batched outputs (host call at both chunkings, and the resident call) equal the looped outputs pair by
pair: counts, and keypoints, descriptors, uRight and depth over the first nL / nR rows."""
import argparse
import ctypes as C
import os
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

BF = 47.9
MAX_D = 47.9 / 0.11
SHAPES = [("EuRoC", 752, 480, 1200), ("KITTI", 1241, 376, 2000)]
SIZES = [64, 256, 512]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except Exception as e:       # reported, not fatal: the numbers still stand with the device name from torch
        return "%s (nvidia-smi unavailable: %s)" % (torch.cuda.get_device_name(0), e)


def timed(fn, reps):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn()
    torch.cuda.synchronize()
    assert torch.cuda.current_stream().cuda_stream != 0
    s.record()
    for _ in range(reps):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_stereo_batch.txt"))
    ap.add_argument("--sizes", default=",".join(map(str, SIZES)))
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    sizes = [int(x) for x in a.sizes.split(",")]
    dev = torch.device("cuda", 0)
    lines = ["# stereo batches (tools/stereo_batch_bench.py): %s" % gpu_info(),
             "# pairs/s; resident = device-generated pairs, e2e = page-locked host pairs in, host slabs out; loop = orbx_extract_stereo per pair",
             "# stereo share = (resident stereo batch - orbx_extract_batch_device over the same 2N frames) / resident stereo batch, CUDA events"]
    ok = True
    for name, cols, rows, nf in SHAPES:
        ex = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
        ex_serial = orbx.ORBextractor(nf, 1.2, 8, 20, 7, max_batch=256)
        exL = orbx.ORBextractor(nf, 1.2, 8, 20, 7); exR = orbx.ORBextractor(nf, 1.2, 8, 20, 7)
        cap = ex.max_keypoints(rows, cols)
        for n in sizes:
            fs = rows * cols
            d_img = torch.empty((2, n, rows, cols), dtype=torch.uint8, device=dev)
            synth.images_device(d_img[0], 900, n, cols, rows, cols, fs, view=0, max_disp=40)
            synth.images_device(d_img[1], 900, n, cols, rows, cols, fs, view=1, max_disp=40)
            kp = torch.empty((2, n, cap * KP_DTYPE.itemsize), dtype=torch.uint8, device=dev)
            de = torch.empty((2, n, cap, 32), dtype=torch.uint8, device=dev)
            cnt = torch.empty((2, n), dtype=torch.int32, device=dev)
            u = torch.empty((2, n, cap), dtype=torch.float32, device=dev)
            nm = torch.empty(2 * n, dtype=torch.int32, device=dev)

            def stereo_dev():
                ex.extract_stereo_batch_device(d_img[0], d_img[1], n, rows, cols, cols, fs, BF, MAX_D, kp[0], de[0], cnt[0], kp[1], de[1],
                                               cnt[1], cap, u[0], u[1], stream=torch.cuda.current_stream().cuda_stream)

            def mono_dev():
                ex.extract_batch_device(d_img, 2 * n, rows, cols, cols, fs, kp, de, cap, cnt, nm, (0, 0),
                                        stream=torch.cuda.current_stream().cuda_stream)

            # alternate the two so drift hits both alike; on a stream of our own (the legacy default stream has handle 0, which the
            # calls read as "the extractor's own stream", where the events would not see the work)
            t_st, t_mono = [], []
            with torch.cuda.stream(torch.cuda.Stream(device=dev)):
                for _ in range(3):
                    t_st.append(timed(stereo_dev, a.reps)); t_mono.append(timed(mono_dev, a.reps))
            ex.sync()
            t_st, t_mono = min(t_st), min(t_mono)
            h = d_img.cpu()
            left = torch.empty((n, rows, cols), dtype=torch.uint8, pin_memory=True); left.copy_(h[0])
            right = torch.empty((n, rows, cols), dtype=torch.uint8, pin_memory=True); right.copy_(h[1])
            L, R = left.numpy(), right.numpy()
            # end to end: page-locked inputs and outputs allocated once, as an offline caller would
            pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()      # noqa: E731
            hk = pin((2, n, cap * KP_DTYPE.itemsize), torch.uint8); hd = pin((2, n, cap, 32), torch.uint8)
            hn = pin((2, n), torch.int32); hu = pin((2, n, cap), torch.float32)
            pl = (C.c_void_p * n)(*[L.ctypes.data + i * L.strides[0] for i in range(n)])
            pr = (C.c_void_p * n)(*[R.ctypes.data + i * R.strides[0] for i in range(n)])

            def stereo_host(h, k, dsc, cn, uu):
                check(lib().orbx_extract_stereo_batch(h._h, pl, pr, n, rows, cols, cols, BF, MAX_D, ptr(k[0]), ptr(dsc[0]), ptr(cn[0]),
                                                      ptr(k[1]), ptr(dsc[1]), ptr(cn[1]), cap, ptr(uu[0]), ptr(uu[1])))

            def host_rate(h, k, dsc, cn, uu):
                stereo_host(h, k, dsc, cn, uu)
                w0 = time.perf_counter()
                for _ in range(a.reps):
                    stereo_host(h, k, dsc, cn, uu)
                return (time.perf_counter() - w0) * 1e3 / a.reps

            sk = pin((2, n, cap * KP_DTYPE.itemsize), torch.uint8); sd = pin((2, n, cap, 32), torch.uint8)
            sn = pin((2, n), torch.int32); su = pin((2, n, cap), torch.float32)
            t_e2e = host_rate(ex, hk, hd, hn, hu)
            t_e2e_serial = host_rate(ex_serial, sk, sd, sn, su)
            # the loop writes the same slab layout into its own page-locked buffers, one orbx_extract_stereo call per pair
            lk = pin((2, n, cap * KP_DTYPE.itemsize), torch.uint8); ld = pin((2, n, cap, 32), torch.uint8)
            ln = pin((2, n), torch.int32); lu = pin((2, n, cap), torch.float32)

            def stereo_one(i):
                check(lib().orbx_extract_stereo(exL._h, exR._h, ptr(L[i]), ptr(R[i]), rows, cols, cols, ptr(lk[0, i]), ptr(ld[0, i]),
                                                ptr(ln[0, i:]), ptr(lk[1, i]), ptr(ld[1, i]), ptr(ln[1, i:]), cap, BF, MAX_D, ptr(lu[0, i]),
                                                ptr(lu[1, i])))

            stereo_one(0)
            w0 = time.perf_counter()
            for i in range(n):
                stereo_one(i)
            t_loop = (time.perf_counter() - w0) * 1e3
            # the resident outputs, from a call of their own
            with torch.cuda.stream(torch.cuda.Stream(device=dev)):
                stereo_dev()
            ex.sync()
            rk, rd, rn, ru = kp.cpu().numpy(), de.cpu().numpy(), cnt.cpu().numpy(), u.cpu().numpy()

            def differs(k, dsc, cn, uu):
                """pairs in which (k, dsc, cn, uu) differ from the loop's slabs over the defined rows"""
                bad = 0
                for i in range(n):
                    a_, b_ = int(ln[0, i]), int(ln[1, i])
                    same = (cn[0][i] == a_ and cn[1][i] == b_ and
                            k[0][i][:a_ * 28].tobytes() == lk[0, i, :a_ * 28].tobytes() and np.array_equal(dsc[0][i][:a_], ld[0, i, :a_]) and
                            k[1][i][:b_ * 28].tobytes() == lk[1, i, :b_ * 28].tobytes() and np.array_equal(dsc[1][i][:b_], ld[1, i, :b_]) and
                            uu[0][i][:a_].tobytes() == lu[0, i, :a_].tobytes() and uu[1][i][:a_].tobytes() == lu[1, i, :a_].tobytes())
                    bad += not same
                return bad

            bad = differs(hk, hd, hn, hu) + differs(sk, sd, sn, su) + differs(rk, rd, rn, ru)
            ok &= bad == 0
            # device time of the two stereo kernels inside one resident call
            split = "kernel split not measured"
            try:
                from torch.profiler import ProfilerActivity, profile
                st = torch.cuda.Stream(device=dev)
                with torch.cuda.stream(st):
                    stereo_dev()
                    torch.cuda.synchronize()
                    with profile(activities=[ProfilerActivity.CUDA], acc_events=True) as prof:
                        for _ in range(2):
                            stereo_dev()
                        torch.cuda.synchronize()
                us = {"stereo_match_kernel": 0.0, "stereo_median_kernel": 0.0}
                for k in prof.key_averages():
                    t = getattr(k, "self_device_time_total", None)
                    t = t if t is not None else getattr(k, "self_cuda_time_total", 0.0)
                    for kname in us:
                        if kname in k.key:
                            us[kname] += t
                split = "match kernel %.3f ms, median kernel %.3f ms per call" % (us["stereo_match_kernel"] / 2e3,
                                                                                 us["stereo_median_kernel"] / 2e3)
            except Exception as e:       # the kernel split is supplementary; the share above stands without it
                split = "kernel split not measured (%s)" % e
            share = max(t_st - t_mono, 0.0) / t_st
            lines.append("%-5s %4dx%-3d nfeat %4d  %3d pairs: resident %8.0f pairs/s (%.3f ms)  e2e %8.0f pairs/s  e2e serial %8.0f pairs/s  "
                         "loop %7.0f pairs/s  stereo share %4.1f %% (%.3f of %.3f ms; %s)  outputs %s" %
                         (name, cols, rows, nf, n, n / t_st * 1e3, t_st, n / t_e2e * 1e3, n / t_e2e_serial * 1e3, n / t_loop * 1e3,
                          100 * share, t_st - t_mono, t_st, split, "identical" if bad == 0 else "DIFFER in %d checks" % bad))
            print(lines[-1], flush=True)
    lines.append("# row buckets (the reference's vRowIndices): not added.  The share above is large, so they are the next step for this"
                 " path; stereo_match_kernel scans every right keypoint of its pair with the row test.")
    lines.append("# %s" % gpu_info())
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    if not ok:
        print("batched and looped outputs differ", file=sys.stderr)
        sys.exit(1)


if __name__ == "__main__":
    main()
