#!/usr/bin/env python3
"""bench.py — ORB front-end throughput on B200 (contract: one JSON line on stdout from rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--batch B] [--no-knn2] [--dump-outputs DIR]

Workload (BASELINE.json metric "ORB extract frames/s (752x480, 1000kp) & 2-NN Hamming compares/s"):
  * main line: batched ORBextractor::operator() on synthetic 752x480 frames, nFeatures=1000, 8 levels, scale 1.2,
    FAST 20/7.  One step = one pass over a batch of B frames per GPU (weak scaling: every rank extracts its own B
    frames, no collective on the data path).  `value` = frames/s with the frames resident in HBM; `e2e` = the same
    through the host-buffer C-ABI call orbx_extract_batch (pinned host images in, keypoints+descriptors out).
  * "knn2" block: brute-force Hamming 2-NN, 100k queries x 10M database rows, database sharded over the ranks,
    per-shard candidates all-gathered with NCCL and merged on the GPU (strong scaling).
  * "cfg4" block: BASELINE.json configs[3] as written — 8192 synthetic 1280x720 frames, 2000 features each, frame range
    [r*F/G, (r+1)*F/G) on rank r (strong scaling, no collective on the data path), resident and host-fed, with a checksum of
    all keypoints / descriptors reduced over the ranks and compared with the value a single GPU produced.
  * --dump-outputs DIR: after the timed steps, what the last resident extraction step and the 2-NN pass returned, as
    DIR/<name>.npy in float32 / float64 (a fixed sample of the frames; about 25 MB), so that two builds can be compared output
    for output.  The inputs are synthetic and seeded: the same arguments give the same inputs on every run.
  * --impl reference: the CPU oracle (a restatement of the reference's CPU path; the reference itself cannot be
    compiled here, see DESIGN.md) on all host threads, same metric / config.  That arm never loads the CUDA library.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # a benchmark run writes nothing into the tree (which may be read-only)

COLS, ROWS, NFEAT, NLEVELS, SCALE, INI_TH, MIN_TH = 752, 480, 1000, 8, 1.2, 20, 7
NQ, NDB = 100_000, 10_000_000
METRIC = "orb_extract_frames_per_s_752x480_1000kp"
DUMP_FRAMES, DUMP_QUERIES = 128, 100_000       # --dump-outputs sample sizes: ~21 MB of extraction + ~4 MB of 2-NN results


def dump_sample(n, k, seed):
    """Ascending indices of a fixed, seeded sample of k of n rows (all rows when n <= k)."""
    import numpy as np
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))


def extraction_outputs(d_kps, d_desc, d_n, d_nm):
    """What one resident extraction step hands its caller, as float arrays: keypoint and monocular counts of every frame and,
    for a sample of the frames, the keypoint rows (x, y, size, angle, response | octave, class_id) and the descriptor bytes,
    zero past each frame's count."""
    import numpy as np
    import torch
    n = d_n.cpu().numpy()
    frames = dump_sample(len(n), DUMP_FRAMES, seed=0)
    sel = torch.as_tensor(frames, device=d_kps.device)
    kps, desc = d_kps[sel].cpu().numpy(), d_desc[sel].cpu().numpy()
    valid = (np.arange(kps.shape[1])[None, :] < n[frames, None])[..., None]
    return {"extract_n_keypoints": n.astype(np.float64), "extract_n_mono": d_nm.cpu().numpy().astype(np.float64),
            "extract_sample_frames": frames.astype(np.float64),
            "extract_keypoints": np.where(valid, kps[..., :5], 0).astype(np.float32),
            "extract_keypoint_octave_class_id": np.where(valid, kps[..., 5:].view(np.int32), 0).astype(np.float32),
            "extract_descriptors": np.where(valid, desc, 0).astype(np.float32)}


def write_outputs(path, arrays):
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def level_sizes():
    import numpy as np
    import wut_cuda_orb_slam3_b200 as orbx
    inv = orbx.compute_tables(NFEAT, SCALE, NLEVELS)["inv"]
    return [(int(np.rint(np.float32(COLS) * inv[l])), int(np.rint(np.float32(ROWS) * inv[l]))) for l in range(NLEVELS)]


def algorithmic_bytes():
    """SURVEY.md §8(d): per-frame algorithmic HBM bytes, whole pipeline and per stage (see DESIGN.md §Roofline)."""
    px = [w * h for (w, h) in level_sizes()]
    total_px = sum(px)
    n = NFEAT
    per_stage = {
        "pyramid": px[0] + sum(px),                 # read level 0, write every level (levels 1-7 from the previous one in cache)
        "fast": total_px,                           # read every level once
        "blur": 2 * total_px,                       # read + write every level once
        "octree": 0,
        "orient_describe": 32 * n,
        "pack": 60 * n,
    }
    whole = px[0] + sum(px[1:]) + 3 * total_px + 60 * n
    return whole, per_stage


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_oracle_throughput(n_frames, threads, seed0=5000):
    """Frames/s of the CPU oracle (restated reference CPU path) on `threads` host threads, one frame per thread at a time."""
    from tests import oracle_lib
    o = oracle_lib.load()
    imgs = [o.synth_image(seed0 + i, COLS, ROWS) for i in range(min(n_frames, 16))]      # csrc/synth.h compiled into the oracle
    exs = [o.extractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH) for _ in range(threads)]
    counter = {"next": 0, "kp": 0}
    lock = threading.Lock()

    def work(t):
        while True:
            with lock:
                i = counter["next"]
                if i >= n_frames:
                    return
                counter["next"] = i + 1
            k, d, nm = exs[t].extract(imgs[i % len(imgs)], (0, 0))
            with lock:
                counter["kp"] += len(k)

    for e in exs[:1]:
        e.extract(imgs[0], (0, 0))      # warm-up (page in the library)
    t0 = time.perf_counter()
    ths = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    dt = time.perf_counter() - t0
    return n_frames / dt, dt, counter["kp"] / max(n_frames, 1)


def cpu_cv2_hybrid(n_frames=24, seed0=5000):
    """How fast could the CPU path be with OpenCV's SIMD kernels where the reference calls OpenCV?  One thread: the oracle's
    own stage times for the reference-owned stages (octree + orientation, descriptors + packing) plus cv2's times for the
    OpenCV-owned ones — the resize / copyMakeBorder chain, cv2.FastFeatureDetector (ONE call per level at iniThFAST with NMS:
    a lower bound of the reference's ~700 per-cell calls plus minThFAST retries) and the eight GaussianBlur calls.  Reported as
    frames/s per thread and, optimistically, times the host threads.  None if cv2 is not importable."""
    try:
        import cv2
    except Exception:
        return None
    import numpy as np
    from tests import oracle_lib
    o = oracle_lib.load()
    cv2.setNumThreads(1)
    ex = o.extractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH)
    imgs = [o.synth_image(seed0 + i, COLS, ROWS) for i in range(4)]
    ex.extract(imgs[0], (0, 0)); ex.stage_times(reset=True)
    t0 = time.perf_counter()
    for i in range(n_frames):
        ex.extract(imgs[i % 4], (0, 0))
    total_ms = (time.perf_counter() - t0) * 1e3 / n_frames
    st = {k: v / n_frames for k, v in ex.stage_times().items()}
    inv = o.tables(NFEAT, SCALE, NLEVELS)["inv"]
    sizes = [(int(np.rint(np.float32(COLS) * inv[l])), int(np.rint(np.float32(ROWS) * inv[l]))) for l in range(NLEVELS)]
    fast = cv2.FastFeatureDetector_create(threshold=INI_TH, nonmaxSuppression=True)
    t_pyr = t_fast = t_blur = 0.0
    for i in range(n_frames):
        img = imgs[i % 4]
        a = time.perf_counter()
        levels = [cv2.copyMakeBorder(img, 19, 19, 19, 19, cv2.BORDER_REFLECT_101)]
        cur = img
        for l in range(1, NLEVELS):
            cur = cv2.resize(cur, sizes[l], interpolation=cv2.INTER_LINEAR)
            levels.append(cv2.copyMakeBorder(cur, 19, 19, 19, 19, cv2.BORDER_REFLECT_101))
        b = time.perf_counter()
        for l in range(NLEVELS):
            w, h = sizes[l]
            fast.detect(levels[l][3:h + 35, 3:w + 35])            # the FAST window [16, w - 16) plus its 3-px ring
        c = time.perf_counter()
        for l in range(NLEVELS):
            w, h = sizes[l]
            cv2.GaussianBlur(levels[l][19:19 + h, 19:19 + w], (7, 7), 2, 2, borderType=cv2.BORDER_REFLECT_101)
        d = time.perf_counter()
        t_pyr += b - a; t_fast += c - b; t_blur += d - c
    cvst = {"pyramid": 1e3 * t_pyr / n_frames, "fast": 1e3 * t_fast / n_frames, "blur": 1e3 * t_blur / n_frames}
    hybrid_ms = cvst["pyramid"] + cvst["fast"] + cvst["blur"] + st["octree_orient"] + st["describe"]
    return {"ms_per_frame_one_thread": hybrid_ms, "frames_per_s_one_thread": 1e3 / hybrid_ms,
            "oracle_ms_per_frame_one_thread": total_ms, "oracle_stage_ms": st, "cv2_stage_ms": cvst, "cv2_version": cv2.__version__,
            "what": "cv2 (SIMD, 1 thread) for pyramid / FAST (one call per level at iniThFAST: a lower bound of the reference's per-cell calls) / "
                    "blur + the oracle's octree, orientation and descriptor stages: an upper bound on a tuned CPU path per thread"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    per_step = 64 * threads                   # ~1.5 s of work per step on all host threads
    for _ in range(args.warmup):
        cpu_oracle_throughput(max(threads, 8), threads)
    t0 = time.perf_counter()
    fps_sum = 0.0
    for _ in range(args.steps):
        fps, dt, kp = cpu_oracle_throughput(per_step, threads)
        fps_sum += fps
    total = time.perf_counter() - t0
    value = per_step * args.steps / total
    sample = "%d frames/step of the 752x480/1000kp workload, %d host threads, one frame per thread" % (per_step, threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": {"workload": "orb_extract 752x480 nfeatures=1000 levels=8 scale=1.2 fast=20/7 (CPU oracle = restated reference CPU path; "
                               "reference itself not buildable here: needs OpenCV/OpenCL/boost)", "frames_per_step": per_step},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist

    import wut_cuda_orb_slam3_b200 as orbx
    from wut_cuda_orb_slam3_b200 import synth
    from wut_cuda_orb_slam3_b200.capi import lib, ptr, check

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = args.batch
    # ---- resident inputs, generated on the device (bit-identical to the host generator) ------------------------------
    d_img = torch.empty((B, ROWS, COLS), dtype=torch.uint8, device=dev)
    synth.images_device(d_img, 1000 + rank * B, B, COLS, ROWS, COLS, ROWS * COLS, device=local_rank)
    ex = orbx.ORBextractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=COLS, max_rows=ROWS, max_batch=B)
    cap = ex.max_keypoints()
    d_kps = torch.zeros((B, cap, 7), dtype=torch.float32, device=dev)
    d_desc = torch.zeros((B, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(B, dtype=torch.int32, device=dev)
    d_nm = torch.zeros(B, dtype=torch.int32, device=dev)
    # a dedicated (non-NULL) torch stream: kernels are launched on it by the library and torch's events time it
    tstream = torch.cuda.Stream(device=dev)
    torch.cuda.synchronize()
    torch.cuda.set_stream(tstream)
    stream = tstream.cuda_stream
    assert stream != 0

    def step():
        ex.extract_batch_device(d_img, B, ROWS, COLS, COLS, ROWS * COLS, d_kps, d_desc, cap, d_n, d_nm, (0, 0), stream=stream)

    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib().orbx_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    launches = lib().orbx_launch_count() - launches0
    outputs = extraction_outputs(d_kps, d_desc, d_n, d_nm) if args.dump_outputs and rank == 0 else None
    # per-stage device times: the same K steps again with CUDA events between the stages (kept out of the timed region above)
    ex.profile_begin()
    for _ in range(args.steps):
        step()
    torch.cuda.synchronize()
    stage_ms, n_chunks = ex.profile_end()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = max_over_ranks(ms)
    value = world * B * args.steps / (ms * 1e-3)
    kp_mean = float(d_n.float().mean().item())

    # ---- end to end through the host-buffer C-ABI call (pinned host memory, H2D + D2H inside the timed region) ----------
    def run_e2e(Be, chunk, probe=None):
        """frames/s through orbx_extract_batch: Be frames per call from pinned host memory (frames repeat modulo B), results
        back in pinned host memory; H2D + compute + D2H all inside the timed region."""
        h_img = torch.empty((Be, ROWS, COLS), dtype=torch.uint8).pin_memory()
        for f0 in range(0, Be, B):
            h_img[f0:f0 + B].copy_(d_img[:min(B, Be - f0)])
        h_kps = torch.empty((Be, cap, 7), dtype=torch.float32).pin_memory()
        h_desc = torch.empty((Be, cap, 32), dtype=torch.uint8).pin_memory()
        h_n = torch.empty(Be, dtype=torch.int32).pin_memory()
        h_nm = torch.empty(Be, dtype=torch.int32).pin_memory()
        ex2 = orbx.ORBextractor(NFEAT, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=COLS, max_rows=ROWS, max_batch=chunk)
        ptrs = (C.c_void_p * Be)(*[h_img.data_ptr() + f * ROWS * COLS for f in range(Be)])

        def e2e_step():
            check(lib().orbx_extract_batch(ex2._h, ptrs, Be, ROWS, COLS, COLS, 0, 0, ptr(h_kps), ptr(h_desc), cap, ptr(h_n), ptr(h_nm)))

        for _ in range(max(args.warmup, 1)):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            e2e_step()
        e2e_s = max_over_ranks(time.perf_counter() - t0)
        assert torch.equal(h_n, d_n.cpu().repeat((Be + B - 1) // B)[:Be]), "host-buffer API and device API disagree"
        ex2.close()
        if probe is not None:       # the link's ceiling measured from the SAME pinned pages the call just streamed
            probe.append(h2d_ceiling(h_img.view(-1)))
        return world * Be * args.steps / e2e_s

    def h2d_ceiling(h_src=None):
        """Pinned host -> device copy bandwidth with ALL ranks copying at once (the box's ceiling for the host-fed path):
        256 MB per copy, 6 copies per rank after a barrier, device-timed, max over ranks; the best of 4 such rounds as the
        aggregate GB/s.  Measured twice — from the pinned buffer of the end-to-end leg itself (h_src) and from a fresh pinned
        allocation — and the larger is reported: on some boxes a fresh allocation lands on pages that copy 20 % slower."""
        nbytes = 256 << 20
        if h_src is not None and h_src.numel() >= nbytes:
            h = h_src[:nbytes]
        else:
            h = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        d.copy_(h, non_blocking=True)
        best = 0.0
        for _round in range(4):
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(6):
                d.copy_(h, non_blocking=True)
            b.record()
            torch.cuda.synchronize()
            t = max_over_ranks(a.elapsed_time(b))
            best = max(best, world * 6 * nbytes / (t * 1e-3) / 1e9)
        return best

    Be = args.e2e_batch
    ceil_same = []
    e2e_value = run_e2e(Be, args.e2e_chunk, ceil_same)
    ceil_gbs = max(ceil_same + [h2d_ceiling()])
    e2e = {"value": e2e_value, "unit": "frames/s", "h2d_bytes_per_step": Be * ROWS * COLS,
           "d2h_bytes_per_step": Be * cap * 60 + Be * 8, "frames_per_step": Be, "pipeline_chunk": args.e2e_chunk,
           "api": "orbx_extract_batch (pinned host buffers; one call = one step)",
           "h2d_ceiling_gbs": ceil_gbs, "h2d_achieved_gbs": e2e_value * ROWS * COLS / 1e9,
           "h2d_ceiling_note": "aggregate pinned host->device bandwidth with all %d rank(s) copying at once (measured here: 256 MB copies, best of 4 rounds, from the call's own pinned buffer and from a fresh one)" % world}
    e2e_small = None
    if Be > B:      # the same call with only as many frames as the resident step, for comparison
        e2e_small = {"value": run_e2e(B, 64), "unit": "frames/s", "frames_per_step": B, "pipeline_chunk": 64}

    # ---- roofline of the dominant kernel ----------------------------------------------------------------------------------
    peak, peak_src = _hbm_peak()
    whole_bytes, stage_bytes = algorithmic_bytes()
    launches_per_stage = n_chunks
    dom = max(stage_ms, key=stage_ms.get)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(dom)
        if traffic is not None:
            traffic = traffic["dram_bytes_per_frame"] * B       # per launch, like `achieved`
    dom_ms = stage_ms[dom] / max(launches_per_stage, 1)
    achieved = stage_bytes[dom] * B / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "avg_launch_ms": dom_ms,
                "algorithmic_bytes_per_launch": stage_bytes[dom] * B}
    stages = {}
    tot_ms = sum(stage_ms.values())
    for k, v in stage_ms.items():
        per = v / max(launches_per_stage, 1)
        gbs = stage_bytes[k] * B / (per * 1e-3) / 1e9 if per > 0 else 0.0
        stages[k] = {"ms_per_step": per, "share": v / tot_ms if tot_ms > 0 else 0.0, "algorithmic_GBps": gbs, "frac_of_hbm_peak": gbs / peak}
    pipeline_gbs = whole_bytes * B * args.steps / (ms * 1e-3) / 1e9
    extra = {"stages": stages, "stages_note": "CUDA-event time per stage from a separate, single-stream profiling pass of the same K steps; in the "
                                               "timed pass the blur runs on a side stream beside FAST (it fills the tails of FAST's launches), "
                                               "so ms_per_step is a little less than the sum of the stages",
             "pipeline": {"algorithmic_bytes_per_frame": whole_bytes, "achieved_GBps": pipeline_gbs, "frac_of_hbm_peak": pipeline_gbs / peak},
             "mean_keypoints_per_frame": kp_mean}
    if e2e_small is not None:
        extra["e2e_small_call"] = e2e_small

    # ---- the other BASELINE.json configs (parity-test shapes), measured briefly on rank 0 for context ---------------------------
    if rank == 0 and not args.no_other:
        ex.close()
        del d_kps, d_desc
        torch.cuda.empty_cache()
        extra["other_configs"] = run_other_configs(local_rank, dev)

    # ---- configs[3] as written: 8192 frames 1280x720 / 2000 features, sharded over the ranks ---------------------------------
    cfg4 = None
    if not args.no_cfg4:
        if not (rank == 0 and not args.no_other):      # (rank 0 released these above when it ran the other configs)
            ex.close()
            del d_kps, d_desc
        del d_img
        torch.cuda.empty_cache()
        cfg4 = run_cfg4(args, rank, world, local_rank, dev, barrier, max_over_ranks)

    # ---- 2-NN Hamming: 100k x 10M, database sharded over the ranks, NCCL all-gather + merge -------------------------------
    knn = None
    if not args.no_knn2:
        knn = run_knn2(args, rank, world, local_rank, dev, barrier, max_over_ranks, outputs)

    # ---- CPU baseline (rank 0, N=1 only): the oracle on all host threads, bounded sample -----------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = os.cpu_count() or 1
        nfr = 384 * threads                     # ~10 s of work on all host threads
        fps, dt, kp = cpu_oracle_throughput(nfr, threads)
        fps1, dt1, _ = cpu_oracle_throughput(240, 1)
        cpu = {"value": fps, "unit": "frames/s", "cores": threads, "kind": "port",
               "sample": "%d frames of the same 752x480/1000kp workload in %.1f s on %d threads (single thread: %.1f frames/s)" % (nfr, dt, threads, fps1),
               "single_thread_value": fps1}
        hyb = cpu_cv2_hybrid()
        if hyb is not None:
            hyb["frames_per_s_all_threads_if_it_scaled_perfectly"] = hyb["frames_per_s_one_thread"] * threads
            cpu["cv2_simd_hybrid"] = hyb

    if outputs is not None:
        write_outputs(args.dump_outputs, outputs)

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
            "data": "synthetic",
            "config": {"workload": "orb_extract 752x480 nfeatures=1000 levels=8 scale=1.2 fast=20/7", "frames_per_gpu_per_step": B,
                       "global_frames_per_step": B * world, "parallelism": "frames sharded over %d GPU(s), no collective" % world,
                       "l2": "inputs larger than L2: %.0f MB of frames + %.1f GB workspace touched per step" % (B * ROWS * COLS / 1e6, B * 10e6 / 1e9)},
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "extra": extra,
        }
        if knn is not None:
            line["knn2"] = knn
        if cfg4 is not None:
            line["cfg4"] = cfg4
        print(json.dumps(line), flush=True)


def run_other_configs(local_rank, dev):
    """configs[1..3] of BASELINE.json as short measurements (host image in -> results out, median of repeated calls):
    EuRoC-shape stereo pair + ComputeStereoMatches, KITTI-shape stereo pair + brute-force 2-NN + ratio test, and the
    resident 1280x720 / 2000-feature batch."""
    import numpy as np
    import torch

    import wut_cuda_orb_slam3_b200 as orbx
    from wut_cuda_orb_slam3_b200 import synth

    def med_ms(fn, reps=30, warm=5):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter(); fn(); ts.append(time.perf_counter() - t0)
        return 1e3 * float(np.median(ts))

    out = {}
    # configs[1]: 752x480 stereo pair, 1200 features per image, extraction x2 + ComputeStereoMatches
    L, R = synth.image(31, 752, 480, view=0, max_disp=40), synth.image(31, 752, 480, view=1, max_disp=40)
    exL = orbx.ORBextractor(1200, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=752, max_rows=480, max_batch=1)
    exR = orbx.ORBextractor(1200, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=752, max_rows=480, max_batch=1)
    res = {}

    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(2)          # the reference extracts left and right on two threads (src/Frame.cc:124-127)

    def stereo():
        fl, fr = pool.submit(exL, L), pool.submit(exR, R)
        (_, kl, dl), (_, kr, dr) = fl.result(), fr.result()
        res["u"], res["d"] = orbx.compute_stereo_matches(exL, exR, kl, dl, kr, dr, 47.9, 435.2)
    ms = med_ms(stereo)
    out["euroc_stereo_pair_1200"] = {"ms_per_pair": ms, "pairs_per_s": 1e3 / ms, "stereo_matches": int((res["u"] >= 0).sum()),
                                     "what": "orbx_extract left | right on two host threads + orbx_stereo_match"}
    # the stereo Frame constructor as ONE C-ABI call (src/Frame.cc:124-143): two extractions on two streams + the matcher on the
    # device-resident features, pinned host buffers in and out
    import ctypes as C
    from wut_cuda_orb_slam3_b200.capi import lib, ptr, check
    hL = torch.from_numpy(L).pin_memory(); hR = torch.from_numpy(R).pin_memory()
    cap = exL.max_keypoints(480, 752)
    pk = [torch.empty((cap, 7), dtype=torch.float32).pin_memory() for _ in range(2)]
    pd = [torch.empty((cap, 32), dtype=torch.uint8).pin_memory() for _ in range(2)]
    pu = torch.empty(cap, dtype=torch.float32).pin_memory(); pz = torch.empty(cap, dtype=torch.float32).pin_memory()
    nLc, nRc = C.c_int(0), C.c_int(0)

    def stereo_one_call():
        check(lib().orbx_extract_stereo(exL._h, exR._h, ptr(hL), ptr(hR), 480, 752, 752, ptr(pk[0]), ptr(pd[0]), C.byref(nLc), ptr(pk[1]), ptr(pd[1]),
                                        C.byref(nRc), cap, 47.9, 435.2, ptr(pu), ptr(pz)))
    ms = med_ms(stereo_one_call, reps=100)
    assert np.array_equal(pu[:nLc.value].numpy(), res["u"]) and np.array_equal(pz[:nLc.value].numpy(), res["d"]), "orbx_extract_stereo disagrees"
    out["euroc_stereo_pair_1200_extract_stereo"] = {"ms_per_pair": ms, "pairs_per_s": 1e3 / ms, "stereo_matches": int((pu[:nLc.value] >= 0).sum()),
                                                    "what": "orbx_extract_stereo: one C-ABI call = ExtractORB left | right + ComputeStereoMatches (Frame.cc:124-143)"}
    exL.close(); exR.close()
    # the same pair as ONE two-frame call on one extractor (both pyramids stay on the device as frames 0 and 1): what a
    # stereo front end built on the batch API does instead of two extractor threads
    exS = orbx.ORBextractor(1200, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=752, max_rows=480, max_batch=2)
    LR = np.stack([L, R])

    def stereo_batched():
        nm, n, kps, desc = exS.extract_batch(LR)
        res["u2"], res["d2"] = orbx.compute_stereo_matches(exS, exS, kps[0, :n[0]], desc[0, :n[0]], kps[1, :n[1]], desc[1, :n[1]], 47.9, 435.2,
                                                           frameL=0, frameR=1)
    ms = med_ms(stereo_batched)
    assert np.array_equal(res["u2"], res["u"]) and np.array_equal(res["d2"], res["d"]), "two-frame call and two-extractor path disagree"
    out["euroc_stereo_pair_1200_one_call"] = {"ms_per_pair": ms, "pairs_per_s": 1e3 / ms, "stereo_matches": int((res["u2"] >= 0).sum()),
                                              "what": "orbx_extract_batch([left, right]) on one extractor + orbx_stereo_match(frames 0, 1)"}
    exS.close()
    # configs[2]: 1241x376 stereo pair, 2000 features, extraction x2 + brute-force 2-NN L->R + 0.7 ratio test
    L, R = synth.image(32, 1241, 376, view=0, max_disp=60), synth.image(32, 1241, 376, view=1, max_disp=60)
    exL = orbx.ORBextractor(2000, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=1241, max_rows=376, max_batch=1)
    exR = orbx.ORBextractor(2000, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=1241, max_rows=376, max_batch=1)
    m = orbx.ORBmatcher(0.7, True, device=local_rank)

    def kitti():
        fl, fr = pool.submit(exL, L), pool.submit(exR, R)
        (_, kl, dl), (_, kr, dr) = fl.result(), fr.result()
        idx, dist = m.knn2(dl, dr)
        res["acc"] = m.ratio_test(dist, mode=2, ratio=0.7)
    ms = med_ms(kitti)
    out["kitti_stereo_pair_2000"] = {"ms_per_pair": ms, "pairs_per_s": 1e3 / ms, "ratio_test_matches": int(res["acc"].sum()),
                                     "what": "orbx_extract left | right on two host threads + orbx_knn2 + orbx_ratio_test (Frame.cc:1174-1181 form)"}
    exL.close(); exR.close()
    # configs[3] (per-GPU share): resident 1280x720 frames, 2000 features
    Bh = 256
    d_img = torch.empty((Bh, 720, 1280), dtype=torch.uint8, device=dev)
    synth.images_device(d_img, 9000, Bh, 1280, 720, 1280, 720 * 1280, device=local_rank)
    ex = orbx.ORBextractor(2000, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=1280, max_rows=720, max_batch=Bh)
    cap = ex.max_keypoints()
    d_kps = torch.zeros((Bh, cap, 7), dtype=torch.float32, device=dev); d_desc = torch.zeros((Bh, cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(Bh, dtype=torch.int32, device=dev); d_nm = torch.zeros(Bh, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        ex.extract_batch_device(d_img, Bh, 720, 1280, 1280, 720 * 1280, d_kps, d_desc, cap, d_n, d_nm, (0, 0), stream=stream)
    for _ in range(3):
        step()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for _ in range(5):
        step()
    e1.record(); torch.cuda.synchronize()
    msb = e0.elapsed_time(e1) / 5
    out["hd720_batch_2000"] = {"frames_per_s": Bh / msb * 1e3, "ms_per_step": msb, "frames_per_step": Bh, "mean_keypoints_per_frame": float(d_n.float().mean().item()),
                               "algorithmic_bytes_per_frame": 11532352, "what": "orbx_extract_batch_device, frames resident in HBM"}
    ex.close()
    return out


# Checksums of configs[3] produced by ONE B200 over all 8192 frames (seeds 9000 .. 9000 + 8191): every N must reproduce them.
# (total keypoints, sum n_out[f] * (f + 1), sum of the int32 words of all valid descriptors, same for the 28-byte keypoints)
CFG4_EXPECTED = {8192: [16438361, 67339139679, 3427532576264195, 92368513198523344]}


def run_cfg4(args, rank, world, local_rank, dev, barrier, max_over_ranks):
    """BASELINE.json configs[3]: F = 8192 synthetic 1280x720 frames, nFeatures = 2000, frames [r*F/G, (r+1)*F/G) on rank r.
    Resident: the rank's frames generated on the device (seed = 9000 + global frame index), one orbx_extract_batch_device call
    over all of them.  Host-fed: the same frames from pinned host memory through orbx_extract_batch.  No collective on the data
    path; the checksums are all-reduced afterwards."""
    import ctypes as C
    import torch
    import torch.distributed as dist

    import wut_cuda_orb_slam3_b200 as orbx
    from wut_cuda_orb_slam3_b200 import synth
    from wut_cuda_orb_slam3_b200.capi import lib, ptr, check

    F, W, H, NF = args.cfg4_frames, 1280, 720, 2000
    per = (F + world - 1) // world
    f0 = min(rank * per, F)
    nloc = max(0, min(per, F - f0))
    chunk = 256
    ex = orbx.ORBextractor(NF, SCALE, NLEVELS, INI_TH, MIN_TH, device=local_rank, max_cols=W, max_rows=H, max_batch=chunk)
    cap = ex.max_keypoints(H, W)
    d_img = torch.empty((max(nloc, 1), H, W), dtype=torch.uint8, device=dev)
    for c0 in range(0, nloc, 1024):
        n = min(1024, nloc - c0)
        synth.images_device(d_img[c0:], 9000 + f0 + c0, n, W, H, W, H * W, device=local_rank)
    d_kps = torch.zeros((max(nloc, 1), cap, 7), dtype=torch.float32, device=dev)
    d_desc = torch.zeros((max(nloc, 1), cap, 32), dtype=torch.uint8, device=dev)
    d_n = torch.zeros(max(nloc, 1), dtype=torch.int32, device=dev); d_nm = torch.zeros_like(d_n)
    stream = torch.cuda.current_stream().cuda_stream

    def resident_pass():
        if nloc:
            ex.extract_batch_device(d_img, nloc, H, W, W, H * W, d_kps, d_desc, cap, d_n, d_nm, (0, 0), stream=stream)

    resident_pass()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    e0.record()
    for _ in range(reps):
        resident_pass()
    e1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1)) / reps

    # checksums over the rank's frames (raw 32-bit words of the valid rows), reduced over the ranks
    def checksums(kps, desc, n):
        n64 = n.to(torch.int64)
        gidx = torch.arange(f0 + 1, f0 + 1 + n.numel(), device=n.device, dtype=torch.int64)
        tot = [int(n64.sum().item()), int((n64 * gidx).sum().item()), 0, 0]
        for c0 in range(0, n.numel(), 512):
            sl = slice(c0, min(c0 + 512, n.numel()))
            valid = (torch.arange(cap, device=n.device)[None, :] < n[sl, None])
            tot[2] += int((desc[sl].view(torch.int32).to(torch.int64).sum(dim=2) * valid).sum().item())
            tot[3] += int((kps[sl].view(torch.int32).to(torch.int64).sum(dim=2) * valid).sum().item())
        return tot
    cs = checksums(d_kps[:nloc], d_desc[:nloc], d_n[:nloc]) if nloc else [0, 0, 0, 0]
    if world > 1:
        t = torch.tensor(cs, dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        cs = [int(v) for v in t.tolist()]

    # host-fed: the rank's frames from pinned host memory, results into pinned host memory
    e2e_fps, e2e_cs_ok = None, None
    if nloc:
        h_img = torch.empty((nloc, H, W), dtype=torch.uint8).pin_memory()
        h_img.copy_(d_img[:nloc])
        n_dev = d_n[:nloc].cpu()
        del d_kps, d_desc
        torch.cuda.empty_cache()
        h_kps = torch.empty((nloc, cap, 7), dtype=torch.float32).pin_memory()
        h_desc = torch.empty((nloc, cap, 32), dtype=torch.uint8).pin_memory()
        h_n = torch.empty(nloc, dtype=torch.int32).pin_memory(); h_nm = torch.empty(nloc, dtype=torch.int32).pin_memory()
        ptrs = (C.c_void_p * nloc)(*[h_img.data_ptr() + f * H * W for f in range(nloc)])

        def host_pass():
            check(lib().orbx_extract_batch(ex._h, ptrs, nloc, H, W, W, 0, 0, ptr(h_kps), ptr(h_desc), cap, ptr(h_n), ptr(h_nm)))
        host_pass()
    barrier()
    t0 = time.perf_counter()
    if nloc:
        host_pass()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    if nloc:
        e2e_cs_ok = bool(torch.equal(h_n, n_dev))
    e2e_fps = F / e2e_s
    ex.close()
    expected = CFG4_EXPECTED.get(F)
    return {"what": "BASELINE configs[3]: %d frames 1280x720, nfeatures=2000, frames [r*F/G, (r+1)*F/G) per rank, no collective" % F,
            "frames": F, "n_gpus": world, "scaling": "strong", "frames_per_rank": per,
            "frames_per_s": F / (ms * 1e-3), "ms_per_pass": ms, "mean_keypoints_per_frame": cs[0] / max(F, 1),
            "algorithmic_bytes_per_frame": 11532352, "hbm_frac": F * 11532352 / (ms * 1e-3) / 1e9 / world / _hbm_peak()[0],
            "e2e": {"value": e2e_fps, "unit": "frames/s", "h2d_bytes": F * H * W, "d2h_bytes": F * (cap * 60 + 8),
                    "api": "orbx_extract_batch, pinned host buffers, one call per rank over its %d frames" % per,
                    "host_counts_equal_device_counts": e2e_cs_ok},
            "checksum": cs, "checksum_expected_from_1_gpu": expected,
            "checksum_matches_n1": (cs == expected) if expected is not None else None}


def _hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


IMMA_PEAK_TOPS = 1139.9     # legacy warp-level int8 MMA (IMMA.16832.U8.U8) issue rate of one B200: tools/micro/imma_rate.cu, profiles/r02g_imma_rate.txt


def knn2_roofline(per_gpu, popc_peak):
    """The matcher's roofline block.  Default kernel = int8 tensor-core dot products on {0,1}-expanded descriptors (8 m16n8k32 MMAs
    per 16 x 8 tile of compares = 512 int8 ops per compare); ORBX_KNN_IMMA=0 = the carry-save POPC kernel of round 1."""
    if os.environ.get("ORBX_KNN_IMMA", "1") != "0":
        tops = per_gpu * 512 / 1e12
        return {"bound": "tensor (warp-level int8 MMA, mma.sync m16n8k32 u8 -> SASS IMMA.16832.U8.U8)", "achieved": tops, "peak": IMMA_PEAK_TOPS,
                "unit": "dense int8 TOPS per GPU", "frac": tops / IMMA_PEAK_TOPS,
                "algorithmic_popc_frac": per_gpu * 8 / popc_peak if popc_peak > 0 else None,
                "note": "Hamming(a, b) = popc(a) + popc(b) - 2 a.b on descriptors expanded to {0,1} bytes in registers; peak = the "
                        "measured issue rate of that MMA on a B200 of this pool (tools/micro/imma_rate.cu, profiles/r02g_imma_rate.txt; "
                        "Blackwell has no 1-bit MMA and tcgen05 kind::i8 is not used here); algorithmic_popc_frac relates the same "
                        "throughput to the 8-POPC-per-compare integer roofline of SURVEY.md §8(d) (POPC peak measured on this GPU) — "
                        "the carry-save POPC kernel (ORBX_KNN_IMMA=0) reaches 1.47 of it, this kernel more because it does not use that pipe"}
    return {"bound": "int-pipe POPC", "achieved": per_gpu * 8, "peak": popc_peak, "unit": "POPC.b32/s per GPU",
            "frac": per_gpu * 8 / popc_peak if popc_peak > 0 else None,
            "frac_issued": per_gpu * 4 / popc_peak if popc_peak > 0 else None,
            "note": "frac counts the ALGORITHMIC 8 POPC per 256-bit compare (SURVEY.md §8(d)) and can exceed 1: the kernel's "
                    "carry-save front end (16 LOP3) issues only 4 POPC per compare — frac_issued is the POPC pipe's real "
                    "utilisation; the co-limiter is the ALU pipe (LOP3/ISETP, ~78 % in ncu: profiles/*knn2_ncu_summary.txt). "
                    "peak = orbx_measure_popc_peak microbenchmark on this GPU"}


def run_knn2(args, rank, world, local_rank, dev, barrier, max_over_ranks, outputs=None):
    """BASELINE.json configs[4]: 100k queries x 10M database rows, database sharded over the ranks.  The whole exchange is inside
    the C ABI: orbx_knn2_sharded = local scan + ONE ncclAllGather of the packed candidates + merge (csrc/api_shard.cu); torch
    only carries rank 0's NCCL id to the other ranks.  The merged answer is verified on every rank (see `verified`)."""
    import numpy as np
    import torch
    import torch.distributed as dist

    import wut_cuda_orb_slam3_b200 as orbx
    from wut_cuda_orb_slam3_b200 import synth
    from wut_cuda_orb_slam3_b200.capi import lib

    nq, ndb, plant = args.knn_nq, args.knn_ndb, 4

    def bcast(b):
        t = torch.zeros(128, dtype=torch.uint8, device=dev)
        if b is not None:
            t.copy_(torch.frombuffer(bytearray(b), dtype=torch.uint8))
        if world > 1:
            dist.broadcast(t, src=0)
        return bytes(t.cpu().numpy().tobytes())

    sm = orbx.ShardedMatcher(rank, world, local_rank, bcast)
    first, nloc = sm.shard_rows(ndb, world, rank)
    d_db = torch.empty((max(nloc, 1), 32), dtype=torch.uint8, device=dev)
    d_q = torch.empty((nq, 32), dtype=torch.uint8, device=dev)
    synth.descriptors_device(d_db, 77, nloc, first_row=first, device=local_rank)
    synth.descriptors_device(d_q, 77, nq, is_query=True, ndb=ndb, plant_every=plant, device=local_rank)
    out_idx = torch.empty((nq, 2), dtype=torch.int32, device=dev); out_dist = torch.empty_like(out_idx)
    stream = torch.cuda.current_stream().cuda_stream

    def step(n_rows):
        sm.knn2(d_q, nq, d_db, n_rows, first, out_idx, out_dist, stream=stream)

    step(min(nloc, 200_000))          # warm-up on a slice (every rank calls: the all-gather is collective)
    barrier()
    l0 = lib().orbx_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = args.knn_reps
    ev0.record()
    for _ in range(reps):
        step(nloc)
    ev1.record()
    torch.cuda.synchronize()
    ms = max_over_ranks(ev0.elapsed_time(ev1))
    launches = lib().orbx_launch_count() - l0
    if outputs is not None:
        qsel = dump_sample(nq, DUMP_QUERIES, seed=1)
        sel = torch.as_tensor(qsel, device=dev)
        outputs.update({"knn2_sample_queries": qsel.astype(np.float64), "knn2_idx": out_idx[sel].cpu().numpy().astype(np.float64),
                        "knn2_dist": out_dist[sel].cpu().numpy().astype(np.float64)})
    compares = float(nq) * float(ndb) * reps
    cps = compares / (ms * 1e-3)
    popc_peak = orbx.measure_popc_peak(local_rank)

    # ---- verification of the merged answer (every rank holds it) ------------------------------------------------------
    # (1) planted queries: query q (q % 4 == 0) is database row q*2654435761 mod ndb with <= k = (q/4) % 61 bits flipped
    #     (csrc/synth.h:88-96); random rows lie ~128 +- 8 bits away, so that row must be the best match at distance <= k.
    qs = torch.arange(0, nq, plant, device=dev, dtype=torch.int64)
    want = (qs * 2654435761) % ndb
    kmax = (qs // plant) % 61
    planted_ok = bool(((out_idx[qs, 0].to(torch.int64) == want) & (out_dist[qs, 0].to(torch.int64) <= kmax)).all().item())
    # (2) 1000 non-planted queries against a single-rank scan of the WHOLE database (regenerated here in 1M-row pieces, each
    #     piece scanned with the single-GPU entry point and merged) — exercises nothing of the sharded path
    sel = (torch.arange(0, 1000, device=dev, dtype=torch.int64) * (nq // 1000 if nq >= 1000 else 1)) | 1
    sel = sel[sel < nq]
    d_qs = d_q[sel].contiguous()
    ns = int(sel.numel())
    piece = 1_000_000
    npieces = (ndb + piece - 1) // piece
    p_idx = torch.empty((npieces, ns, 2), dtype=torch.int32, device=dev); p_dist = torch.empty_like(p_idx)
    d_piece = torch.empty((piece, 32), dtype=torch.uint8, device=dev)
    for pi in range(npieces):
        r0 = pi * piece
        nr = min(piece, ndb - r0)
        synth.descriptors_device(d_piece, 77, nr, first_row=r0, device=local_rank, stream=stream)
        orbx.knn2_device(d_qs, ns, d_piece, nr, p_idx[pi], p_dist[pi], index_base=r0, device=local_rank, stream=stream)
    f_idx = torch.empty((ns, 2), dtype=torch.int32, device=dev); f_dist = torch.empty_like(f_idx)
    orbx.knn2_merge_device(p_idx, p_dist, npieces, ns, f_idx, f_dist, device=local_rank, stream=stream)
    torch.cuda.synchronize()
    sample_ok = bool(torch.equal(f_idx, out_idx[sel]) and torch.equal(f_dist, out_dist[sel]))
    # (3) 4 queries against a brute force written in torch (XOR + byte popcount table), independent of every kernel of ours
    lut = torch.tensor([bin(i).count("1") for i in range(256)], dtype=torch.int16, device=dev)
    torch_ok = True
    for qi in [1, nq // 3 | 1, nq // 2 | 1, nq - 1]:
        best = []
        for pi in range(npieces):
            r0 = pi * piece
            nr = min(piece, ndb - r0)
            synth.descriptors_device(d_piece, 77, nr, first_row=r0, device=local_rank, stream=stream)
            dd = lut[(d_piece[:nr] ^ d_q[qi][None, :]).to(torch.int64)].sum(dim=1, dtype=torch.int32)
            v, i = torch.sort(dd.to(torch.int64) * (1 << 32) + torch.arange(r0, r0 + nr, device=dev, dtype=torch.int64))
            best += [int(x) for x in v[:2].tolist()]
        best.sort()
        exp = [(b >> 32, b & 0xffffffff) for b in best[:2]]
        got = [(int(out_dist[qi, k]), int(out_idx[qi, k])) for k in range(2)]
        torch_ok = torch_ok and exp == got
    flags = torch.tensor([planted_ok, sample_ok, torch_ok], dtype=torch.int32, device=dev)
    if world > 1:
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    planted_ok, sample_ok, torch_ok = [bool(v) for v in flags.tolist()]
    nccl_version = sm.nccl_version()
    sm.close()
    per_gpu = cps / world
    return {"metric": "hamming_2nn_compares_per_s", "value": cps, "unit": "compares/s", "nq": nq, "ndb": ndb, "n_gpus": world,
            "scaling": "strong", "ms_per_pass": ms / reps, "gpu_launches": int(launches),
            "api": "orbx_knn2_sharded (C ABI: knn2_imma_kernel + one ncclAllGather of 16 B/query + knn2_merge_kernel)", "nccl_version": nccl_version,
            "verified": planted_ok and sample_ok and torch_ok,
            "verification": {"planted_queries_hit_their_row_within_k": planted_ok, "planted_queries": int(qs.numel()),
                             "sample_vs_single_rank_full_scan": sample_ok, "sample_queries": ns,
                             "four_queries_vs_torch_bruteforce": torch_ok},
            "roofline": knn2_roofline(per_gpu, popc_peak)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=512, help="frames per GPU per step")
    ap.add_argument("--e2e-batch", type=int, default=8192, help="frames per host-API call (as many as configs[3] streams)")
    ap.add_argument("--e2e-chunk", type=int, default=256, help="pipeline chunk of the host API (max_batch of its extractor)")
    ap.add_argument("--no-knn2", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-other", action="store_true", help="skip the short measurements of the other BASELINE configs")
    ap.add_argument("--no-cfg4", action="store_true", help="skip configs[3] (8192 x 1280x720 / 2000 features, sharded)")
    ap.add_argument("--cfg4-frames", type=int, default=8192, help="total frames of configs[3] over all ranks")
    ap.add_argument("--knn-nq", type=int, default=NQ)
    ap.add_argument("--knn-ndb", type=int, default=NDB)
    ap.add_argument("--knn-reps", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last resident extraction step and "
                    "the 2-NN pass returned as DIR/<name>.npy (float32 / float64, a fixed sample of the frames; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 0)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"      # NCCL prints its version banner on STDOUT; keep stdout = one JSON line
        import torch
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
