"""Per-call latency of the search part of ORBmatcher::Fuse at the shapes of LocalMapping::SearchInNeighbors
(src/LocalMapping.cc:766-803), next to the CPU oracle's single-thread time on the same inputs.

  forward: 30 target key frames x the current key frame's 1200 map points, timed as ONE batched orbx_fuse call, as 30
           per-key-frame orbx_fuse calls, and as the oracle on one CPU thread;
  reverse: 1 key frame x 20 000 points (the neighbours' points fused into the current key frame).

Each GPU call takes host arrays and returns host results (one pinned upload, grid + scan kernels, one download and a stream
synchronise inside the call), so the host clock around it measures the whole call.  5 warm-up calls, then 50 timed calls; the
results must be identical to the oracle's.  The card's name and power limit are read with a read-only nvidia-smi query in the
same run.

    python tools/fuse_latency.py [--out FILE]
"""
import argparse
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import wut_cuda_orb_slam3_b200 as orbx  # noqa: E402
from tests import fuse_oracle  # noqa: E402
from tests.fuse_synth import BOUNDS, scene  # noqa: E402


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError) as e:
        return "unknown (%s)" % e


def stats(ts):
    ts = np.array(ts) * 1e6
    return "median %.0f us, min %.0f us" % (np.median(ts), ts.min())


def timed(fn, warm=5, n=50):
    for _ in range(warm):
        r = fn()
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return r, ts


def views(kfs):
    return [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS, k["inv_sigma2"], k["bf"], u_right=k["ur"]) for k in kfs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if orbx.lib().orbx_device_count() < 1:
        sys.exit("no CUDA device: this tool measures the GPU path")
    fo = fuse_oracle.load()
    lines = ["ORBmatcher::Fuse search (orbx_fuse), th 3.0; scenes of tests/fuse_synth.py (752 x 480, 8 levels, stereo and monocular "
             "key frames)", "card: %s" % card()]
    same = True
    # forward
    X, pd, kfs, P = scene(1, n_kf=30, n_points=1200, n_distract=800)
    V = views(kfs)
    args = (P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0)
    want = fo.fuse(kfs, *args)
    got, t_batch = timed(lambda: orbx.fuse(V, *args))
    same &= np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    M = 1200
    sub = [(k, P["kf_offsets"][k], P["kf_offsets"][k + 1]) for k in range(30)]

    def per_kf():
        out = []
        for k, q0, q1 in sub:
            out.append(orbx.fuse([V[k]], [0, q1 - q0], pd, P["point"][q0:q1], P["valid"][q0:q1], P["u"][q0:q1], P["v"][q0:q1],
                                 P["invz"][q0:q1], P["level"][q0:q1], 3.0))
        return out
    got_k, t_loop = timed(per_kf)
    same &= np.array_equal(np.concatenate([g[0] for g in got_k]), want[0])
    _, t_cpu = timed(lambda: fo.fuse(kfs, *args), warm=1, n=10)
    nfeat = sum(len(k["kp"]) for k in kfs)
    lines += ["forward: 30 key frames (%d features in all) x %d map points = %d pairs, %d valid, %d fused" %
              (nfeat, M, len(P["u"]), int(P["valid"].sum()), int(want[1].sum())),
              "  one batched call (5 warm-up + 50 timed): %s" % stats(t_batch),
              "  30 per-key-frame calls (5 warm-up + 50 timed): %s" % stats(t_loop),
              "  CPU oracle, one thread (g++ -O3, 1 warm-up + 10 timed): %s" % stats(t_cpu)]
    # reverse
    X, pd, kfs, P = scene(2, n_kf=1, n_points=20000, n_distract=1500, see=0.12)
    V = views(kfs)
    args = (P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0)
    want = fo.fuse(kfs, *args)
    got, t_rev = timed(lambda: orbx.fuse(V, *args))
    same &= np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    _, t_rcpu = timed(lambda: fo.fuse(kfs, *args), warm=1, n=10)
    lines += ["reverse: 1 key frame (%d features) x %d points, %d valid, %d fused" % (len(kfs[0]["kp"]), len(P["u"]), int(P["valid"].sum()),
                                                                                   int(want[1].sum())),
              "  one call (5 warm-up + 50 timed): %s" % stats(t_rev),
              "  CPU oracle, one thread (1 warm-up + 10 timed): %s" % stats(t_rcpu),
              "identical to the oracle: %s" % same]
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    if not same:
        sys.exit("GPU result differs from the oracle")


if __name__ == "__main__":
    main()
