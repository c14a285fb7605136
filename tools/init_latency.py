"""Per-call latency of SearchForInitialization at the Tracking::MonocularInitialization shape (src/Tracking3.cc:740-741:
ORBmatcher(0.9, true), windowSize 100, frames of a 5 x nFeatures initialisation extractor), next to the CPU oracle's
single-thread time on the same inputs.

Each GPU call takes host arrays and returns host results (one pinned upload, grid + scan + resolve kernels, one download and a
stream synchronise inside the call), so the host clock around it measures the whole call.  5 warm-up calls, then 50 timed
calls.  The card's name and power limit are read with a read-only nvidia-smi query in the same run.

    python tools/init_latency.py [--out FILE]
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
from tests import init_oracle  # noqa: E402
from tests.init_synth import BOUNDS, bounds_grid, init_pair  # noqa: E402
from tests.proj_synth import SCALE  # noqa: E402


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], text=True).strip().splitlines()[0]
    except (OSError, subprocess.CalledProcessError) as e:
        return "unknown (%s)" % e


def stats(ts):
    ts = np.array(ts) * 1e6
    return "mean %.0f us, median %.0f us, min %.0f us" % (ts.mean(), np.median(ts), ts.min())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--seed", type=int, default=1)
    a = ap.parse_args()
    if orbx.lib().orbx_device_count() < 1:
        sys.exit("no CUDA device: this tool measures the GPU path")
    io = init_oracle.load()
    kp1, d1, prev, kp2, d2 = init_pair(a.seed, 5000)
    fv = orbx.FrameView(kp2, d2, SCALE, BOUNDS)
    bg = bounds_grid()
    lines = ["SearchForInitialization, MonocularInitialization shape: F1 %d features (%d at level 0), F2 %d features (%d at level 0), "
             "windowSize 100, nnratio 0.9, checkOri true" % (len(kp1), (kp1["octave"] == 0).sum(), len(kp2), (kp2["octave"] == 0).sum()),
             "card: %s" % card()]
    for _ in range(5):
        got = orbx.search_for_initialization(kp1, d1, fv, prev, 100, 0.9, True)
    ts = []
    for _ in range(50):
        t0 = time.perf_counter()
        got = orbx.search_for_initialization(kp1, d1, fv, prev, 100, 0.9, True)
        ts.append(time.perf_counter() - t0)
    rounds = orbx.projection_rounds()
    want = io.search_for_initialization(kp1, d1, kp2, d2, bg, prev, 100, 0.9, True)
    same = got[1] == want[1] and np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])
    cs = []
    for _ in range(10):
        t0 = time.perf_counter()
        io.search_for_initialization(kp1, d1, kp2, d2, bg, prev, 100, 0.9, True)
        cs.append(time.perf_counter() - t0)
    lines += ["GPU call (host arrays in, results out, 5 warm-up + 50 timed): %s" % stats(ts),
              "CPU oracle, one thread (g++ -O3, 10 timed): %s" % stats(cs),
              "speculation rounds (orbx_projection_rounds): %d" % rounds,
              "nmatches %d, identical to the oracle: %s" % (got[1], same)]
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
