"""Per-call latency of ORBmatcher::SearchForTriangulation at the shapes of LocalMapping::CreateNewMapPoints (one key frame
against its neighbours), next to the CPU oracle's single-thread time on the same inputs.

  10 neighbours x 1200 features (stereo / RGB-D: nn = 10) and 30 neighbours x 1500 features (monocular: nn = 30), each timed as
  ONE orbx_search_for_triangulation_batch call, as one orbx_search_for_triangulation call per neighbour, and as the oracle on one
  CPU thread.  bCoarse = false, no rotation filter: ORBmatcher(0.6, false) as CreateNewMapPoints builds it.

Each GPU call takes host arrays and returns host results (uploads, kernels, download and a synchronise inside the call), so the
host clock around it measures the whole call.  5 warm-up calls, then 50 timed calls.  The tool fails unless the batched output
equals the per-neighbour output and the oracle's.  The card's name, power limit and SM clocks are read with a read-only
nvidia-smi query in the same run.

    python tools/triangulation_latency.py [--out FILE]
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
from tests import bow_synth, oracle_lib  # noqa: E402
from tests.tri_synth import make_scene  # noqa: E402


def card():
    try:
        return subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                                       text=True).strip().splitlines()[0]
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


def fvt(fv):
    return (fv.node_ids, fv.offsets, fv.indices)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if orbx.lib().orbx_device_count() < 1:
        sys.exit("no CUDA device: this tool measures the GPU path")
    o = oracle_lib.load()
    parent, desc, weights = bow_synth.make_vocab(601, 10, 4)
    voc = (orbx.ORBVocabulary(parent, desc, weights, 10, 4), desc, parent)
    lines = ["ORBmatcher::SearchForTriangulation (bOnlyStereo false, bCoarse false, no rotation filter); scenes of tests/tri_synth.py "
             "(752 x 480, vocabulary k = 10, L = 4, nodes at levelsup 2, 4-12 levels per neighbour)",
             "card (name, power limit, SM clock, max SM clock): %s" % card()]
    same = True
    for n_kf, n in ((10, 1200), (30, 1500)):
        A, nbs = make_scene(voc, 100 + n_kf, n, n_kf, n)
        args = (A["kp"], A["desc"], A["free"], A["stereo"], A["fv"])
        (m, nm), t_batch = timed(lambda: orbx.search_for_triangulation_batch(*args, nbs, check_orientation=False))

        def per_kf():
            return [orbx.search_for_triangulation(*args, nb["kp"], nb["desc"], nb["free"], nb["stereo"], nb["fv"], nb["F12"], nb["ep"],
                                                  nb["scale"], nb["sigma2"], check_orientation=False) for nb in nbs]
        rows, t_loop = timed(per_kf)

        def oracle():
            return [o.search_for_triangulation(A["kp"], A["desc"], A["free"], A["stereo"], fvt(A["fv"]), nb["kp"], nb["desc"], nb["free"],
                                               nb["stereo"], fvt(nb["fv"]), nb["F12"], nb["ep"], nb["scale"], nb["sigma2"], False, False, False)
                    for nb in nbs]
        want, t_cpu = timed(oracle, warm=1, n=10)
        for k in range(n_kf):
            same &= np.array_equal(m[k], rows[k][0]) and nm[k] == rows[k][1]
            same &= np.array_equal(m[k], want[k][0]) and nm[k] == want[k][1]
        lines += ["%d neighbours x %d features (KF1 %d features, %d free), %d matches in all" % (n_kf, n, n, int(A["free"].sum()), int(nm.sum())),
                  "  one batched call (5 warm-up + 50 timed): %s" % stats(t_batch),
                  "  %d per-neighbour calls (5 warm-up + 50 timed): %s" % (n_kf, stats(t_loop)),
                  "  CPU oracle, one thread (g++ -O3, 1 warm-up + 10 timed): %s" % stats(t_cpu)]
    lines.append("batched identical to the per-neighbour calls and to the oracle: %s" % same)
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    if not same:
        sys.exit("batched result differs from the per-neighbour calls or the oracle")


if __name__ == "__main__":
    main()
