"""Per-call latency of ORBmatcher::SearchByBoW at the shapes of the two place-recognition loops, next to the CPU oracle's
single-thread time on the same inputs.

  Relocalization: mode 0 (KF -> Frame), ORBmatcher(0.75, true), a 1000-feature Frame against 20 candidate key frames of 1000
                  features (Tracking::Relocalization).
  Loop detection: mode 1 (KF -> KF), ORBmatcher(0.9, true), a 1200-feature KF1 against 30 KF2s of 1200 features
                  (LoopClosing::DetectCommonRegionsFromBoW).
Each is timed as ONE orbx_search_by_bow_batch call, as one orbx_search_by_bow call per key frame, and as the oracle on one CPU
thread.  Batches of tests/bow_batch_synth.py, vocabulary k = 10, L = 4, nodes at levelsup 2.

Each GPU call takes host arrays and returns host results (upload, kernels, download and a synchronise inside the call), so the
host clock around it measures the whole call.  5 warm-up calls, then 50 timed calls, for all three.  The tool fails unless the
batched rows equal the single calls and the oracle.  The card's name, power limit and SM clocks are read with a read-only
nvidia-smi query in the same run.

    python tools/bow_batch_latency.py [--out FILE]
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
from tests import bow_batch_synth, bow_synth, oracle_lib  # noqa: E402


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
    voc = orbx.ORBVocabulary(parent, desc, weights, 10, 4)
    lines = ["ORBmatcher::SearchByBoW with the rotation filter; batches of tests/bow_batch_synth.py (vocabulary k = 10, L = 4, nodes at levelsup 2)",
             "card (name, power limit, SM clock, max SM clock): %s" % card()]
    same = True
    for name, mode, ratio, n, n_kf in (("Relocalization (mode 0, KF -> Frame)", 0, 0.75, 1000, 20),
                                       ("Loop detection (mode 1, KF -> KF)", 1, 0.9, 1200, 30)):
        B = bow_batch_synth.attach_fvs(bow_batch_synth.make_batch(500 + mode, desc, parent, n, [n] * n_kf),
                                       lambda d: voc.transform(d, 2)[1])
        valid = B["valid"] if mode == 1 else None
        (m, nm), t_batch = timed(lambda: orbx.search_by_bow_batch(B["desc"], B["angle"], valid, B["fv"], B["kfs"], kf_kf=mode == 1, nnratio=ratio))

        def per_kf():
            if mode == 0:
                return [orbx.search_by_bow(kf["desc"], kf["angle"], kf["valid"], kf["fv"], B["desc"], B["angle"], B["fv"], nnratio=ratio)[0::2]
                        for kf in B["kfs"]]
            return [orbx.search_by_bow(B["desc"], B["angle"], B["valid"], B["fv"], kf["desc"], kf["angle"], kf["fv"], valid_b=kf["valid"],
                                       kf_kf=True, nnratio=ratio)[1:] for kf in B["kfs"]]
        rows, t_loop = timed(per_kf)

        def oracle():
            if mode == 0:
                return [o.search_by_bow_kf_frame(kf["desc"], kf["angle"], kf["valid"], fvt(kf["fv"]), B["desc"], B["angle"], fvt(B["fv"]), -1,
                                                 ratio, True) for kf in B["kfs"]]
            return [o.search_by_bow_kf_kf(B["desc"], B["angle"], B["valid"], fvt(B["fv"]), kf["desc"], kf["angle"], kf["valid"], fvt(kf["fv"]),
                                          ratio, True) for kf in B["kfs"]]
        want, t_cpu = timed(oracle)
        ok = True
        for k in range(n_kf):
            ok &= np.array_equal(m[k], rows[k][0]) and nm[k] == rows[k][1]
            ok &= np.array_equal(m[k], want[k][0]) and nm[k] == want[k][1]
        same &= ok
        lines += ["%s: ratio %.2f, %d features against %d key frames of %d features, %d matches in all" % (name, ratio, n, n_kf, n, int(nm.sum())),
                  "  one batched call (5 warm-up + 50 timed): %s" % stats(t_batch),
                  "  %d single calls (5 warm-up + 50 timed): %s" % (n_kf, stats(t_loop)),
                  "  CPU oracle, one thread (g++ -O3, 5 warm-up + 50 timed): %s" % stats(t_cpu),
                  "  batched rows identical to the single calls and to the oracle: %s" % ok]
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(text)
    if not same:
        sys.exit("batched result differs from the single calls or the oracle")


if __name__ == "__main__":
    main()
