"""Per-call latency of loop closing's two searches, next to the CPU oracle's single-thread time on the same inputs.

  Sim3 SearchByProjection (orbx_search_by_projection_sim3): 1 key frame (~2000 features, 30 % of its slots matched on entry)
      x 8000 points, at the DetectCommonRegionsFromBoW shape (th 8, ratio 1.5) and the FindMatchesByProjection shape (3, 1.5),
      with the speculation rounds each needed;
  Sim3 Fuse (orbx_fuse_sim3) at the shape of LoopClosing::SearchAndFuse: 30 key frames x 5000 loop points, timed as ONE batched
      call, as 30 per-key-frame calls, and as the oracle on one CPU thread.

Each GPU call takes host arrays and returns host results (one pinned upload, the kernels, one download and a stream synchronise
inside the call), so the host clock around it measures the whole call.  5 warm-up calls, then 50 timed calls; the results must
be identical to the oracle's.  The card's name and power limit are read with a read-only nvidia-smi query in the same run.

    python tools/loop_latency.py [--out FILE]
"""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import wut_cuda_orb_slam3_b200 as orbx  # noqa: E402
from tests import loop_oracle  # noqa: E402
from tests.fuse_synth import BOUNDS  # noqa: E402
from tests.loop_synth import fuse_scene, sbp_scene  # noqa: E402
from tools.fuse_latency import card, stats, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if orbx.lib().orbx_device_count() < 1:
        sys.exit("no CUDA device: this tool measures the GPU path")
    lo = loop_oracle.load()
    lines = ["Loop closing's Sim3 searches; scenes of tests/loop_synth.py (752 x 480, 8 levels, monocular key frames)", "card: %s" % card()]
    same = True
    # Sim3 SearchByProjection
    K, occ, P, pd = sbp_scene(1, n_points=8000, see=0.22, n_distract=400)
    fv = orbx.FrameView(K["kp"], K["desc"], K["scale"], BOUNDS, occupied=occ)
    lines.append("SearchByProjection (Sim3): 1 key frame (%d features, %d matched on entry) x %d points, %d valid" %
                 (len(K["kp"]), int(occ.sum()), len(P["u"]), int(P["valid"].sum())))
    for name, th, ratio in (("DetectCommonRegionsFromBoW", 8, 1.5), ("FindMatchesByProjection", 3, 1.5)):
        args = (P["valid"], P["u"], P["v"], P["level"], pd, th, ratio)
        want = lo.search_by_projection_sim3(K, occ, *args)
        got, t_gpu = timed(lambda: orbx.search_by_projection_sim3(fv, *args))
        rounds = orbx.projection_rounds()
        same &= got[1] == want[1] and np.array_equal(got[0], want[0])
        _, t_cpu = timed(lambda: lo.search_by_projection_sim3(K, occ, *args), warm=1, n=10)
        lines += ["  %s (th %d, ratio %.1f): %d matches, %d speculation rounds" % (name, th, ratio, want[1], rounds),
                  "    one call (5 warm-up + 50 timed): %s" % stats(t_gpu),
                  "    CPU oracle, one thread (g++ -O3, 1 warm-up + 10 timed): %s" % stats(t_cpu)]
    # Sim3 Fuse, SearchAndFuse
    n_kf, M = 30, 5000
    kfs, P, pd = fuse_scene(3, n_kf=n_kf, n_points=M, n_distract=800)
    V = [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS) for k in kfs]
    args = (P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], 4.0)
    want = lo.fuse_sim3(kfs, *args)
    got, t_batch = timed(lambda: orbx.fuse_sim3(V, *args))
    same &= np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    sub = [(k, P["kf_offsets"][k], P["kf_offsets"][k + 1]) for k in range(n_kf)]

    def per_kf():
        return [orbx.fuse_sim3([V[k]], [0, q1 - q0], pd, P["point"][q0:q1], P["valid"][q0:q1], P["u"][q0:q1], P["v"][q0:q1],
                               P["level"][q0:q1], 4.0) for k, q0, q1 in sub]
    got_k, t_loop = timed(per_kf)
    same &= np.array_equal(np.concatenate([g[0] for g in got_k]), want[0])
    _, t_cpu = timed(lambda: lo.fuse_sim3(kfs, *args), warm=1, n=10)
    nfeat = sum(len(k["kp"]) for k in kfs)
    lines += ["Fuse (Sim3), SearchAndFuse: %d key frames (%d features in all) x %d loop points = %d pairs, %d valid, %d fused, th 4" %
              (n_kf, nfeat, M, len(P["u"]), int(P["valid"].sum()), int(want[1].sum())),
              "  one batched call (5 warm-up + 50 timed): %s" % stats(t_batch),
              "  %d per-key-frame calls (5 warm-up + 50 timed): %s" % (n_kf, stats(t_loop)),
              "  CPU oracle, one thread (g++ -O3, 1 warm-up + 10 timed): %s" % stats(t_cpu),
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
