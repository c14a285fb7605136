"""Writes tests/golden/loop_golden.json: answers of the loop-closing oracle (tests/cpp/loop_oracle.cpp) on seeded scenes
(tests/loop_synth.py): the Sim3 SearchByProjection at the shapes of DetectCommonRegionsFromBoW and FindMatchesByProjection, and
the Sim3 Fuse over several key frames.  Run from the repository root: python tests/golden/make_loop_golden.py"""
import json
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import loop_oracle  # noqa: E402
from tests.loop_synth import fuse_scene, sbp_scene  # noqa: E402

CASES = [dict(kind="sbp", seed=961, n_points=3000, crowd=0, th=8, ratio=1.5),
         dict(kind="sbp", seed=962, n_points=2000, crowd=5, th=5, ratio=1.0),
         dict(kind="sbp", seed=963, n_points=3000, crowd=0, th=3, ratio=1.5),
         dict(kind="fuse", seed=964, n_kf=6, n_points=1000, crowd=0, th=4.0),
         dict(kind="fuse", seed=965, n_kf=3, n_points=800, crowd=5, th=4.0)]


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def main():
    o = loop_oracle.load()
    out = []
    for c in CASES:
        if c["kind"] == "sbp":
            K, occ, P, pd = sbp_scene(c["seed"], n_points=c["n_points"], crowd=c["crowd"])
            kfs = [K]
            m, n = o.search_by_projection_sim3(K, occ, P["valid"], P["u"], P["v"], P["level"], pd, c["th"], c["ratio"])
        else:
            kfs, P, pd = fuse_scene(c["seed"], n_kf=c["n_kf"], n_points=c["n_points"], crowd=c["crowd"])
            m, nf = o.fuse_sim3(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], c["th"])
            n = nf.tolist()
        out.append(dict(c, kp_crc=crc(np.concatenate([k["kp"] for k in kfs])), desc_crc=crc(pd), u_crc=crc(P["u"]), match_crc=crc(m), n=n))
        print(c["kind"], c["seed"], len(m), n)
    with open(os.path.join(ROOT, "tests", "golden", "loop_golden.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_loop_golden.py", "cases": out}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
