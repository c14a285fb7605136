"""Writes tests/golden/fuse_golden.json: answers of the Fuse oracle (tests/cpp/fuse_oracle.cpp) on seeded local-mapping scenes
(tests/fuse_synth.py).  Run from the repository root: python tests/golden/make_fuse_golden.py"""
import json
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import fuse_oracle  # noqa: E402
from tests.fuse_synth import scene  # noqa: E402

CASES = [dict(seed=951, n_kf=8, n_points=1200, crowd=0, th=3.0),
         dict(seed=952, n_kf=4, n_points=800, crowd=5, th=3.0),
         dict(seed=953, n_kf=3, n_points=1000, crowd=0, th=5.0)]


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def main():
    o = fuse_oracle.load()
    out = []
    for c in CASES:
        X, pd, kfs, P = scene(c["seed"], n_kf=c["n_kf"], n_points=c["n_points"], crowd=c["crowd"], forward=True)
        m, nf = o.fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], c["th"])
        out.append(dict(c, kp_crc=crc(np.concatenate([k["kp"] for k in kfs])), desc_crc=crc(pd), u_crc=crc(P["u"]), match_crc=crc(m),
                        n_fused=nf.tolist()))
        print(c["seed"], len(m), nf.tolist())
    with open(os.path.join(ROOT, "tests", "golden", "fuse_golden.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_fuse_golden.py", "cases": out}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
