"""Writes tests/golden/init_golden.json: SearchForInitialization answers of the oracle (tests/cpp/init_oracle.cpp) on seeded
initialisation pairs (tests/init_synth.py).  Run from the repository root: python tests/golden/make_init_golden.py"""
import json
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from tests import init_oracle  # noqa: E402
from tests.init_synth import bounds_grid, init_pair  # noqa: E402

CASES = [dict(seed=901, n2=5000, crowd=0, dup=1, window=100, ratio=0.9, check_orientation=True),
         dict(seed=902, n2=5000, crowd=0, dup=1, window=100, ratio=0.9, check_orientation=False),
         dict(seed=903, n2=1200, crowd=5, dup=3, window=100, ratio=0.9, check_orientation=True),
         dict(seed=904, n2=800, crowd=3, dup=4, window=50, ratio=0.7, check_orientation=True)]


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def main():
    o = init_oracle.load()
    out = []
    for c in CASES:
        kp1, d1, prev, kp2, d2 = init_pair(c["seed"], c["n2"], crowd=c["crowd"], dup=c["dup"])
        m, nm, p = o.search_for_initialization(kp1, d1, kp2, d2, bounds_grid(), prev, c["window"], c["ratio"], c["check_orientation"])
        out.append(dict(c, kp1_crc=crc(kp1), desc1_crc=crc(d1), kp2_crc=crc(kp2), desc2_crc=crc(d2), n_matches=int(nm),
                        matches12_crc=crc(m), prev_crc=crc(p)))
        print(c["seed"], len(kp1), nm)
    with open(os.path.join(ROOT, "tests", "golden", "init_golden.json"), "w") as f:
        json.dump({"generator": "tests/golden/make_init_golden.py", "cases": out}, f, indent=1)
        f.write("\n")


if __name__ == "__main__":
    main()
