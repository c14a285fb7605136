#!/usr/bin/env python3
"""Generates tests/golden/ref_golden.json from the REFERENCE's own compiled functions (oracle/_ref/libref.so, built by
oracle/build_ref.sh from the reference checkout named by ORB_REFERENCE_ROOT).  tests/test_golden.py re-computes every case with
the oracle and compares, so the pin holds where neither the reference nor libref.so exists.  Run from the repo root:
    ORB_REFERENCE_ROOT=<checkout> sh oracle/build_ref.sh && python tests/golden/make_ref_golden.py
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import oracle_lib, ref_cases, ref_lib  # noqa: E402


def main():
    assert ref_lib.available(), "oracle/_ref/libref.so missing: run sh oracle/build_ref.sh (needs ORB_REFERENCE_ROOT)"
    out = {"generator": "tests/golden/make_ref_golden.py (reference functions compiled by oracle/build_ref.sh)",
           "cases": ref_cases.run_all(oracle_lib.load(), ref_lib.load())}
    with open(os.path.join(ROOT, "tests", "golden", "ref_golden.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote %d cases" % len(out["cases"]))


if __name__ == "__main__":
    main()
