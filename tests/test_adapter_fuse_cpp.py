"""ORBmatcher::Fuse through the C++ class of csrc/adapter/ORBmatcher.h (the reference's declaration, and the batched overload for
the forward loop of LocalMapping::SearchInNeighbors), against the reference's Fuse loop restated over the same stand-in
KeyFrame / MapPoint types in tests/cpp/fuse_adapter_test.cpp: the whole final state of two identical worlds must agree."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "fuse_adapter_test.cpp")
EXE = os.path.join(ROOT, "build", "fuse_adapter_test")
SCENES = {0: "same empty slot, both Replace directions, tie", 1: "slot holds a bad point", 2: "replaced in A, skipped in B",
          3: "new descriptor after Replace matches another feature in B", 4: "gains an observation of B through Replace",
          5: "duplicate entry fires the in-loop re-search"}


def build_exe():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "tests", "cpp", "cv_stub"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200", "csrc", "adapter"), "-o", EXE, SRC,
                           "-L" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200"), "-lorbx",
                           "-Wl,-rpath," + os.path.join(ROOT, "wut_cuda_orb_slam3_b200")])


def test_fuse_adapter_compiles():
    """CPU: both Fuse overloads compile against stand-ins and link; the existing adapter drivers still compile (their stand-ins
    lack what Fuse reads, which the member templates never instantiate for them)."""
    build_exe()
    assert os.path.exists(EXE)


def test_reference_scenes_do_what_they_say():
    """CPU: the reference loop alone on each scene (no device needed), checked against what the scene is built to exercise."""
    build_exe()
    out = {s: subprocess.run([EXE, str(s), "ref"], check=True, capture_output=True, text=True).stdout for s in SCENES}
    assert "nFused ref=5" in out[0] and "point 1 bad=1" in out[0] and "point 4 bad=1" in out[0] and "point 6 bad=1" in out[0]
    assert "point 7 bad=0 nObs=4" in out[0]                     # tie: the slot's point was replaced
    assert "nFused ref=1" in out[1] and "point 1 bad=0 nObs=0 obs: desc" in out[1]
    assert "nFused ref=1" in out[2] and "point 1 bad=1" in out[2]
    assert "nFused ref=2" in out[3] and "kf3/1" in out[3]       # matched the second feature of B (the new descriptor's)
    assert "nFused ref=1" in out[4] and "point 1 bad=0 nObs=7 obs: kf0/0 kf1/0" in out[4]
    assert "nFused ref=2" in out[5]


@pytest.mark.gpu
@pytest.mark.parametrize("scene", sorted(SCENES))
def test_fuse_adapter_matches_reference_loop(scene):
    build_exe()
    r = subprocess.run([EXE, str(scene)], capture_output=True, text=True)
    assert r.returncode == 0, SCENES[scene] + "\n" + r.stdout + r.stderr
    m = re.search(r"researched=(\d+) calls=(\d+)", r.stdout)
    researched, calls = int(m.group(1)), int(m.group(2))
    if scene == 3:
        assert researched > 0 and calls == 1                   # the stale pair of B, in one extra call before B is applied
    if scene == 5:
        assert researched == 1 and calls == 1                  # the safety net inside the apply loop
    if scene in (0, 1, 2, 4):
        assert researched == 0 and calls == 0
