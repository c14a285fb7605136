"""Loop closing's searches through the C++ class of csrc/adapter/ORBmatcher.h — both Sim3 SearchByProjection overloads, the Sim3
Fuse with the reference's declaration and the batched SearchAndFuse — against the reference loops restated over the same stand-in
types in tests/cpp/loop_adapter_test.cpp: the whole final state of identical worlds must agree."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "loop_adapter_test.cpp")
EXE = os.path.join(ROOT, "build", "loop_adapter_test")
SCENES = {0: "Replace gives the survivor a descriptor that matches another feature of the next key frame",
          1: "the survivor gains a slot of the next key frame and is skipped there", 2: "a pRep that is itself a loop point turns bad",
          3: "two loop points on one empty slot", 4: "slot holds a bad point", 5: "duplicate entry missed by the snapshot",
          6: "SearchByProjection, both overloads"}


def build_exe():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "tests", "cpp", "cv_stub"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200", "csrc", "adapter"), "-o", EXE, SRC,
                           "-L" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200"), "-lorbx",
                           "-Wl,-rpath," + os.path.join(ROOT, "wut_cuda_orb_slam3_b200")])


def test_loop_adapter_compiles():
    """CPU: the Sim3 members compile against stand-ins and link; the existing drivers' stand-ins have no Sim3 type, GetMapPoints
    or GetMap, which the member templates never instantiate for them (tests/test_adapter_fuse_cpp.py still compiles them)."""
    build_exe()
    assert os.path.exists(EXE)


def test_reference_scenes_do_what_they_say():
    """CPU: the reference loops alone on each scene (no device needed), checked against what the scene is built to exercise."""
    build_exe()
    out = {s: subprocess.run([EXE, str(s), "ref"], check=True, capture_output=True, text=True).stdout for s in SCENES}
    assert "nFused ref=2" in out[0] and "point 1 bad=1" in out[0] and "kf3/1" in out[0]        # matched Bk's second feature
    assert "nFused ref=1" in out[1] and "point 1 bad=0 nObs=2 obs: kf0/0 kf1/0\n" in out[1]   # no third observation from Bk
    assert "nFused ref=2" in out[2] and "point 0 bad=1" in out[2] and "point 1 bad=0 nObs=2 obs: kf0/0 kf1/1" in out[2]
    assert "nFused ref=2" in out[3] and "point 0 bad=1" in out[3] and "point 1 bad=0 nObs=1 obs: kf0/0" in out[3]
    assert "nFused ref=1" in out[4] and "point 1 bad=0 nObs=0 obs:\n" in out[4]
    assert "nFused ref=4" in out[5] and "point 0 bad=0 nObs=2 obs: kf0/0 kf1/0" in out[5]
    assert "nmatches ref=5,5 matched: 0/1 1/2 6/-1 2/1 3/2 3/1 4/-1 -1/-1" in out[6]


@pytest.mark.gpu
@pytest.mark.parametrize("scene", sorted(SCENES))
def test_loop_adapter_matches_reference_loop(scene):
    build_exe()
    r = subprocess.run([EXE, str(scene)], capture_output=True, text=True)
    assert r.returncode == 0, SCENES[scene] + "\n" + r.stdout + r.stderr
    if scene == 6:
        return
    m = re.search(r"researched=(\d+) calls=(\d+)", r.stdout)
    researched, calls = int(m.group(1)), int(m.group(2))
    if scene in (0, 2):
        assert researched == 1 and calls == 1                   # the stale pair of the next key frame, in one extra call
    else:
        assert researched == 0 and calls == 0
