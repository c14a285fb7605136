"""ORBmatcher::SearchForTriangulation through the C++ class of csrc/adapter/ORBmatcher.h (the reference's declaration, and the
batched overload for the neighbour loop of LocalMapping::CreateNewMapPoints), against the reference restated over the same
stand-in KeyFrame / MapPoint types in tests/cpp/triangulation_adapter_test.cpp: per-neighbour matches, return values and the
final map-point slots of a CreateNewMapPoints-shaped loop must agree."""
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "triangulation_adapter_test.cpp")
EXE = os.path.join(ROOT, "build", "triangulation_adapter_test")
SCENES = {0: "a KF1 feature matched by neighbour 0 is dropped from later neighbours", 1: "rotation filter after the drop",
          2: "the body changes a later neighbour's slot", 3: "early stop", 4: "two-camera key frame throws",
          5: "overlapping neighbours, stereo only, mixed coarse, rotation filter"}


def build_exe():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "tests", "cpp", "cv_stub"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200", "csrc", "adapter"), "-o", EXE, SRC,
                           "-L" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200"), "-lorbx",
                           "-Wl,-rpath," + os.path.join(ROOT, "wut_cuda_orb_slam3_b200")])


def ref_counts(scene):
    out = subprocess.run([EXE, str(scene), "ref"], check=True, capture_output=True, text=True).stdout
    return [int(x) for x in re.search(r"ref n=([\d ]*)", out).group(1).split()]


def test_triangulation_adapter_compiles():
    """CPU: both SearchForTriangulation overloads compile against the stand-ins and link; the other adapter drivers, whose
    stand-ins lack what these members read, still compile because the member templates are never instantiated for them."""
    build_exe()
    assert os.path.exists(EXE)


def test_reference_scenes_do_what_they_say():
    """CPU: the reference loop alone on each scene (no device needed), checked against what the scene is built for."""
    build_exe()
    assert ref_counts(0) == [55, 10, 0]          # neighbours 1 and 2 see the 60 points neighbour 0 took (5 were occupied)
    assert ref_counts(1) == [150, 10]            # neighbour 1 keeps its 10 matches of rotation bin 5
    assert ref_counts(2) == [20, 20, 19]         # the poked feature of neighbour 2 is no longer a candidate
    assert ref_counts(3) == [30, 10]             # stopped after neighbour 1; neighbour 1 overlaps neighbour 0 in 20 points
    c = ref_counts(5)
    assert len(c) == 4 and min(c) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("scene", sorted(SCENES))
def test_triangulation_adapter_matches_reference_loop(scene):
    build_exe()
    r = subprocess.run([EXE, str(scene)], capture_output=True, text=True)
    assert r.returncode == 0, SCENES[scene] + "\n" + r.stdout + r.stderr
    if scene == 4:
        return
    m = re.search(r"researched=(\d+) dropped=(\d+)", r.stdout)
    researched, dropped = int(m.group(1)), int(m.group(2))
    assert researched == (1 if scene == 2 else 0)
    if scene in (0, 1):
        assert dropped > 0
