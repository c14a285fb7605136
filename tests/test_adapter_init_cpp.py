"""ORBmatcher::SearchForInitialization through the C++ class of csrc/adapter/ORBmatcher.h (the reference's declaration, cv::Point2f
vbPrevMatched), driven like Tracking::MonocularInitialization, against the oracle's sequential loop."""
import os
import subprocess

import numpy as np
import pytest

from tests.init_synth import bounds_grid, init_pair, next_frame
from tests.proj_synth import SCALE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "initialization_adapter_test.cpp")
EXE = os.path.join(ROOT, "build", "initialization_adapter_test")


def build_exe():
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "tests", "cpp", "cv_stub"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200", "csrc", "adapter"), "-o", EXE, SRC,
                           "-L" + os.path.join(ROOT, "wut_cuda_orb_slam3_b200"), "-lorbx",
                           "-Wl,-rpath," + os.path.join(ROOT, "wut_cuda_orb_slam3_b200")])


def test_initialization_adapter_compiles():
    """CPU: ORBmatcher::SearchForInitialization with the reference's declaration compiles and links (no compute call)."""
    build_exe()
    assert os.path.exists(EXE)


@pytest.mark.gpu
@pytest.mark.parametrize("check_ori", [True, False])
def test_initialization_adapter_matches_oracle(tmp_path, check_ori):
    from tests import init_oracle
    io = init_oracle.load()
    build_exe()
    kp1, d1, prev, kp2, d2 = init_pair(71 + int(check_ori), 5000)
    kp3, d3 = next_frame(81, kp2, d2)
    bg = bounds_grid()
    ratio, window = 0.9, 100
    scene = tmp_path / "scene.bin"; result = tmp_path / "result.bin"
    with open(scene, "wb") as f:
        f.write(np.array([len(kp1), len(kp2), len(kp3), len(SCALE), window, int(check_ori)], np.int32).tobytes())
        f.write(np.array(list(bg) + [ratio], np.float32).tobytes()); f.write(SCALE.tobytes())
        for kp, d in ((kp1, d1), (kp2, d2), (kp3, d3)):
            f.write(kp.tobytes()); f.write(d.tobytes())
    subprocess.check_call([EXE, str(scene), str(result)])
    raw = np.fromfile(result, np.uint8)
    n1 = len(kp1)
    rec = 4 + 4 * n1 + 8 * n1
    assert len(raw) == 2 * rec
    for k, (kp, d) in enumerate(((kp2, d2), (kp3, d3))):
        r = raw[k * rec:(k + 1) * rec]
        nm = int(r[:4].view(np.int32)[0]); m12 = r[4:4 + 4 * n1].view(np.int32); out = r[4 + 4 * n1:].view(np.float32).reshape(n1, 2)
        want, wnm, prev = io.search_for_initialization(kp1, d1, kp, d, bg, prev, window, ratio, check_ori)
        assert nm == wnm and nm > 500 and np.array_equal(m12, want) and np.array_equal(out, prev), k
