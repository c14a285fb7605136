"""The batched ORBmatcher::SearchByBoW overloads of csrc/adapter/ORBmatcher.h (the candidate loop of Tracking::Relocalization and
the covisible loop of LoopClosing::DetectCommonRegionsFromBoW in one call each), driven by tests/cpp/bow_batch_adapter_test.cpp
against the same loops over the single overloads and over the CPU oracle, with NULL and bad key frames mixed in."""
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "bow_batch_adapter_test.cpp")
EXE = os.path.join(ROOT, "build", "bow_batch_adapter_test")
ORACLE_DIR = os.path.join(ROOT, "oracle", "_build")
LIB_DIR = os.path.join(ROOT, "wut_cuda_orb_slam3_b200")


def build_exe():
    from tests import oracle_lib
    oracle_lib.load()                              # builds oracle/_build/liborb_oracle.so if it is missing
    os.makedirs(os.path.dirname(EXE), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-Wall", "-I" + os.path.join(ROOT, "tests", "cpp", "cv_stub"), "-I" + os.path.join(ROOT, "include"),
                           "-I" + os.path.join(LIB_DIR, "csrc", "adapter"), "-o", EXE, SRC, "-L" + LIB_DIR, "-lorbx", "-L" + ORACLE_DIR,
                           "-lorb_oracle", "-Wl,-rpath," + LIB_DIR, "-Wl,-rpath," + ORACLE_DIR])


def write_set(f, desc, angle, mp_bits, fv):
    f.write(np.array([len(desc)], np.int32).tobytes())
    f.write(np.ascontiguousarray(desc, np.uint8).tobytes())
    f.write(np.ascontiguousarray(angle, np.float32).tobytes())
    f.write(np.ascontiguousarray(mp_bits, np.uint8).tobytes())
    f.write(np.array([len(fv.node_ids)], np.int32).tobytes())
    f.write(fv.node_ids.astype(np.uint32).tobytes()); f.write(fv.offsets.astype(np.int32).tobytes()); f.write(fv.indices.astype(np.uint32).tobytes())


@pytest.mark.gpu
def test_batched_overloads_match_single_and_oracle(tmp_path):
    import wut_cuda_orb_slam3_b200 as orbx
    from tests import bow_batch_synth as S
    from tests import bow_synth
    build_exe()
    parent, desc, weights = bow_synth.make_vocab(12, 10, 4)
    voc = orbx.ORBVocabulary(parent, desc, weights, 10, 4)
    sizes = [900, 1200, 700, 1000, 0, 800, 1100, 600, 1000, 950]
    kinds = [S.NORMAL] * len(sizes)
    kinds[4] = S.EMPTY
    kinds[7] = S.DISJOINT
    B = S.attach_fvs(S.make_batch(41, desc, parent, 1000, sizes, kinds), lambda d: voc.transform(d, 2)[1])
    # slot states: 0 = key frame, 1 = NULL, 2 = isBad()
    state = np.array([0, 1, 0, 2, 0, 0, 2, 0, 1, 0], np.int32)
    rng = np.random.default_rng(5)

    def bits(valid):                               # bit 0: the feature holds a map point, bit 1: that map point isBad()
        return (valid | ((rng.random(len(valid)) < 0.05).astype(np.uint8) << 1)).astype(np.uint8)
    scene = tmp_path / "scene.bin"
    with open(scene, "wb") as f:
        f.write(np.array([len(sizes)], np.int32).tobytes()); f.write(state.tobytes())
        write_set(f, B["desc"], B["angle"], bits(B["valid"]), B["fv"])
        for kf in B["kfs"]:
            write_set(f, kf["desc"], kf["angle"], bits(kf["valid"]), kf["fv"])
    r = subprocess.run([EXE, str(scene)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    m = re.search(r"reloc=(\d+) loop=(\d+)", r.stdout)
    assert m and int(m.group(1)) > 300 and int(m.group(2)) > 300, r.stdout
