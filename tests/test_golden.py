"""Known-answer tests against the committed fixture tests/golden/orb_golden.json (made by tests/golden/make_golden.py).
CPU: the oracle still reproduces the fixture.  GPU: the CUDA path reproduces the fixture without touching oracle code."""
import json
import os
import zlib

import numpy as np
import pytest

from wut_cuda_orb_slam3_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = json.load(open(os.path.join(ROOT, "tests", "golden", "orb_golden.json")))


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def check_case(ex, c, extract):
    img = synth.image(c["seed"], c["cols"], c["rows"])
    assert crc(img) == c["image_crc"]
    kps, desc, nm = extract(img, tuple(c["lapping"]))
    assert (len(kps), nm) == (c["n"], c["n_mono"])
    assert crc(kps) == c["keypoints_crc"] and crc(desc) == c["descriptors_crc"]
    for l, g in enumerate(c["levels"]):
        assert crc(ex.pyramid_level(l, with_border=True)) == g["pyramid_crc"], l
        assert crc(ex.blurred_level(l)) == g["blur_crc"], l
        xs, ys, sc = ex.candidates(l)
        assert len(xs) == g["n_candidates"] and crc(np.stack([xs, ys, sc], 1).astype(np.int32)) == g["candidates_crc"], l
        lk, ld = ex.level_keypoints(l)
        assert len(lk) == g["n_keypoints"], l
        assert crc(np.stack([lk["x"], lk["y"], lk["response"]], 1).astype(np.float32)) == g["keypoints_xy_crc"], l
        assert crc(lk["angle"]) == g["angles_crc"] and crc(ld) == g["desc_crc"], l
    if "keypoints" in c:
        for k, ref in zip(kps, c["keypoints"]):
            assert [float(k["x"]), float(k["y"]), float(k["size"]), float(k["angle"]), float(k["response"]), int(k["octave"])] == ref
        assert [bytes(d).hex() for d in desc[:40]] == c["descriptors_hex"]


@pytest.mark.parametrize("i", range(len(GOLD["cases"])))
def test_oracle_reproduces_golden(oracle, i):
    c = GOLD["cases"][i]
    ex = oracle.extractor(c["nfeatures"], 1.2, 8, 20, 7)
    check_case(ex, c, lambda img, lap: ex.extract(img, lap))


def test_oracle_knn2_golden(oracle):
    g = GOLD["knn2"]
    db = synth.descriptors(g["seed"], g["ndb"]); q = synth.descriptors(g["seed"], g["nq"], is_query=True, ndb=g["ndb"], plant_every=g["plant_every"])
    idx, dist = oracle.knn2(q, db)
    assert crc(idx) == g["idx_crc"] and crc(dist) == g["dist_crc"]


@pytest.mark.gpu
@pytest.mark.parametrize("i", range(len(GOLD["cases"])))
def test_cuda_reproduces_golden(i):
    import wut_cuda_orb_slam3_b200 as orbx
    c = GOLD["cases"][i]
    ex = orbx.ORBextractor(c["nfeatures"], 1.2, 8, 20, 7)

    def extract(img, lap):
        nm, kps, desc = ex(img, None, lap)
        return kps, desc, nm
    check_case(ex, c, extract)


@pytest.mark.gpu
def test_cuda_knn2_golden():
    import wut_cuda_orb_slam3_b200 as orbx
    g = GOLD["knn2"]
    db = synth.descriptors(g["seed"], g["ndb"]); q = synth.descriptors(g["seed"], g["nq"], is_query=True, ndb=g["ndb"], plant_every=g["plant_every"])
    idx, dist = orbx.ORBmatcher().knn2(q, db)
    assert crc(idx) == g["idx_crc"] and crc(dist) == g["dist_crc"]
    assert idx[:8].tolist() == g["first"][0] and dist[:8].tolist() == g["first"][1]


def test_oracle_reproduces_reference_golden(oracle):
    """tests/golden/ref_golden.json holds answers of the REFERENCE's own compiled functions (oracle/_ref, made by
    tests/golden/make_ref_golden.py where the reference is built); the oracle must reproduce every one of them."""
    import json
    import os

    from tests import ref_cases
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_golden.json")) as f:
        gold = json.load(f)["cases"]
    got = ref_cases.run_all(oracle)
    assert set(got) == set(gold)
    bad = [k for k in gold if got[k] != gold[k]]
    assert not bad, bad
