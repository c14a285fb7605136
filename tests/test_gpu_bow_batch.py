"""orbx_search_by_bow_batch on the GPU: every row against orbx_search_by_bow on that key frame and against the CPU oracle
(bit-exact), in both modes, over the edge cases of tests/bow_batch_synth.py, argument errors and two threads at once."""
import ctypes as C
import threading

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import bow_batch_synth as S
from tests import bow_synth
from wut_cuda_orb_slam3_b200 import capi

pytestmark = pytest.mark.gpu


def fv_tuple(fv):
    return (fv.node_ids, fv.offsets, fv.indices)


@pytest.fixture(scope="module")
def voc():
    parent, desc, weights = bow_synth.make_vocab(601, 10, 4)
    return orbx.ORBVocabulary(parent, desc, weights, 10, 4), parent, desc


def make(voc, seed, n, sizes, kinds=None, levelsup=2):
    v, parent, desc = voc
    return S.attach_fvs(S.make_batch(seed, desc, parent, n, sizes, kinds), lambda d: v.transform(d, levelsup)[1])


def batch(B, mode, nleft=-1, ratio=0.6, check_ori=True):
    return orbx.search_by_bow_batch(B["desc"], B["angle"], B["valid"] if mode == 1 else None, B["fv"], B["kfs"], kf_kf=mode == 1,
                                    nleft=nleft, nnratio=ratio, check_orientation=check_ori)


def check_rows(oracle, B, mode, match, nm, nleft=-1, ratio=0.6, check_ori=True):
    """Row k == the single call on key frame k == the oracle; returns the total."""
    n = len(B["desc"])
    assert match.shape == (len(B["kfs"]), n) and nm.shape == (len(B["kfs"]),)
    for k, kf in enumerate(B["kfs"]):
        if mode == 0:
            one, _, n1 = orbx.search_by_bow(kf["desc"], kf["angle"], kf["valid"], kf["fv"], B["desc"], B["angle"], B["fv"], nleft_b=nleft,
                                            nnratio=ratio, check_orientation=check_ori)
            want, wn = oracle.search_by_bow_kf_frame(kf["desc"], kf["angle"], kf["valid"], fv_tuple(kf["fv"]), B["desc"], B["angle"],
                                                     fv_tuple(B["fv"]), nleft, ratio, check_ori)
        else:
            _, one, n1 = orbx.search_by_bow(B["desc"], B["angle"], B["valid"], B["fv"], kf["desc"], kf["angle"], kf["fv"], valid_b=kf["valid"],
                                            kf_kf=True, nnratio=ratio, check_orientation=check_ori)
            want, wn = oracle.search_by_bow_kf_kf(B["desc"], B["angle"], B["valid"], fv_tuple(B["fv"]), kf["desc"], kf["angle"], kf["valid"],
                                                  fv_tuple(kf["fv"]), ratio, check_ori)
        assert np.array_equal(match[k], one) and nm[k] == n1, (k, kf["kind"])
        assert np.array_equal(match[k], want) and nm[k] == wn, (k, kf["kind"])
        assert nm[k] == int((match[k] >= 0).sum())
    return int(nm.sum())


# (mode, n_kf, ratio, check_orientation, nleft); the fixed side has 2000 features, key frames 150..2000
CASES = [(0, 1, 0.6, True, -1), (0, 7, 0.75, True, -1), (0, 64, 0.75, True, -1), (0, 7, 0.9, False, -1), (0, 64, 0.6, False, -1),
         (0, 7, 0.6, True, 1100), (0, 64, 0.9, True, 700),
         (1, 1, 0.9, True, -1), (1, 7, 0.6, True, -1), (1, 64, 0.9, True, -1), (1, 7, 0.75, False, -1), (1, 64, 0.6, False, -1)]


@pytest.mark.parametrize("mode,n_kf,ratio,check_ori,nleft", CASES)
def test_rows_equal_single_calls_and_oracle(oracle, voc, mode, n_kf, ratio, check_ori, nleft):
    rng = np.random.default_rng(n_kf * 10 + mode)
    sizes = [2000] + rng.integers(150, 2001, n_kf - 1).tolist()
    B = make(voc, 3000 + 17 * n_kf + mode, 2000, sizes)
    match, nm = batch(B, mode, nleft, ratio, check_ori)
    total = check_rows(oracle, B, mode, match, nm, nleft, ratio, check_ori)
    assert total > 30 * n_kf


@pytest.mark.parametrize("mode", [0, 1])
def test_edge_key_frames(oracle, voc, mode):
    """A key frame with n = 0, one sharing no vocabulary node with the fixed side and one without a usable map point, between
    normal ones; levelsup 4 puts every feature in the root node (one job per key frame holding the whole sets)."""
    kinds = [S.NORMAL, S.EMPTY, S.DISJOINT, S.INVALID, S.NORMAL, S.EMPTY]
    for levelsup in (2, 4):
        B = make(voc, 3100 + mode + levelsup, 1200, [900, 500, 1000, 800, 1300, 10], kinds, levelsup)
        match, nm = batch(B, mode, ratio=0.9)
        check_rows(oracle, B, mode, match, nm, ratio=0.9)
        for k, kind in enumerate(kinds):
            if kind != S.NORMAL:
                assert nm[k] == 0 and (match[k] < 0).all(), (levelsup, k, kind)
            else:
                assert nm[k] > 20


@pytest.mark.parametrize("mode", [0, 1])
def test_empty_fixed_side(voc, mode):
    B = make(voc, 3200 + mode, 0, [300, 0, 500])
    match, nm = batch(B, mode)
    assert match.shape == (3, 0) and (nm == 0).all()


@pytest.mark.parametrize("mode", [0, 1])
def test_bad_view_leaves_outputs_untouched(voc, mode):
    B = make(voc, 3300 + mode, 500, [400, 400, 400, 400, 400])
    views = (capi.BowViewC * 5)()
    keep = []
    for k, kf in enumerate(B["kfs"]):
        fv = kf["fv"] if k != 3 else orbx.FeatureVector(kf["fv"].node_ids, kf["fv"].offsets, kf["fv"].indices + 400)
        keep.append(fv)
        views[k].n = 400; views[k].desc = capi.ptr(kf["desc"]); views[k].angle = capi.ptr(kf["angle"])
        views[k].valid = capi.ptr(kf["valid"]); views[k].fv = fv.c_struct()
    match = np.full((5, 500), 4242, np.int32)
    nm = np.full(5, 99, np.int32)
    f = B["fv"].c_struct()
    rc = capi.lib().orbx_search_by_bow_batch(0, mode, capi.ptr(B["desc"]), capi.ptr(B["angle"]), capi.ptr(B["valid"]), 500, C.addressof(f), -1, 5,
                                             C.addressof(views), 0.6, 1, capi.ptr(match), capi.ptr(nm))
    assert rc == capi.ORBX_ERR_INVALID_ARG and b"kfs[3].fv" in capi.lib().orbx_last_error()
    assert (match == 4242).all() and (nm == 99).all()


def test_two_threads(oracle, voc):
    """A relocalization batch (tracking scratch) and a loop-detection batch (loop-closing scratch) at once from two threads
    (ctypes releases the GIL): both stay exact."""
    B0 = make(voc, 3400, 1500, [1500, 1200, 1000, 800, 1400, 1100, 900, 1300])
    B1 = make(voc, 3401, 1800, [1800, 1600, 1400, 1200, 1700, 1500])
    want0 = batch(B0, 0, ratio=0.75)
    want1 = batch(B1, 1, ratio=0.9)
    check_rows(oracle, B0, 0, *want0, ratio=0.75)
    check_rows(oracle, B1, 1, *want1, ratio=0.9)
    got = {}

    def run(key, B, mode, ratio):
        got[key] = [batch(B, mode, ratio=ratio) for _ in range(3)]
    ts = [threading.Thread(target=run, args=(0, B0, 0, 0.75)), threading.Thread(target=run, args=(1, B1, 1, 0.9))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for key, want in ((0, want0), (1, want1)):
        assert len(got[key]) == 3
        for m, nm in got[key]:
            assert np.array_equal(m, want[0]) and np.array_equal(nm, want[1])
