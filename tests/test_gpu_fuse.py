"""GPU parity of the search part of ORBmatcher::Fuse (src/ORBmatcher2.cc:420-610): orbx_fuse through the Python binding against
the oracle's sequential loop (tests/cpp/fuse_oracle.cpp), bit-exact in match and n_fused."""
import ctypes as C
import json
import os
import threading
import zlib

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import fuse_oracle, oracle_lib
from tests.fuse_synth import BOUNDS, scene
from tests.proj_synth import SCALE, make_frame, make_points

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def fo():
    return fuse_oracle.load()


def views(kfs):
    return [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS, k["inv_sigma2"], k["bf"], u_right=k["ur"]) for k in kfs]


def check(fo, kfs, pd, P, th=3.0):
    got = orbx.fuse(views(kfs), P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], th)
    want = fo.fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], th)
    assert np.array_equal(got[0], want[0]), np.flatnonzero(got[0] != want[0])[:10]
    assert np.array_equal(got[1], want[1])
    return got


def test_forward_shape_of_search_in_neighbors(fo):
    """20 key frames x 1500 map points of the current key frame, in one call."""
    X, pd, kfs, P = scene(1, n_kf=20, n_points=1500)
    m, nf = check(fo, kfs, pd, P)
    assert len(m) == 30000 and nf.min() > 200


def test_reverse_shape(fo):
    """1 key frame x 15 000 points (the neighbours' points fused into the current key frame)."""
    X, pd, kfs, P = scene(2, n_kf=1, n_points=15000, n_distract=1500)
    m, nf = check(fo, kfs, pd, P)
    assert nf[0] > 2000


@pytest.mark.parametrize("seed,crowd", [(3, 1), (4, 3), (5, 8)])
def test_crowded_scenes(fo, seed, crowd):
    """Many points project onto the same few features: windows of hundreds of candidates, ties everywhere."""
    X, pd, kfs, P = scene(seed, n_kf=4, n_points=2000, crowd=crowd, n_distract=50, max_flip=20)
    for th in (3.0, 8.0):
        check(fo, kfs, pd, P, th)


def test_random_scenes(fo):
    for seed in range(400, 460):
        rng = np.random.default_rng(seed)
        X, pd, kfs, P = scene(seed, n_kf=int(rng.integers(1, 7)), n_points=int(rng.integers(1, 700)), crowd=int(rng.choice([0, 0, 2, 6])),
                              n_distract=int(rng.integers(0, 400)), pose_noise=float(rng.choice([0.3, 1.0, 3.0])),
                              max_flip=int(rng.choice([10, 40, 80])))
        if rng.random() < 0.5:                                   # few distinct descriptors: equal distances in most windows
            pd = pd[rng.integers(0, 4, len(pd))]
            for k in kfs:
                k["desc"] = pd[rng.integers(0, len(pd), len(k["desc"]))]
        check(fo, kfs, pd, P, float(rng.choice([1.0, 3.0, 5.0])))


def test_empty_cases(fo):
    X, pd, kfs, P = scene(6, n_kf=3, n_points=300)
    kfs[1] = dict(kfs[1], kp=kfs[1]["kp"][:0], desc=kfs[1]["desc"][:0], ur=None if kfs[1]["ur"] is None else kfs[1]["ur"][:0])
    m, nf = check(fo, kfs, pd, P)                                # a key frame with N = 0
    assert nf[1] == 0 and (m[300:600] == -1).all() and nf[0] > 0
    m, nf = orbx.fuse([], [0], pd, [], [], [], [], [], [])       # n_kf = 0
    assert len(m) == 0 and len(nf) == 0
    m, nf = orbx.fuse(views(kfs), [0, 0, 0, 0], pd, [], [], [], [], [], [])   # nq = 0
    assert len(m) == 0 and nf.tolist() == [0, 0, 0]
    P0 = dict(P, valid=np.zeros_like(P["valid"]))                # nothing valid
    m, nf = check(fo, kfs, pd, P0)
    assert (m == -1).all()


def test_bad_arguments():
    X, pd, kfs, P = scene(7, n_kf=2, n_points=100)
    V = views(kfs)
    ok = dict(kfs=V, kf_offsets=P["kf_offsets"], point_desc=pd, point=P["point"], valid=P["valid"], u=P["u"], v=P["v"], invz=P["invz"],
              level=P["level"])
    orbx.fuse(**ok)
    bad = [dict(kf_offsets=np.array([0, 120, 100], np.int32)),                       # non-monotone
           dict(kf_offsets=np.array([5, 100, 200], np.int32)),                       # not starting at 0
           dict(point=np.where(np.arange(200) == 17, 100, P["point"])),              # point == n_desc
           dict(point=np.where(np.arange(200) == 3, -1, P["point"])),
           dict(level=np.where(np.arange(200) == np.flatnonzero(P["valid"])[0], 8, P["level"])),   # level == n_levels on a valid pair
           dict(level=np.where(np.arange(200) == np.flatnonzero(P["valid"])[0], -1, P["level"]))]
    for b in bad:
        with pytest.raises(orbx.OrbxError) as e:
            orbx.fuse(**dict(ok, **b))
        assert e.value.code == orbx.capi.ORBX_ERR_INVALID_ARG
    lv = P["level"].copy(); lv[np.flatnonzero(P["valid"] == 0)[0]] = 99               # out-of-range level on an invalid pair: ignored
    orbx.fuse(**dict(ok, level=lv))
    # null arrays and a missing inv_level_sigma2, through the C ABI
    arr = (orbx.capi.KeyFrameViewC * 2)(*[k.kc for k in V])
    a = [np.ascontiguousarray(x) for x in (P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"])]
    match = np.zeros(200, np.int32); nf = np.zeros(2, np.int32)
    args = [0, 2, C.addressof(arr), a[0].ctypes.data, len(pd), a[1].ctypes.data, a[2].ctypes.data, a[3].ctypes.data, a[4].ctypes.data,
            a[5].ctypes.data, a[6].ctypes.data, a[7].ctypes.data, 3.0, match.ctypes.data, nf.ctypes.data]
    assert orbx.lib().orbx_fuse(*args) == 0
    for k in (2, 3, 5, 6, 7, 8, 9, 10, 11, 13, 14):
        b = list(args); b[k] = None
        assert orbx.lib().orbx_fuse(*b) == orbx.capi.ORBX_ERR_INVALID_ARG, k
    arr[1].inv_level_sigma2 = None
    assert orbx.lib().orbx_fuse(*args) == orbx.capi.ORBX_ERR_INVALID_ARG


def test_two_threads_do_not_share_scratch(fo):
    """search_by_projection_map (tracking thread) and fuse (local-mapping thread) at once, 50 calls each, both bit-exact."""
    o = oracle_lib.load()
    rng = np.random.default_rng(8)
    kp, desc, ur, occ, bounds = make_frame(rng, 2000)
    Pm = make_points(rng, kp, desc, ur, 1500)
    fv = orbx.FrameView(kp, desc, SCALE, bounds, u_right=ur, occupied=occ)
    bg = fv.bounds_grid()
    margs = (Pm["in_view"], Pm["bad"], Pm["x"], Pm["y"], Pm["xr"], Pm["view_cos"], Pm["depth"], Pm["level"], Pm["n_obs"], Pm["desc"])
    want_m = o.search_by_projection_map(kp, desc, ur, occ, bg, SCALE, *margs, 1.0, False, 0.0, 0.8)
    X, pd, kfs, P = scene(9, n_kf=10, n_points=1200)
    want_f = fo.fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0)
    V = views(kfs)
    errors = []

    def tracking():
        try:
            for _ in range(50):
                got = orbx.search_by_projection_map(fv, *margs, th=1.0, nnratio=0.8)
                assert got[1] == want_m[1] and np.array_equal(got[0], want_m[0])
        except BaseException as e:       # noqa: BLE001
            errors.append(e)

    def mapping():
        try:
            for _ in range(50):
                got = orbx.fuse(V, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0)
                assert np.array_equal(got[0], want_f[0]) and np.array_equal(got[1], want_f[1])
        except BaseException as e:       # noqa: BLE001
            errors.append(e)

    ts = [threading.Thread(target=tracking), threading.Thread(target=mapping)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def test_cuda_reproduces_fuse_golden():
    """tests/golden/fuse_golden.json, without touching oracle code."""
    with open(os.path.join(ROOT, "tests", "golden", "fuse_golden.json")) as f:
        gold = json.load(f)["cases"]
    for c in gold:
        X, pd, kfs, P = scene(c["seed"], n_kf=c["n_kf"], n_points=c["n_points"], crowd=c["crowd"], forward=True)
        assert crc(np.concatenate([k["kp"] for k in kfs])) == c["kp_crc"] and crc(pd) == c["desc_crc"] and crc(P["u"]) == c["u_crc"]
        m, nf = orbx.fuse(views(kfs), P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], c["th"])
        assert crc(m) == c["match_crc"] and nf.tolist() == c["n_fused"], c["seed"]
