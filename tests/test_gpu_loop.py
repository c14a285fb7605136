"""GPU parity of loop closing's two searches against the oracle's sequential loops (tests/cpp/loop_oracle.cpp), bit-exact:
the Sim3 SearchByProjection (src/ORBmatcher1.cc:429-648) through orbx_search_by_projection_sim3 in match_f / nmatches, and the
search part of the Sim3 Fuse (src/ORBmatcher2.cc:612-729) through orbx_fuse_sim3 in match / n_fused."""
import ctypes as C
import json
import os
import threading
import zlib

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import fuse_oracle, loop_oracle, oracle_lib
from tests.fuse_synth import BOUNDS, scene
from tests.loop_synth import fuse_scene, sbp_scene
from tests.proj_synth import SCALE, make_frame, make_points

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lo():
    return loop_oracle.load()


def frame(K, occ):
    return orbx.FrameView(K["kp"], K["desc"], K["scale"], BOUNDS, occupied=occ)


def views(kfs):
    return [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS) for k in kfs]


def check_sbp(lo, K, occ, P, pd, th, ratio):
    got = orbx.search_by_projection_sim3(frame(K, occ), P["valid"], P["u"], P["v"], P["level"], pd, th, ratio)
    want = lo.search_by_projection_sim3(K, occ, P["valid"], P["u"], P["v"], P["level"], pd, th, ratio)
    assert np.array_equal(got[0], want[0]), np.flatnonzero(got[0] != want[0])[:10]
    assert got[1] == want[1]
    return got


def check_fuse(lo, kfs, P, pd, th=4.0):
    got = orbx.fuse_sim3(views(kfs), P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], th)
    want = lo.fuse_sim3(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], th)
    assert np.array_equal(got[0], want[0]), np.flatnonzero(got[0] != want[0])[:10]
    assert np.array_equal(got[1], want[1])
    return got


def test_detect_common_regions_shape(lo):
    """1 key frame (~2000 features), 8000 points, 30 % of the slots matched on entry: (th 8, ratio 1.5), then (5, 1.0) chained
    on its vpMatched (the points it matched folded out of valid: spAlreadyFound), and (5, 1.0) on the entry state."""
    K, occ, P, pd = sbp_scene(1, n_points=8000, see=0.22, n_distract=400)
    assert 1500 <= len(K["kp"]) <= 2600
    m1, n1 = check_sbp(lo, K, occ, P, pd, 8, 1.5)
    assert n1 > 500
    occ2 = (occ.astype(bool) | (m1 >= 0)).astype(np.uint8)
    found = np.zeros(len(P["u"]), bool)
    found[m1[m1 >= 0]] = True
    P2 = dict(P, valid=(P["valid"].astype(bool) & ~found).astype(np.uint8))
    m2, n2 = check_sbp(lo, K, occ2, P2, pd, 5, 1.0)
    assert not (m2[m1 >= 0] >= 0).any()
    m3, n3 = check_sbp(lo, K, occ, P, pd, 5, 1.0)
    assert 0 < n3 < n1


def test_find_matches_by_projection_shape(lo):
    K, occ, P, pd = sbp_scene(2, n_points=8000, see=0.3, n_distract=600)
    m, n = check_sbp(lo, K, occ, P, pd, 3, 1.5)
    assert n > 500


@pytest.mark.parametrize("seed,crowd", [(3, 1), (4, 3), (5, 8)])
def test_crowded_sbp_scenes(lo, seed, crowd):
    """Many points on the same few features: long chains of points whose windows overlap, resolved over many rounds."""
    K, occ, P, pd = sbp_scene(seed, n_points=3000, see=0.5, n_distract=50, crowd=crowd, max_flip=20, occ_frac=0.1)
    rounds = []
    for th, ratio in ((3, 1.0), (8, 1.5), (15, 2.0)):
        check_sbp(lo, K, occ, P, pd, th, ratio)
        rounds.append(orbx.projection_rounds())
    assert max(rounds) >= 2, rounds


def test_worst_case_chain(lo):
    """Identical descriptors in one cluster: every point claims every feature of its window, so the speculation decides about
    one point per round; the result must still equal the sequential loop."""
    rng = np.random.default_rng(20)
    K, occ, P, pd = sbp_scene(20, n_points=10)
    n, m = 64, 200
    kp = K["kp"][:n].copy()
    kp["x"] = 300 + rng.normal(0, 3.0, n); kp["y"] = 200 + rng.normal(0, 3.0, n); kp["octave"] = 2
    K = dict(K, kp=kp, desc=np.repeat(pd[:1], n, 0))
    P = dict(valid=np.ones(m, np.uint8), u=(300 + rng.normal(0, 2.0, m)).astype(np.float32), v=(200 + rng.normal(0, 2.0, m)).astype(np.float32),
             level=np.full(m, 2, np.int32))
    got, nm = check_sbp(lo, K, np.zeros(n, np.uint8), P, np.repeat(pd[:1], m, 0), 15, 1.0)
    assert nm > 40 and orbx.projection_rounds() >= 10


@pytest.mark.parametrize("seed,crowd", [(6, 1), (7, 4)])
def test_crowded_fuse_scenes(lo, seed, crowd):
    kfs, P, pd = fuse_scene(seed, n_kf=4, n_points=2000, crowd=crowd, n_distract=50, max_flip=20)
    for th in (4.0, 8.0):
        check_fuse(lo, kfs, P, pd, th)


def test_random_scenes(lo):
    """60 random scenes of each search, half of them with few distinct descriptors (equal distances in most windows)."""
    for seed in range(500, 560):
        rng = np.random.default_rng(seed)
        K, occ, P, pd = sbp_scene(seed, n_points=int(rng.integers(1, 1500)), see=float(rng.choice([0.2, 0.6])),
                                  n_distract=int(rng.integers(0, 300)), occ_frac=float(rng.choice([0.0, 0.3, 0.8])),
                                  crowd=int(rng.choice([0, 0, 2, 6])), pose_noise=float(rng.choice([0.3, 1.0, 3.0])),
                                  max_flip=int(rng.choice([10, 40, 80])))
        kfs, Pf, pdf = fuse_scene(seed, n_kf=int(rng.integers(1, 7)), n_points=int(rng.integers(1, 700)), crowd=int(rng.choice([0, 0, 2, 6])),
                                  n_distract=int(rng.integers(0, 400)), max_flip=int(rng.choice([10, 40, 80])))
        if rng.random() < 0.5:
            pd = pd[rng.integers(0, 4, len(pd))]
            K["desc"] = pd[rng.integers(0, len(pd), len(K["desc"]))]
            pdf = pdf[rng.integers(0, 4, len(pdf))]
            for k in kfs:
                k["desc"] = pdf[rng.integers(0, len(pdf), len(k["desc"]))]
        check_sbp(lo, K, occ, P, pd, int(rng.choice([3, 5, 8, 15])), float(rng.choice([0.5, 1.0, 1.5, 2.5])))
        check_fuse(lo, kfs, Pf, pdf, float(rng.choice([1.0, 4.0, 8.0])))


def test_search_and_fuse_shapes(lo):
    """25 key frames x 4000 loop points in one call, and 1 key frame x 15 000 points."""
    kfs, P, pd = fuse_scene(10, n_kf=25, n_points=4000, n_distract=800)
    m, nf = check_fuse(lo, kfs, P, pd)
    assert len(m) == 100000 and nf.min() > 300
    kfs, P, pd = fuse_scene(11, n_kf=1, n_points=15000, n_distract=1500)
    m, nf = check_fuse(lo, kfs, P, pd)
    assert nf[0] > 2000


def test_empty_cases(lo):
    K, occ, P, pd = sbp_scene(12, n_points=300)
    fv = frame(K, occ)
    m, n = orbx.search_by_projection_sim3(fv, [], [], [], [], np.zeros((0, 32), np.uint8), 8, 1.5)   # no points
    assert n == 0 and (m == -1).all() and orbx.projection_rounds() == 0
    K0 = dict(K, kp=K["kp"][:0], desc=K["desc"][:0])
    m, n = check_sbp(lo, K0, occ[:0], P, pd, 8, 1.5)                                                  # N = 0
    assert n == 0 and len(m) == 0
    m, n = check_sbp(lo, K, occ, dict(P, valid=np.zeros_like(P["valid"])), pd, 8, 1.5)               # nothing valid
    assert n == 0
    m, n = check_sbp(lo, K, np.ones_like(occ), P, pd, 8, 1.5)                                         # every slot matched
    assert n == 0
    kfs, Pf, pdf = fuse_scene(13, n_kf=3, n_points=300)
    kfs[1] = dict(kfs[1], kp=kfs[1]["kp"][:0], desc=kfs[1]["desc"][:0])
    m, nf = check_fuse(lo, kfs, Pf, pdf)                                                              # a key frame with N = 0
    assert nf[1] == 0 and (m[300:600] == -1).all() and nf[0] > 0
    m, nf = orbx.fuse_sim3([], [0], pdf, [], [], [], [], [])
    assert len(m) == 0 and len(nf) == 0
    m, nf = orbx.fuse_sim3(views(kfs), [0, 0, 0, 0], pdf, [], [], [], [], [])
    assert len(m) == 0 and nf.tolist() == [0, 0, 0]


def test_sbp_bad_arguments():
    K, occ, P, pd = sbp_scene(14, n_points=100)
    fv = frame(K, occ)
    a = [np.ascontiguousarray(x) for x in (P["valid"], P["u"], P["v"], P["level"], pd)]
    mf = np.zeros(len(K["kp"]), np.int32); nm = C.c_int(0)
    args = [0, C.addressof(fv.c), 100, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data, a[3].ctypes.data, a[4].ctypes.data, 8.0, 1.5,
            mf.ctypes.data, C.addressof(nm)]
    f = orbx.lib().orbx_search_by_projection_sim3
    assert f(*args) == 0
    for k in (1, 3, 4, 5, 6, 7, 10, 11):
        b = list(args); b[k] = None
        assert f(*b) == orbx.capi.ORBX_ERR_INVALID_ARG, k
    b = list(args); b[2] = -1
    assert f(*b) == orbx.capi.ORBX_ERR_INVALID_ARG
    for ratio in (5.12, 6.0, float("nan"), float("inf")):          # TH_LOW * ratio >= 256: the reference writes vpMatched[-1]
        b = list(args); b[9] = ratio
        assert f(*b) == orbx.capi.ORBX_ERR_INVALID_ARG, ratio
    b = list(args); b[9] = 5.1                                     # 255: the largest threshold that is defined
    assert f(*b) == 0
    first = int(np.flatnonzero(P["valid"])[0])
    for lv in (8, -1):
        bad = P["level"].copy(); bad[first] = lv
        with pytest.raises(orbx.OrbxError) as e:
            orbx.search_by_projection_sim3(fv, P["valid"], P["u"], P["v"], bad, pd, 8, 1.5)
        assert e.value.code == orbx.capi.ORBX_ERR_INVALID_ARG
    lv = P["level"].copy(); lv[np.flatnonzero(P["valid"] == 0)[0]] = 99     # out-of-range level on an invalid point: ignored
    orbx.search_by_projection_sim3(fv, P["valid"], P["u"], P["v"], lv, pd, 8, 1.5)
    fv.c.scale_factors = None                                      # the window needs mvScaleFactors
    assert f(*args) == orbx.capi.ORBX_ERR_INVALID_ARG


def test_fuse_bad_arguments():
    kfs, P, pd = fuse_scene(15, n_kf=2, n_points=100)
    V = views(kfs)
    ok = dict(kfs=V, kf_offsets=P["kf_offsets"], point_desc=pd, point=P["point"], valid=P["valid"], u=P["u"], v=P["v"], level=P["level"])
    orbx.fuse_sim3(**ok)
    first = int(np.flatnonzero(P["valid"])[0])
    bad = [dict(kf_offsets=np.array([0, 120, 100], np.int32)),
           dict(kf_offsets=np.array([5, 100, 200], np.int32)),
           dict(point=np.where(np.arange(200) == 17, 100, P["point"])),
           dict(point=np.where(np.arange(200) == 3, -1, P["point"])),
           dict(level=np.where(np.arange(200) == first, 8, P["level"])),
           dict(level=np.where(np.arange(200) == first, -1, P["level"]))]
    for b in bad:
        with pytest.raises(orbx.OrbxError) as e:
            orbx.fuse_sim3(**dict(ok, **b))
        assert e.value.code == orbx.capi.ORBX_ERR_INVALID_ARG
    arr = (orbx.capi.KeyFrameViewC * 2)(*[k.kc for k in V])
    a = [np.ascontiguousarray(x) for x in (P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"])]
    match = np.zeros(200, np.int32); nf = np.zeros(2, np.int32)
    args = [0, 2, C.addressof(arr), a[0].ctypes.data, len(pd), a[1].ctypes.data, a[2].ctypes.data, a[3].ctypes.data, a[4].ctypes.data,
            a[5].ctypes.data, a[6].ctypes.data, 4.0, match.ctypes.data, nf.ctypes.data]
    assert orbx.lib().orbx_fuse_sim3(*args) == 0                   # inv_level_sigma2 NULL and bf 0: not read
    for k in (2, 3, 5, 6, 7, 8, 9, 10, 12, 13):
        b = list(args); b[k] = None
        assert orbx.lib().orbx_fuse_sim3(*b) == orbx.capi.ORBX_ERR_INVALID_ARG, k
    b = list(args); b[1] = -1
    assert orbx.lib().orbx_fuse_sim3(*b) == orbx.capi.ORBX_ERR_INVALID_ARG
    arr[1].frame.scale_factors = None
    assert orbx.lib().orbx_fuse_sim3(*args) == orbx.capi.ORBX_ERR_INVALID_ARG


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def test_cuda_reproduces_loop_golden():
    """tests/golden/loop_golden.json, without touching oracle code."""
    with open(os.path.join(ROOT, "tests", "golden", "loop_golden.json")) as f:
        gold = json.load(f)["cases"]
    for c in gold:
        if c["kind"] == "sbp":
            K, occ, P, pd = sbp_scene(c["seed"], n_points=c["n_points"], crowd=c["crowd"])
            kfs = [K]
            m, n = orbx.search_by_projection_sim3(frame(K, occ), P["valid"], P["u"], P["v"], P["level"], pd, c["th"], c["ratio"])
        else:
            kfs, P, pd = fuse_scene(c["seed"], n_kf=c["n_kf"], n_points=c["n_points"], crowd=c["crowd"])
            m, nf = orbx.fuse_sim3(views(kfs), P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], c["th"])
            n = nf.tolist()
        assert crc(np.concatenate([k["kp"] for k in kfs])) == c["kp_crc"] and crc(pd) == c["desc_crc"] and crc(P["u"]) == c["u_crc"]
        assert crc(m) == c["match_crc"] and n == c["n"], c["seed"]


def test_three_threads_do_not_share_scratch(lo):
    """Tracking (search_by_projection_map), local mapping (fuse) and loop closing (both Sim3 calls) at once, 50 calls each,
    all bit-exact."""
    o = oracle_lib.load()
    rng = np.random.default_rng(16)
    kp, desc, ur, occ, bounds = make_frame(rng, 2000)
    Pm = make_points(rng, kp, desc, ur, 1500)
    fv = orbx.FrameView(kp, desc, SCALE, bounds, u_right=ur, occupied=occ)
    margs = (Pm["in_view"], Pm["bad"], Pm["x"], Pm["y"], Pm["xr"], Pm["view_cos"], Pm["depth"], Pm["level"], Pm["n_obs"], Pm["desc"])
    want_m = o.search_by_projection_map(kp, desc, ur, occ, fv.bounds_grid(), SCALE, *margs, 1.0, False, 0.0, 0.8)
    X, pd, kfs, P = scene(17, n_kf=10, n_points=1200)
    want_f = fuse_oracle.load().fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0)
    V = [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS, k["inv_sigma2"], k["bf"], u_right=k["ur"]) for k in kfs]
    K, socc, Ps, pds = sbp_scene(18, n_points=4000)
    want_s = lo.search_by_projection_sim3(K, socc, Ps["valid"], Ps["u"], Ps["v"], Ps["level"], pds, 8, 1.5)
    lkfs, Pl, pdl = fuse_scene(19, n_kf=8, n_points=1500)
    want_l = lo.fuse_sim3(lkfs, Pl["kf_offsets"], pdl, Pl["point"], Pl["valid"], Pl["u"], Pl["v"], Pl["level"], 4.0)
    sfv, LV = frame(K, socc), views(lkfs)
    errors = []

    def run(fn):
        def body():
            try:
                for _ in range(50):
                    fn()
            except BaseException as e:       # noqa: BLE001
                errors.append(e)
        return body

    def tracking():
        got = orbx.search_by_projection_map(fv, *margs, th=1.0, nnratio=0.8)
        assert got[1] == want_m[1] and np.array_equal(got[0], want_m[0])

    def mapping():
        got = orbx.fuse(V, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0)
        assert np.array_equal(got[0], want_f[0]) and np.array_equal(got[1], want_f[1])

    def loop():
        got = orbx.search_by_projection_sim3(sfv, Ps["valid"], Ps["u"], Ps["v"], Ps["level"], pds, 8, 1.5)
        assert got[1] == want_s[1] and np.array_equal(got[0], want_s[0])
        got = orbx.fuse_sim3(LV, Pl["kf_offsets"], pdl, Pl["point"], Pl["valid"], Pl["u"], Pl["v"], Pl["level"], 4.0)
        assert np.array_equal(got[0], want_l[0]) and np.array_equal(got[1], want_l[1])

    ts = [threading.Thread(target=run(f)) for f in (tracking, mapping, loop)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
