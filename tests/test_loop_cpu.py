"""The loop-closing oracle (tests/cpp/loop_oracle.cpp) against an independent numpy restatement (CPU): the Sim3
SearchByProjection as a sequential loop with vpMatched updated in place and 'bestDist <= TH_LOW * ratioHamming' in float32, the
search part of the Sim3 Fuse without a reprojection gate, candidates by brute force ordered by (cell column, cell row, index).
One hand-built scene per rule that is easy to get wrong, random scenes and a frozen golden file."""
import json
import os
import zlib

import numpy as np
import pytest

from tests import fuse_oracle, loop_oracle
from tests.fuse_synth import BOUNDS, bounds_grid
from tests.loop_synth import fuse_scene, sbp_scene
from tests.oracle_lib import KP_DTYPE
from tests.proj_synth import SCALE
from tests.test_fuse_cpu import py_kf_area
from tests.test_projection_cpu import hamming, py_cells

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BG = bounds_grid()
F32 = np.float32


@pytest.fixture(scope="module")
def lo():
    return loop_oracle.load()


def in_image(bg, x, y):
    return x >= bg[0] and x < bg[2] and y >= bg[1] and y < bg[3]


def py_sbp_sim3(K, occupied, P, pdesc, th, ratio=1.0):
    kp, bg = K["kp"], K["bg"]
    cells = py_cells(kp, bg)
    taken = np.asarray(occupied, bool).copy()
    match_f = np.full(len(kp), -1, np.int32)
    lim = float(F32(F32(50) * F32(ratio)))
    nm = 0
    for i in range(len(P["u"])):
        x, y, lvl = F32(P["u"][i]), F32(P["v"][i]), int(P["level"][i])
        if not P["valid"][i] or not in_image(bg, x, y):
            continue
        r = F32(F32(th) * F32(K["scale"][lvl]))
        best, bi = 256, -1
        for j in py_kf_area(kp, cells, bg, x, y, r):
            o = int(kp["octave"][j])
            if taken[j] or o < lvl - 1 or o > lvl:
                continue
            d = hamming(pdesc[i], K["desc"][j])
            if d < best:
                best, bi = d, int(j)
        if best <= lim:
            assert bi >= 0
            taken[bi] = True
            match_f[bi] = i
            nm += 1
    return match_f, nm


def py_fuse_sim3(kfs, P, pdesc, th=4.0):
    offs = P["kf_offsets"]
    match = np.full(int(offs[-1]), -1, np.int32)
    n_fused = np.zeros(len(kfs), np.int32)
    for k, K in enumerate(kfs):
        kp, bg = K["kp"], K["bg"]
        cells = py_cells(kp, bg)
        for q in range(offs[k], offs[k + 1]):
            x, y, lvl = F32(P["u"][q]), F32(P["v"][q]), int(P["level"][q])
            if not P["valid"][q] or not in_image(bg, x, y):
                continue
            r = F32(F32(th) * F32(K["scale"][lvl]))
            best, bi = 1 << 31, -1
            for j in py_kf_area(kp, cells, bg, x, y, r):
                o = int(kp["octave"][j])
                if o < lvl - 1 or o > lvl:
                    continue
                d = hamming(pdesc[P["point"][q]], K["desc"][j])
                if d < best:
                    best, bi = d, int(j)
            if best <= 50:
                match[q] = bi
                n_fused[k] += 1
    return match, n_fused


class Scene:
    """Hand-built key frame: features placed one by one, points given by (u, v, level, bit flips from the base descriptor)."""

    def __init__(self, seed=0):
        rng = np.random.default_rng(seed)
        self.base = rng.integers(0, 256, size=32, dtype=np.uint8)
        self.feat, self.pts, self.occ = [], [], []

    def desc_at(self, d):
        bits = np.unpackbits(self.base.copy())
        bits[:d] ^= 1
        return np.packbits(bits)

    def feature(self, x, y, d, octave=0, occupied=False):
        self.feat.append((F32(x), F32(y), octave, self.desc_at(d)))
        self.occ.append(occupied)
        return len(self.feat) - 1

    def point(self, u, v, level=0, d=0, valid=True):
        self.pts.append((F32(u), F32(v), level, self.desc_at(d), valid))
        return len(self.pts) - 1

    def arrays(self):
        kp = np.zeros(len(self.feat), KP_DTYPE)
        for i, (x, y, o, _) in enumerate(self.feat):
            kp[i]["x"], kp[i]["y"], kp[i]["octave"] = x, y, o
        kp["size"] = 31.0; kp["class_id"] = -1
        K = dict(kp=kp, desc=np.array([f[3] for f in self.feat], np.uint8).reshape(-1, 32), ur=None, bg=BG, scale=SCALE)
        n = len(self.pts)
        P = dict(kf_offsets=np.array([0, n], np.int32), point=np.arange(n, dtype=np.int32),
                 valid=np.array([p[4] for p in self.pts], np.uint8), u=np.array([p[0] for p in self.pts], np.float32),
                 v=np.array([p[1] for p in self.pts], np.float32), level=np.array([p[2] for p in self.pts], np.int32))
        return K, np.array(self.occ, np.uint8), P, np.array([p[3] for p in self.pts], np.uint8).reshape(-1, 32)


def sbp_both(lo, s, th=3, ratio=1.0):
    K, occ, P, pd = s.arrays()
    got = lo.search_by_projection_sim3(K, occ, P["valid"], P["u"], P["v"], P["level"], pd, th, ratio)
    want = py_sbp_sim3(K, occ, P, pd, th, ratio)
    assert np.array_equal(got[0], want[0]) and got[1] == want[1], (got, want)
    return got[0]


def fuse_both(lo, s, th=4.0):
    K, _, P, pd = s.arrays()
    got = lo.fuse_sim3([K], P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], th)
    want = py_fuse_sim3([K], P, pd, th)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (got, want)
    return got[0]


def both(lo, s, th=3, ratio=1.0):
    """SearchByProjection's match_f, and Fuse's match of the same points (Fuse ignores occupancy and ratio)."""
    return sbp_both(lo, s, th, ratio), fuse_both(lo, s, float(th))


def test_slot_occupied_on_entry(lo):
    s = Scene(1)
    s.feature(200, 200, 3, occupied=True); s.feature(201, 200, 9)
    s.point(200, 200)
    m, f = both(lo, s)
    assert list(m) == [-1, 0] and list(f) == [0]            # the Fuse search does not read the slots


def test_two_points_compete_for_one_feature(lo):
    s = Scene(2)
    s.feature(200, 200, 2); s.feature(201, 200, 10)          # point 1 takes its next best
    s.feature(400, 200, 4)                                   # point 3's only candidate is taken: nothing
    s.point(200, 200, d=0); s.point(200.5, 200, d=0); s.point(400, 200, d=0); s.point(400, 200, d=1)
    m, f = both(lo, s)
    assert list(m) == [0, 1, 2] and list(f) == [0, 0, 2, 2]


def test_duplicate_point_entry(lo):
    """vpPoints holds the same point twice: the snapshot does not see the first acceptance, the occupancy does."""
    s = Scene(3)
    s.feature(300, 300, 5); s.feature(302, 300, 7)
    s.point(300, 300, d=0); s.point(300, 300, d=0)
    m, f = both(lo, s)
    assert list(m) == [0, 1] and list(f) == [0, 0]


@pytest.mark.parametrize("ratio,acc", [(1.0, 50), (1.5, 75)])
def test_threshold_edges(lo, ratio, acc):
    s = Scene(4)
    s.feature(100, 100, acc); s.feature(300, 100, acc + 1)
    s.point(100, 100); s.point(300, 100)
    assert list(sbp_both(lo, s, ratio=ratio)) == [0, -1]


def ratio_below_integer():
    """The first two-decimal ratio k / 50 (as a float32) whose float product 50 * ratio falls below the integer k."""
    for k in range(51, 256):
        r = F32(k / 50.0)
        if F32(F32(50) * r) < k:
            return k, r
    raise AssertionError("no such ratio")


def test_ratio_product_just_below_an_integer(lo):
    """F32(1.06) * 50 = 52.999996: distance 52 is accepted and 53 is not, although the ratio was written as 53 / 50."""
    k, r = ratio_below_integer()
    assert F32(F32(50) * r) == np.nextafter(F32(k), F32(0), dtype=np.float32)
    s = Scene(5)
    s.feature(100, 100, k - 1); s.feature(300, 100, k)
    s.point(100, 100); s.point(300, 100)
    assert list(sbp_both(lo, s, ratio=float(r))) == [0, -1]
    r2 = np.nextafter(r, F32(10), dtype=np.float32)           # the next float reaches k
    assert F32(F32(50) * r2) >= k
    assert list(sbp_both(lo, s, ratio=float(r2))) == [0, 1]


def test_only_candidate_at_distance_256(lo):
    s = Scene(6)
    s.feature(100, 100, 256)
    s.point(100, 100)
    assert list(sbp_both(lo, s, ratio=5.1)) == [-1]           # 50 * 5.1 = 255: bestDist 256 never becomes a match
    assert list(fuse_both(lo, s)) == [-1]


def test_level_gate_both_ends_and_level_0(lo):
    s = Scene(7)
    for o in range(4):                                        # one feature per level at one spot
        s.feature(200, 200, {0: 0, 1: 20, 2: 10, 3: 0}[o], octave=o)
    s.feature(400, 300, 30, octave=0); s.feature(400, 300, 5, octave=1)
    s.point(200, 200, level=2)                                # levels 1 and 2: the level-2 feature at 10
    s.point(400, 300, level=0)                                # level 0 only: the level-1 feature at 5 is not a candidate
    m, f = both(lo, s, th=3, ratio=1.0)
    assert list(m) == [-1, -1, 0, -1, 1, -1] and list(f) == [2, 4]


def test_image_bounds(lo):
    """u == mnMaxX and v == mnMaxY are rejected, u == mnMinX accepted (KeyFrame::IsInImage); level 5, window 7.46 px."""
    s = Scene(8)
    s.feature(746.0, 100, 0, octave=5); s.feature(100, 474.5, 0, octave=5); s.feature(3.0, 100, 0, octave=5)
    s.point(752.0, 100, 5); s.point(100, 480.0, 5); s.point(np.nextafter(F32(0.0), F32(-1)), 100, 5); s.point(0.0, 100, 5)
    s.point(np.nextafter(F32(752.0), F32(0)), 100, 5)
    m, f = both(lo, s)
    assert list(f) == [-1, -1, -1, 2, 0] and list(m) == [4, -1, 3]


def test_windows_clipped_at_the_grid_edges(lo):
    s = Scene(9)
    s.feature(0.5, 0.5, 3, octave=7); s.feature(745.5, 474.0, 2, octave=7); s.feature(2, 470, 1, octave=6)
    s.point(1.0, 1.0, level=7); s.point(751.0, 479.0, level=7); s.point(3.0, 472.0, level=7)
    m, f = both(lo, s, th=15)
    assert list(m) == [0, 1, 2] and list(f) == [0, 1, 2]


def test_ties_follow_column_row_index(lo):
    """Cell columns have boundaries at 11.75 * (k + 0.5), rows at 10 * (k + 0.5)."""
    s = Scene(10)
    x0 = 11.75 * 10.5
    s.feature(x0 + 1.5, 105, 7); s.feature(x0 - 1.5, 105, 7)          # column 11 (index 0), column 10 (index 1): 1 wins
    s.point(x0, 105)
    s.feature(300, 106.5, 9); s.feature(300.5, 103.5, 9)               # row 11 (index 2) and row 10 (index 3): 3 wins
    s.point(300, 105)
    s.feature(500, 200.5, 4); s.feature(500.5, 200, 4)                 # same cell: the lower index (4) wins
    s.point(500, 200)
    s.point(x0, 105)                                                   # the same tie again: feature 1 is taken, so 0
    m, f = both(lo, s)
    assert list(m) == [3, 0, -1, 1, 2, -1] and list(f) == [1, 3, 4, 1]


def test_fuse_has_no_reprojection_gate(lo):
    """2.9 px off at level 0: e2 = 8.41 > 5.99 fails orbx_fuse's monocular gate; the Sim3 Fuse accepts it."""
    s = Scene(11)
    s.feature(102.9, 100, 4)
    s.point(100, 100)
    assert list(fuse_both(lo, s)) == [0]
    K, _, P, pd = s.arrays()
    m, _ = fuse_oracle.load().fuse([dict(K, inv_sigma2=np.ones(8, np.float32), bf=F32(40))], P["kf_offsets"], pd, P["point"], P["valid"],
                                   P["u"], P["v"], np.full(1, 0.1, np.float32), P["level"], 4.0)
    assert list(m) == [-1]


@pytest.mark.parametrize("seed,crowd,th,ratio", [(21, 0, 8, 1.5), (22, 4, 5, 1.0), (23, 0, 3, 1.5)])
def test_random_sbp_scenes_match_numpy(lo, seed, crowd, th, ratio):
    K, occ, P, pd = sbp_scene(seed, n_points=500, see=0.4, n_distract=150, crowd=crowd)
    got = lo.search_by_projection_sim3(K, occ, P["valid"], P["u"], P["v"], P["level"], pd, th, ratio)
    want = py_sbp_sim3(K, occ, P, pd, th, ratio)
    assert np.array_equal(got[0], want[0]) and got[1] == want[1] and got[1] > 30


@pytest.mark.parametrize("seed,crowd,th", [(31, 0, 4.0), (32, 4, 4.0), (33, 0, 3.0)])
def test_random_fuse_scenes_match_numpy(lo, seed, crowd, th):
    kfs, P, pd = fuse_scene(seed, n_kf=3, n_points=250, crowd=crowd, n_distract=150)
    got = lo.fuse_sim3(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], th)
    want = py_fuse_sim3(kfs, P, pd, th)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]) and got[1].sum() > 50


def test_no_device_is_an_error_not_a_fallback():
    import wut_cuda_orb_slam3_b200 as orbx
    if orbx.lib().orbx_device_count() > 0:
        pytest.skip("a GPU is visible")
    K, occ, P, pd = sbp_scene(41, n_points=100)
    fv = orbx.FrameView(K["kp"], K["desc"], K["scale"], BOUNDS, occupied=occ)
    with pytest.raises(orbx.OrbxError) as e:
        orbx.search_by_projection_sim3(fv, P["valid"], P["u"], P["v"], P["level"], pd, 8, 1.5)
    assert e.value.code == orbx.capi.ORBX_ERR_NO_DEVICE
    with pytest.raises(orbx.OrbxError) as e:                  # argument errors are reported before the device is looked for
        orbx.search_by_projection_sim3(fv, P["valid"], P["u"], P["v"], P["level"], pd, 8, 5.12)
    assert e.value.code == orbx.capi.ORBX_ERR_INVALID_ARG
    kfs, P, pd = fuse_scene(42, n_kf=2, n_points=50)
    V = [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS) for k in kfs]
    with pytest.raises(orbx.OrbxError) as e:
        orbx.fuse_sim3(V, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"])
    assert e.value.code == orbx.capi.ORBX_ERR_NO_DEVICE


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def golden_inputs(c):
    if c["kind"] == "sbp":
        K, occ, P, pd = sbp_scene(c["seed"], n_points=c["n_points"], crowd=c["crowd"])
        return [K], occ, P, pd
    kfs, P, pd = fuse_scene(c["seed"], n_kf=c["n_kf"], n_points=c["n_points"], crowd=c["crowd"])
    return kfs, None, P, pd


def test_oracle_reproduces_loop_golden(lo):
    """tests/golden/loop_golden.json (made by tests/golden/make_loop_golden.py from this oracle) still holds."""
    with open(os.path.join(ROOT, "tests", "golden", "loop_golden.json")) as f:
        gold = json.load(f)["cases"]
    for c in gold:
        kfs, occ, P, pd = golden_inputs(c)
        assert crc(np.concatenate([k["kp"] for k in kfs])) == c["kp_crc"] and crc(pd) == c["desc_crc"] and crc(P["u"]) == c["u_crc"]
        if c["kind"] == "sbp":
            m, n = lo.search_by_projection_sim3(kfs[0], occ, P["valid"], P["u"], P["v"], P["level"], pd, c["th"], c["ratio"])
            assert crc(m) == c["match_crc"] and n == c["n"], c["seed"]
        else:
            m, nf = lo.fuse_sim3(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["level"], c["th"])
            assert crc(m) == c["match_crc"] and nf.tolist() == c["n"], c["seed"]
