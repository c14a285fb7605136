"""The Fuse oracle (tests/cpp/fuse_oracle.cpp) against an independent numpy restatement (CPU): float32 arithmetic, the product
'e2 * mvInvLevelSigma2' rounded to float and compared with the double constant explicitly, candidates by brute force ordered
by (cell column, cell row, index).  One hand-built scene per rule that is easy to get wrong, random scenes and a frozen
golden file."""
import json
import os
import zlib

import numpy as np
import pytest

from tests import fuse_oracle, oracle_lib
from tests.fuse_synth import BOUNDS, INV_SIGMA2, bounds_grid, scene
from tests.oracle_lib import KP_DTYPE
from tests.proj_synth import SCALE
from tests.test_projection_cpu import hamming, py_cells

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BG = bounds_grid()
F32 = np.float32


@pytest.fixture(scope="module")
def fo():
    return fuse_oracle.load()


def py_kf_area(kp, cells, bg, x, y, r):
    """KeyFrame::GetFeaturesInArea by brute force: cell range in float32, box test, ordered by (cell id, index)."""
    x0 = max(0, int(np.floor((x - bg[0] - r) * bg[4]))); x1 = min(63, int(np.ceil((x - bg[0] + r) * bg[4])))
    y0 = max(0, int(np.floor((y - bg[1] - r) * bg[5]))); y1 = min(47, int(np.ceil((y - bg[1] + r) * bg[5])))
    if x0 >= 64 or x1 < 0 or y0 >= 48 or y1 < 0:
        return np.zeros(0, np.int64)
    cx, cy = cells // 48, cells % 48
    m = (cells >= 0) & (cx >= x0) & (cx <= x1) & (cy >= y0) & (cy <= y1)
    m &= (np.abs(kp["x"] - x) < r) & (np.abs(kp["y"] - y) < r)
    idx = np.flatnonzero(m)
    return idx[np.lexsort((idx, cells[idx]))]


def py_fuse(kfs, P, pdesc, th=3.0):
    offs = P["kf_offsets"]
    match = np.full(int(offs[-1]), -1, np.int32)
    n_fused = np.zeros(len(kfs), np.int32)
    th = F32(th)
    for k, K in enumerate(kfs):
        kp, bg = K["kp"], K["bg"]
        cells = py_cells(kp, bg)
        kur = np.full(len(kp), -1, np.float32) if K["ur"] is None else K["ur"]
        for q in range(offs[k], offs[k + 1]):
            if not P["valid"][q]:
                continue
            x, y, lvl = F32(P["u"][q]), F32(P["v"][q]), int(P["level"][q])
            if not (x >= bg[0] and x < bg[2] and y >= bg[1] and y < bg[3]):
                continue
            ur = F32(x - F32(F32(K["bf"]) * F32(P["invz"][q])))
            r = F32(th * F32(K["scale"][lvl]))
            best, bi = 256, -1
            for i in py_kf_area(kp, cells, bg, x, y, r):
                o = int(kp["octave"][i])
                if o < lvl - 1 or o > lvl:
                    continue
                ex, ey = F32(x - kp["x"][i]), F32(y - kp["y"][i])
                inv = F32(K["inv_sigma2"][o])
                if kur[i] >= 0:
                    er = F32(ur - kur[i])
                    e2 = F32(F32(F32(ex * ex) + F32(ey * ey)) + F32(er * er))
                    if float(F32(e2 * inv)) > 7.8:
                        continue
                else:
                    e2 = F32(F32(ex * ex) + F32(ey * ey))
                    if float(F32(e2 * inv)) > 5.99:
                        continue
                d = hamming(pdesc[P["point"][q]], K["desc"][i])
                if d < best:
                    best, bi = d, int(i)
            if best <= 50:
                match[q] = bi
                n_fused[k] += 1
    return match, n_fused


class KFScene:
    """Hand-built key frame: features placed one by one, pairs given by (u, v, level); every point has the base descriptor."""

    def __init__(self, seed=0, stereo=False, bf=40.0):
        self.rng = np.random.default_rng(seed)
        self.base = self.rng.integers(0, 256, size=32, dtype=np.uint8)
        self.feat, self.pairs, self.stereo, self.bf = [], [], stereo, F32(bf)

    def desc_at(self, d):
        bits = np.unpackbits(self.base.copy())
        bits[:d] ^= 1
        return np.packbits(bits)

    def feature(self, x, y, d, octave=0, ur=-1.0):
        self.feat.append((F32(x), F32(y), octave, self.desc_at(d), F32(ur)))
        return len(self.feat) - 1

    def pair(self, u, v, level=0, invz=0.1):
        self.pairs.append((F32(u), F32(v), level, F32(invz)))
        return len(self.pairs) - 1

    def arrays(self):
        kp = np.zeros(len(self.feat), KP_DTYPE)
        for i, (x, y, o, _, _) in enumerate(self.feat):
            kp[i]["x"], kp[i]["y"], kp[i]["octave"] = x, y, o
        kp["size"] = 31.0; kp["class_id"] = -1
        desc = np.array([f[3] for f in self.feat], np.uint8).reshape(-1, 32)
        ur = np.array([f[4] for f in self.feat], np.float32) if self.stereo else None
        K = dict(kp=kp, desc=desc, ur=ur, bg=BG, scale=SCALE, inv_sigma2=INV_SIGMA2, bf=self.bf)
        n = len(self.pairs)
        P = dict(kf_offsets=np.array([0, n], np.int32), point=np.zeros(n, np.int32), valid=np.ones(n, np.uint8),
                 u=np.array([p[0] for p in self.pairs], np.float32), v=np.array([p[1] for p in self.pairs], np.float32),
                 invz=np.array([p[3] for p in self.pairs], np.float32), level=np.array([p[2] for p in self.pairs], np.int32))
        return [K], P, self.base.reshape(1, 32)


def run_both(fo, s, th=3.0):
    kfs, P, pd = s.arrays()
    got = fo.fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], th)
    want = py_fuse(kfs, P, pd, th)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (got, want)
    return got[0]


def test_kf_features_in_area_equals_frame_version(fo):
    """KeyFrame::GetFeaturesInArea = Frame::GetFeaturesInArea without levels: same cells, box test and visiting order."""
    o = oracle_lib.load()
    rng = np.random.default_rng(3)
    K = scene(3, n_kf=1, n_points=800)[2][0]
    for _ in range(300):
        x, y = F32(rng.uniform(-30, 780)), F32(rng.uniform(-30, 510))
        r = F32(rng.choice([2.0, 3.0, 6.2208, 12.0, 40.0]))
        got = fo.kf_get_features_in_area(K["kp"], BG, x, y, r)
        assert np.array_equal(got, o.get_features_in_area(K["kp"], BG, x, y, r, -1, -1))
        assert np.array_equal(got, py_kf_area(K["kp"], py_cells(K["kp"], BG), BG, x, y, r))


def test_level_gate_both_ends_and_level_0(fo):
    s = KFScene(1)
    for o in range(4):                                       # one feature per level at the same spot: level 3 and 0 are exact
        s.feature(200, 200, {0: 0, 1: 20, 2: 10, 3: 0}[o], octave=o)
    s.feature(400, 300, 30, octave=0); s.feature(400, 300, 5, octave=1)
    p2 = s.pair(200, 200, level=2)                           # levels 1 and 2 only: the level-2 feature at 10
    p0 = s.pair(400, 300, level=0)                           # level 0 (and -1) only: the level-1 feature at 5 is not a candidate
    p1 = s.pair(200, 200, level=1)                           # levels 0 and 1: the level-0 feature at 0
    m = run_both(fo, s)
    assert m[p2] == 2 and m[p0] == 4 and m[p1] == 0


def test_uright_zero_takes_the_stereo_gate(fo):
    s = KFScene(2, stereo=True, bf=40.0)
    s.feature(100, 100, 0, ur=0.0)                          # ur of the pair = 100 - 40 * 0.1 = 96: er = 96 -> rejected
    s.feature(300, 100, 0, ur=-1.0)                         # monocular feature: the 2-D gate passes
    s.feature(500, 100, 0, ur=96.0 + 400.0)                 # stereo, er = 0 at u = 500: ur = 496
    s.pair(100, 100); s.pair(300, 100); s.pair(500, 100)
    m = run_both(fo, s)
    assert list(m) == [-1, 1, 2]


def gate_boundary(inv, thr, stereo, bf=F32(40.0), invz=F32(0.1)):
    """A feature at (100, 100) and the two pair positions either side of the gate: the largest reachable F32(e2 * inv) that is
    not > thr (as a double) and the next one.  ex sets the coarse value, a small ey (monocular) or er (stereo, through the
    feature's mvuRight) the fine one.  Returns ((u, v, kpr, p) accepted, (u, v, kpr, p) rejected)."""
    kpx = kpy = F32(100.0)
    ulp = F32(2.0 ** -17)                                   # spacing of float32 in [64, 128)
    u = F32(kpx + F32(np.sqrt(thr / float(inv)) - 4e-4))
    acc = None
    for _ in range(400):
        ex = F32(u - kpx)
        base = F32(ex * ex)
        for n in range(4000):
            d = F32(n * ulp)
            if stereo:
                ur = F32(u - F32(bf * invz))
                kpr = F32(ur - d)
                er = F32(ur - kpr)
                e2 = F32(F32(base + F32(F32(0.0) * F32(0.0))) + F32(er * er))
                v = kpy
            else:
                v = F32(kpy + d)
                ey = F32(v - kpy)
                e2 = F32(base + F32(ey * ey))
                kpr = F32(-1.0)
            p = F32(e2 * inv)
            if float(p) > thr:
                if acc is not None:
                    return acc, (u, v, kpr, p)
                break
            acc = (u, v, kpr, p)
        u = np.nextafter(u, F32(1e9), dtype=np.float32)
    raise AssertionError("no boundary found")


@pytest.mark.parametrize("lvl", [0, 1, 2, 3])
def test_reprojection_gate_edges(fo, lvl):
    """Pairs either side of 5.99 (monocular) and 7.8 (stereo).  At level 0 (inv = 1) the float product reaches every float:
    F32(5.99) lies just below 5.99 and passes; F32(7.8) lies just ABOVE 7.8 and fails against the double constant, which a
    float compare would have let pass."""
    inv = INV_SIGMA2[lvl]
    for thr, stereo in ((5.99, False), (7.8, True)):
        acc, rej = gate_boundary(inv, thr, stereo)
        if lvl == 0:
            assert acc[3] == np.nextafter(rej[3], F32(0), dtype=np.float32)
            assert (acc[3] == F32(5.99)) if thr == 5.99 else (rej[3] == F32(7.8))
        for (u, v, kpr, _), want in ((acc, 0), (rej, -1)):
            s = KFScene(3, stereo=stereo, bf=40.0)
            s.feature(100, 100, 0, octave=lvl, ur=kpr)
            s.pair(u, v, level=lvl, invz=0.1)
            assert list(run_both(fo, s)) == [want], (lvl, thr, u, v, kpr)


def test_distance_50_accepted_51_rejected(fo):
    s = KFScene(5)
    s.feature(100, 100, 50); s.feature(300, 100, 51)
    s.pair(100, 100); s.pair(300, 100)
    assert list(run_both(fo, s)) == [0, -1]


def test_ties_follow_column_row_index(fo):
    """Cell columns have boundaries at 11.75 * (k + 0.5), rows at 10 * (k + 0.5)."""
    s = KFScene(6)
    x0 = 11.75 * 10.5
    s.feature(x0 + 1.5, 105, 7); s.feature(x0 - 1.5, 105, 7)          # column 11 (index 0), column 10 (index 1): 1 wins
    s.pair(x0, 105)
    s.feature(300, 106.5, 9); s.feature(300.5, 103.5, 9)               # same column, row 11 (index 2) and row 10 (index 3): 3 wins
    s.pair(300, 105)
    s.feature(500, 200.5, 4); s.feature(500.5, 200, 4)                 # same cell: the lower index (4) wins
    s.pair(500, 200)
    assert list(run_both(fo, s)) == [1, 3, 4]


def test_upper_image_bounds_are_strict(fo):
    """Level 5 (window 7.46 px, gate e2 <= 37.1): features in the last grid column / row, pairs on and just inside the bounds."""
    s = KFScene(7)
    s.feature(746.0, 100, 0, octave=5); s.feature(100, 474.5, 0, octave=5); s.feature(3.0, 100, 0, octave=5)
    s.pair(752.0, 100, 5); s.pair(np.nextafter(F32(752.0), F32(0)), 100, 5)   # u == mnMaxX rejected, just below accepted
    s.pair(100, 480.0, 5); s.pair(100, np.nextafter(F32(480.0), F32(0)), 5)
    s.pair(np.nextafter(F32(0.0), F32(-1)), 100, 5); s.pair(0.0, 100, 5)       # the lower bounds are inclusive
    assert list(run_both(fo, s)) == [-1, 0, -1, 1, -1, 2]


def test_windows_clipped_at_the_grid_edges(fo):
    """th = 15 at levels 6-7: every window runs past the grid on at least one side and is clamped to it."""
    s = KFScene(8)
    s.feature(0.5, 0.5, 3, octave=7); s.feature(745.5, 474.0, 2, octave=7); s.feature(2, 470, 1, octave=6)
    s.pair(1.0, 1.0, level=7); s.pair(751.0, 479.0, level=7); s.pair(3.0, 472.0, level=7)
    assert list(run_both(fo, s, th=15.0)) == [0, 1, 2]


@pytest.mark.parametrize("seed,crowd,th", [(11, 0, 3.0), (12, 4, 3.0), (13, 0, 5.0)])
def test_random_scenes_match_numpy(fo, seed, crowd, th):
    X, pd, kfs, P = scene(seed, n_kf=3, n_points=250, crowd=crowd, n_distract=150)
    got = fo.fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], th)
    want = py_fuse(kfs, P, pd, th)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    assert got[1].sum() > 50


def test_no_device_is_an_error_not_a_fallback():
    import wut_cuda_orb_slam3_b200 as orbx
    if orbx.lib().orbx_device_count() > 0:
        pytest.skip("a GPU is visible")
    X, pd, kfs, P = scene(21, n_kf=2, n_points=50)
    V = [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS, k["inv_sigma2"], k["bf"], u_right=k["ur"]) for k in kfs]
    with pytest.raises(orbx.OrbxError) as e:
        orbx.fuse(V, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"])
    assert e.value.code == orbx.capi.ORBX_ERR_NO_DEVICE
    with pytest.raises(orbx.OrbxError) as e:                 # argument errors are reported before the device is looked for
        orbx.fuse(V, [0, 60, 50], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"])
    assert e.value.code == orbx.capi.ORBX_ERR_INVALID_ARG


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def test_oracle_reproduces_fuse_golden(fo):
    """tests/golden/fuse_golden.json (made by tests/golden/make_fuse_golden.py from this oracle) still holds."""
    with open(os.path.join(ROOT, "tests", "golden", "fuse_golden.json")) as f:
        gold = json.load(f)["cases"]
    for c in gold:
        X, pd, kfs, P = scene(c["seed"], n_kf=c["n_kf"], n_points=c["n_points"], crowd=c["crowd"], forward=True)
        assert crc(np.concatenate([k["kp"] for k in kfs])) == c["kp_crc"] and crc(pd) == c["desc_crc"] and crc(P["u"]) == c["u_crc"]
        m, nf = fo.fuse(kfs, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], c["th"])
        assert crc(m) == c["match_crc"] and nf.tolist() == c["n_fused"], c["seed"]
