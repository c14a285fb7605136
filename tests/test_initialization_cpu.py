"""The SearchForInitialization oracle (tests/cpp/init_oracle.cpp) against an independent brute-force Python restatement of
src/ORBmatcher1.cc:650-765 (CPU), on hand-built scenes for each rule that is easy to get wrong, random initialisation pairs, and
the frozen answers of tests/golden/init_golden.json."""
import json
import os
import zlib

import numpy as np
import pytest

from tests import init_oracle
from tests.init_synth import bounds_grid, init_pair, next_frame
from tests.oracle_lib import KP_DTYPE
from tests.test_projection_cpu import hamming, py_area, py_cells

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BG = bounds_grid()


@pytest.fixture(scope="module")
def ioracle():
    return init_oracle.load()


def c_round(v):
    """C round(): half away from zero."""
    return int(np.floor(v + 0.5)) if v >= 0 else int(np.ceil(v - 0.5))


def three_maxima(counts):
    m1 = m2 = m3 = 0
    i1 = i2 = i3 = -1
    for i, s in enumerate(counts):
        if s > m1:
            m3, m2, m1, i3, i2, i1 = m2, m1, s, i2, i1, i
        elif s > m2:
            m3, m2, i3, i2 = m2, s, i2, i
        elif s > m3:
            m3, i3 = s, i
    if m2 < np.float32(0.1) * np.float32(m1):
        i2 = i3 = -1
    elif m3 < np.float32(0.1) * np.float32(m1):
        i3 = -1
    return {i1, i2, i3}


def py_search_init(kp1, desc1, kp2, desc2, prev, window, ratio, check_ori):
    """src/ORBmatcher1.cc:650-765 written out from its semantics over py_area (brute force over all features, ordered by
    (cell id, index)): skip when vMatchedDistance <= dist before the top-2 update, INT_MAX 'no second-best', take-overs, the
    histogram keeping superseded acceptances, the filter unmatching only live ones."""
    cells = py_cells(kp2, BG)
    n1, n2 = len(kp1), len(kp2)
    m12 = [-1] * n1; m21 = [-1] * n2; md = [2 ** 31 - 1] * n2
    hist = [[] for _ in range(30)]
    nm = 0
    for i1 in range(n1):
        lvl = int(kp1["octave"][i1])
        if lvl > 0:
            continue
        best = best2 = 2 ** 31 - 1
        bi = -1
        for i2 in py_area(kp2, cells, BG, prev[i1][0], prev[i1][1], np.float32(window), lvl, lvl):
            d = hamming(desc1[i1], desc2[i2])
            if md[i2] <= d:
                continue
            if d < best:
                best2, best, bi = best, d, i2
            elif d < best2:
                best2 = d
        if best <= 50 and np.float32(best) < np.float32(best2) * np.float32(ratio):
            if m21[bi] >= 0:
                m12[m21[bi]] = -1
                nm -= 1
            m12[i1] = bi; m21[bi] = i1; md[bi] = best
            nm += 1
            if check_ori:
                rot = np.float32(kp1["angle"][i1]) - np.float32(kp2["angle"][bi])
                if rot < 0:
                    rot = np.float32(rot + np.float32(360))
                b = c_round(np.float32(rot * (np.float32(1) / np.float32(30))))
                hist[0 if b == 30 else b].append(i1)
    if check_ori:
        keep = three_maxima([len(h) for h in hist])
        for b in range(30):
            if b not in keep:
                for i1 in hist[b]:
                    if m12[i1] >= 0:
                        m12[i1] = -1
                        nm -= 1
    out = np.array(prev, np.float32).reshape(n1, 2).copy()
    for i1 in range(n1):
        if m12[i1] >= 0:
            out[i1] = (kp2["x"][m12[i1]], kp2["y"][m12[i1]])
    return np.array(m12, np.int32), nm, out


class Scene:
    """Hand-built pair: features of F2 far apart (70 px), so a query's window holds exactly the candidates placed next to it."""

    def __init__(self, seed=0):
        self.rng = np.random.default_rng(seed)
        self.base = self.rng.integers(0, 256, size=32, dtype=np.uint8)
        self.f2, self.q = [], []

    def desc_at(self, d):
        """A descriptor at Hamming distance d from the base (the first d bits flipped)."""
        bits = np.unpackbits(self.base.copy())
        bits[:d] ^= 1
        return np.packbits(bits)

    def feature(self, x, y, d, octave=0, angle=0.0):
        self.f2.append((x, y, angle, octave, self.desc_at(d)))
        return len(self.f2) - 1

    def query(self, x, y, octave=0, angle=0.0):
        self.q.append((x, y, angle, octave, self.base.copy()))
        return len(self.q) - 1

    @staticmethod
    def _kp(rows):
        kp = np.zeros(len(rows), KP_DTYPE)
        for i, (x, y, a, o, _) in enumerate(rows):
            kp[i]["x"], kp[i]["y"], kp[i]["angle"], kp[i]["octave"] = x, y, a, o
        kp["size"] = 31.0; kp["class_id"] = -1
        return kp, np.array([r[4] for r in rows], np.uint8).reshape(len(rows), 32)

    def arrays(self):
        kp1, d1 = self._kp(self.q)
        kp2, d2 = self._kp(self.f2)
        return kp1, d1, np.stack([kp1["x"], kp1["y"]], 1).astype(np.float32), kp2, d2


def run_both(ioracle, s, window=10, ratio=0.9, check_ori=False):
    kp1, d1, prev, kp2, d2 = s.arrays()
    got = ioracle.search_for_initialization(kp1, d1, kp2, d2, BG, prev, window, ratio, check_ori)
    want = py_search_init(kp1, d1, kp2, d2, prev, window, ratio, check_ori)
    assert got[1] == want[1] and np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])
    return got


def test_distance_256_is_a_real_second_best(ioracle):
    s = Scene(1)
    s.feature(100, 100, 30); s.feature(104, 100, 256)
    s.query(101, 100)
    m, nm, _ = run_both(ioracle, s, ratio=0.1)
    assert nm == 0 and m[0] == -1                          # 30 < 256 * 0.1 fails: the 256 candidate counts


def test_no_second_best_always_passes(ioracle):
    s = Scene(2)
    s.feature(100, 100, 40)
    s.query(101, 100)
    m, nm, prev = run_both(ioracle, s, ratio=0.1)
    assert nm == 1 and m[0] == 0 and tuple(prev[0]) == (100.0, 100.0)


def test_skip_applies_before_the_top2(ioracle):
    """Query 0 takes f at 10.  Query 1 sees g at 4 and f at 14 >= vMatchedDistance[f]: f is skipped before the top-2 update, so
    query 1 has no second-best and passes even ratio 0.25 (with f as its second-best, 4 < 14 * 0.25 would fail)."""
    s = Scene(3)
    f = s.feature(100, 100, 10); g = s.feature(115, 100, 20)
    s.query(100, 100)                                      # window 10 around x = 100: g (x = 115) is outside
    s.q.append((108, 100, 0.0, 0, s.desc_at(24)))          # window around x = 108 holds both
    m, nm, _ = run_both(ioracle, s, ratio=0.25)
    assert list(m) == [f, g] and nm == 2


def test_replacement_and_nondecreasing_distance(ioracle):
    s = Scene(4)
    f = s.feature(200, 200, 0)
    s.q.append((200, 200, 0.0, 0, s.desc_at(30)))          # accepted at 30
    s.q.append((200, 200, 0.0, 0, s.desc_at(20)))          # takes f over at 20: query 0 unmatched
    s.q.append((200, 200, 0.0, 0, s.desc_at(20)))          # 20 again: skipped (vMatchedDistance 20 <= 20)
    s.q.append((200, 200, 0.0, 0, s.desc_at(25)))          # 25 > 20: skipped; unmatching query 0 did not restore 30
    m, nm, _ = run_both(ioracle, s)
    assert list(m) == [-1, f, -1, -1] and nm == 1


def test_superseded_acceptances_count_in_the_histogram(ioracle):
    """Bins 0..3 hold 5, 4, 3 and 1 live matches; bin 3 also holds 3 superseded acceptances, so it outranks bin 2 (4 > 3) and
    bin 2's live matches are the ones the filter removes."""
    s = Scene(5)
    spot = iter([(40.0 + 70 * (k % 10), 40.0 + 70 * (k // 10)) for k in range(20)])
    live = {0: 2, 1: 4, 2: 3, 3: 1}                        # bin 0 gets 3 more live matches from the take-overs below
    for b, k in live.items():
        for _ in range(k):
            x, y = next(spot)
            s.feature(x, y, 0); s.q.append((x, y, 30.0 * b, 0, s.desc_at(0)))
    taken = []
    for _ in range(3):
        x, y = next(spot)
        s.feature(x, y, 0); taken.append((x, y))
        s.q.append((x, y, 90.0, 0, s.desc_at(30)))         # bin 3, accepted at 30 ...
    for x, y in taken:
        s.q.append((x, y, 0.0, 0, s.desc_at(10)))          # ... and taken over at 10 by a bin-0 query
    for check in (False, True):
        m, nm, _ = run_both(ioracle, s, check_ori=check)
    kp1 = s.arrays()[0]
    bins = np.rint(kp1["angle"] / 30).astype(int)
    assert nm == 2 + 4 + 1 + 3 and (m[bins == 2] == -1).all() and (m[bins == 1] >= 0).all()


def test_ties_follow_the_grid_order(ioracle):
    """Equal distances: the first candidate of GetFeaturesInArea (cell column, cell row, index) wins — here feature 1, which
    sits one grid column left of feature 0; with ratio 1.5 the tie passes the ratio test."""
    s = Scene(6)
    s.feature(306, 300, 12); s.feature(294, 300, 12)
    s.query(300, 300)
    m, nm, _ = run_both(ioracle, s, ratio=1.5)
    assert m[0] == 1 and nm == 1
    m, nm, _ = run_both(ioracle, s, ratio=0.9)           # tie at the best distance fails 12 < 12 * 0.9
    assert nm == 0


def test_level_and_window_rules(ioracle):
    s = Scene(7)
    s.feature(100, 100, 5, octave=1)                       # not level 0: invisible
    s.feature(500, 300, 5)
    s.query(100, 100)                                      # window holds nothing usable
    s.query(500, 300, octave=2)                            # level1 > 0: skipped
    s.query(-500, -500)                                    # window outside the grid
    m, nm, _ = run_both(ioracle, s)
    assert nm == 0 and (m == -1).all()


@pytest.mark.parametrize("seed,n2,crowd,ratio,check", [(11, 1500, 0, 0.9, True), (12, 1500, 0, 0.9, False), (13, 600, 4, 0.7, True),
                                                        (14, 400, 2, 1.2, True)])
def test_random_pairs_match_python(ioracle, seed, n2, crowd, ratio, check):
    kp1, d1, prev, kp2, d2 = init_pair(seed, n2, crowd=crowd, dup=1 if not crowd else 3, max_flip=50)
    got = ioracle.search_for_initialization(kp1, d1, kp2, d2, BG, prev, 100, ratio, check)
    want = py_search_init(kp1, d1, kp2, d2, prev, 100, ratio, check)
    assert got[1] == want[1] and np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])
    assert got[1] > 20
    # a chained call on the updated positions, as Tracking does frame after frame
    kp3, d3 = next_frame(seed + 1000, kp2, d2)
    got2 = ioracle.search_for_initialization(kp1, d1, kp3, d3, BG, got[2], 100, ratio, check)
    want2 = py_search_init(kp1, d1, kp3, d3, got[2], 100, ratio, check)
    assert got2[1] == want2[1] and np.array_equal(got2[0], want2[0]) and np.array_equal(got2[2], want2[2])


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def test_oracle_reproduces_init_golden(ioracle):
    """tests/golden/init_golden.json (made by tests/golden/make_init_golden.py from this oracle) still holds."""
    with open(os.path.join(ROOT, "tests", "golden", "init_golden.json")) as f:
        gold = json.load(f)["cases"]
    for c in gold:
        kp1, d1, prev, kp2, d2 = init_pair(c["seed"], c["n2"], crowd=c["crowd"], dup=c["dup"])
        assert crc(kp1) == c["kp1_crc"] and crc(d1) == c["desc1_crc"] and crc(kp2) == c["kp2_crc"] and crc(d2) == c["desc2_crc"]
        m, nm, out = ioracle.search_for_initialization(kp1, d1, kp2, d2, BG, prev, c["window"], c["ratio"], c["check_orientation"])
        assert nm == c["n_matches"] and crc(m) == c["matches12_crc"] and crc(out) == c["prev_crc"], c["seed"]
