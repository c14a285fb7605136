"""GPU parity of SearchForInitialization (src/ORBmatcher1.cc:650-765): the CUDA path (mode 2 of the projection search, DESIGN.md
§5b) through the C ABI against the oracle's sequential loop, bit-exact in vnMatches12, the return value and vbPrevMatched."""
import ctypes as C
import json
import os
import zlib

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import init_oracle
from tests.init_synth import BOUNDS, bounds_grid, init_pair, make_f1, make_f2, next_frame
from tests.proj_synth import SCALE

pytestmark = pytest.mark.gpu
BG = bounds_grid()
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ioracle():
    return init_oracle.load()


def view(kp2, desc2):
    return orbx.FrameView(kp2, desc2, SCALE, BOUNDS)


def check(ioracle, kp1, d1, prev, kp2, d2, window=100, ratio=0.9, ori=True):
    got = orbx.search_for_initialization(kp1, d1, view(kp2, d2), prev, window, ratio, ori)
    want = ioracle.search_for_initialization(kp1, d1, kp2, d2, BG, prev, window, ratio, ori)
    assert got[1] == want[1], (got[1], want[1], orbx.projection_rounds())
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2])
    return got


@pytest.mark.parametrize("seed", [1, 2])
def test_initialisation_pair_and_chained_call(ioracle, seed):
    """5000 F2 features (about 30 % at level 0), F1 = its level-0 features moved 0-40 px with 0-60 flipped bits plus distractors."""
    kp1, d1, prev, kp2, d2 = init_pair(seed, 5000)
    for ori in (True, False):
        m, nm, out = check(ioracle, kp1, d1, prev, kp2, d2, ori=ori)
        assert nm > 500
    kp3, d3 = next_frame(seed + 100, kp2, d2)
    check(ioracle, kp1, d1, out, kp3, d3)                   # next frame, on the updated vbPrevMatched


@pytest.mark.parametrize("seed,n2,crowd,dup,ratio", [(21, 300, 2, 6, 0.9), (22, 1200, 5, 3, 0.9), (23, 800, 3, 4, 1.3), (24, 40, 1, 10, 0.7)])
def test_crowded_scenes(ioracle, seed, n2, crowd, dup, ratio):
    """Many queries near the same few features: take-overs, superseded histogram entries, several speculation rounds."""
    kp1, d1, prev, kp2, d2 = init_pair(seed, n2, crowd=crowd, dup=dup, max_flip=45, max_move=10.0)
    for ori in (True, False):
        check(ioracle, kp1, d1, prev, kp2, d2, window=60, ratio=ratio, ori=ori)


def test_random_scenes_with_ties(ioracle):
    """Few distinct descriptors: equal distances everywhere, shared second-best candidates, out-of-order decisions."""
    for seed in range(300, 360):
        rng = np.random.default_rng(seed)
        n2 = int(rng.integers(20, 600))
        kp2, d2 = make_f2(rng, n2, crowd=int(rng.integers(1, 6)), p0=0.6)
        d2 = d2[rng.integers(0, max(2, n2 // 8), n2)]
        kp1, d1, prev = make_f1(rng, kp2, d2, max_move=15.0, max_flip=30, n_distract=int(rng.integers(0, 100)), dup=int(rng.integers(1, 5)))
        window = int(rng.choice([10, 30, 100])); ratio = float(rng.choice([0.6, 0.9, 1.0, 1.5]))
        got = orbx.search_for_initialization(kp1, d1, view(kp2, d2), prev, window, ratio, True)
        want = ioracle.search_for_initialization(kp1, d1, kp2, d2, BG, prev, window, ratio, True)
        assert got[1] == want[1] and np.array_equal(got[0], want[0]) and np.array_equal(got[2], want[2]), (seed, orbx.projection_rounds())


def test_identical_descriptors(ioracle):
    """Every query claims every feature of its window: one decision per round, and the result still equals the loop."""
    rng = np.random.default_rng(41)
    kp2, d2 = make_f2(rng, 64, crowd=1, p0=1.0)
    d2[:] = d2[0]
    kp1, d1, prev = make_f1(rng, kp2, d2, max_move=5.0, max_flip=0, n_distract=0, dup=3)
    check(ioracle, kp1, d1, prev, kp2, d2, window=100, ori=False)
    assert orbx.projection_rounds() >= 10


def test_empty_cases(ioracle):
    kp1, d1, prev, kp2, d2 = init_pair(51, 400)
    m, nm, out = check(ioracle, kp1[:0], d1[:0], prev[:0], kp2, d2)                     # n1 = 0
    assert nm == 0 and len(m) == 0
    m, nm, out = check(ioracle, kp1, d1, prev, kp2[:0], d2[:0])                         # F2.N = 0
    assert nm == 0 and (m == -1).all() and np.array_equal(out, prev)
    k2 = kp2.copy(); k2["octave"] = np.maximum(k2["octave"], 1)                        # no level-0 feature in F2
    m, nm, _ = check(ioracle, kp1, d1, prev, k2, d2)
    assert nm == 0
    far = np.full_like(prev, -5000.0)                                                   # every window outside the grid
    m, nm, _ = check(ioracle, kp1, d1, far, kp2, d2)
    assert nm == 0


def test_bad_arguments():
    kp1, d1, prev, kp2, d2 = init_pair(61, 600)
    k1 = kp1.copy(); k1["angle"] = 1000.0                                               # rot = 1000 - angle2: outside the histogram
    with pytest.raises(orbx.OrbxError):
        orbx.search_for_initialization(k1, d1, view(kp2, d2), prev, 100, 0.9, True)
    orbx.search_for_initialization(k1, d1, view(kp2, d2), prev, 100, 0.9, False)       # no histogram: nothing to assert
    fv = view(kp2, d2)
    nm = C.c_int(0)
    kp1c = np.ascontiguousarray(kp1); d1c = np.ascontiguousarray(d1); pc = prev.copy(); m = np.zeros(len(kp1), np.int32)
    args = [0, kp1c.ctypes.data, d1c.ctypes.data, len(kp1), C.addressof(fv.c), pc.ctypes.data, 100, 0.9, 1, m.ctypes.data, C.addressof(nm)]
    for k in (9, 10, 5):                                                                # null matches12, n_matches, prev_matched
        a = list(args); a[k] = None
        with pytest.raises(orbx.OrbxError):
            orbx.capi.check(orbx.lib().orbx_search_for_initialization(*a))


def crc(a):
    return zlib.crc32(np.ascontiguousarray(a).tobytes()) & 0xFFFFFFFF


def test_cuda_reproduces_init_golden():
    """tests/golden/init_golden.json, without touching oracle code."""
    with open(os.path.join(ROOT, "tests", "golden", "init_golden.json")) as f:
        gold = json.load(f)["cases"]
    for c in gold:
        kp1, d1, prev, kp2, d2 = init_pair(c["seed"], c["n2"], crowd=c["crowd"], dup=c["dup"])
        assert crc(kp1) == c["kp1_crc"] and crc(d2) == c["desc2_crc"]
        m, nm, out = orbx.search_for_initialization(kp1, d1, view(kp2, d2), prev, c["window"], c["ratio"], c["check_orientation"])
        assert nm == c["n_matches"] and crc(m) == c["matches12_crc"] and crc(out) == c["prev_crc"], c["seed"]
