"""GPU parity of orbx_search_for_triangulation_batch: ORBmatcher::SearchForTriangulation (src/ORBmatcher2.cc:173-471) of one key
frame against many neighbours in one call.  Every neighbour's row must be bit-identical to the single-pair call
orbx_search_for_triangulation and to the CPU oracle."""
import ctypes as C
import threading

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import bow_synth
from tests.proj_synth import SCALE, make_frame, make_points
from tests.tri_synth import make_scene
from wut_cuda_orb_slam3_b200 import capi

pytestmark = pytest.mark.gpu


def fv_tuple(fv):
    return (fv.node_ids, fv.offsets, fv.indices)


@pytest.fixture(scope="module")
def voc():
    parent, desc, weights = bow_synth.make_vocab(601, 10, 4)
    return orbx.ORBVocabulary(parent, desc, weights, 10, 4), desc, parent


def single(A, nb, only_stereo, check_ori):
    return orbx.search_for_triangulation(A["kp"], A["desc"], A["free"], A["stereo"], A["fv"], nb["kp"], nb["desc"], nb["free"], nb["stereo"],
                                         nb["fv"], nb["F12"], nb["ep"], nb["scale"], nb["sigma2"], only_stereo=only_stereo,
                                         coarse=nb.get("coarse", False), check_orientation=check_ori)


def oracle_one(o, A, nb, only_stereo, check_ori):
    return o.search_for_triangulation(A["kp"], A["desc"], A["free"], A["stereo"], fv_tuple(A["fv"]), nb["kp"], nb["desc"], nb["free"],
                                      nb["stereo"], fv_tuple(nb["fv"]), nb["F12"], nb["ep"], nb["scale"], nb["sigma2"], only_stereo,
                                      nb.get("coarse", False), check_ori)


def batch(A, nbs, only_stereo=False, check_ori=True):
    return orbx.search_for_triangulation_batch(A["kp"], A["desc"], A["free"], A["stereo"], A["fv"], nbs, only_stereo=only_stereo,
                                               check_orientation=check_ori)


def check_rows(oracle, A, nbs, only_stereo, check_ori, with_oracle=True):
    m, nm = batch(A, nbs, only_stereo, check_ori)
    assert m.shape == (len(nbs), len(A["kp"])) and nm.shape == (len(nbs),)
    for k, nb in enumerate(nbs):
        sm, snm = single(A, nb, only_stereo, check_ori)
        assert np.array_equal(m[k], sm) and nm[k] == snm, (k, np.flatnonzero(m[k] != sm)[:10])
        if with_oracle:
            om, onm = oracle_one(oracle, A, nb, only_stereo, check_ori)
            assert np.array_equal(m[k], om) and nm[k] == onm, k
    return m, nm


@pytest.mark.parametrize("check_ori", [True, False])
@pytest.mark.parametrize("coarse", [False, True])
@pytest.mark.parametrize("only_stereo", [False, True])
def test_thirty_neighbours_match_single_calls_and_oracle(oracle, voc, only_stereo, coarse, check_ori):
    """The monocular CreateNewMapPoints shape: 30 neighbours x 1500 features, every neighbour with its own pose and levels."""
    A, nbs = make_scene(voc, 11 + 2 * only_stereo + coarse, 1500, 30, 1500)
    for nb in nbs:
        nb["coarse"] = coarse
    assert len({len(nb["scale"]) for nb in nbs}) > 1
    m, nm = check_rows(oracle, A, nbs, only_stereo, check_ori)
    assert (nm == (m >= 0).sum(axis=1)).all() and nm.sum() > (100 if not coarse else 1000)


def test_mixed_coarse_flags(oracle, voc):
    """bCoarse is per neighbour (the inertial mPrevKF chain searches coarse, the covisible neighbours do not)."""
    A, nbs = make_scene(voc, 31, 1200, 10, 1300)
    for k, nb in enumerate(nbs):
        nb["coarse"] = k % 3 == 0
    check_rows(oracle, A, nbs, False, True)
    check_rows(oracle, A, nbs, True, False)


def test_empty_and_degenerate_neighbours(oracle, voc):
    """No common node, n_b = 0, and (in a second call) every KF1 feature occupied."""
    A, nbs = make_scene(voc, 41, 800, 4, 900)
    nbs[1]["fv"] = orbx.FeatureVector(nbs[1]["fv"].node_ids + 100000, nbs[1]["fv"].offsets, nbs[1]["fv"].indices)
    empty = orbx.FeatureVector(np.zeros(0, np.uint32), np.zeros(1, np.int32), np.zeros(0, np.uint32))
    nbs[2] = dict(nbs[2], kp=nbs[2]["kp"][:0], desc=nbs[2]["desc"][:0], free=nbs[2]["free"][:0], stereo=nbs[2]["stereo"][:0], fv=empty)
    m, nm = check_rows(oracle, A, nbs, False, True)
    assert nm[1] == 0 and nm[2] == 0 and (m[1] < 0).all() and (m[2] < 0).all() and nm[0] > 0 and nm[3] > 0
    A0 = dict(A, free=np.zeros_like(A["free"]))
    m, nm = check_rows(oracle, A0, nbs, False, True)
    assert (m < 0).all() and (nm == 0).all()


def test_no_kf1_features_and_no_neighbours(voc):
    A, nbs = make_scene(voc, 51, 300, 3, 300)
    m, nm = batch(A, [])
    assert m.shape == (0, 300) and nm.shape == (0,)
    empty = orbx.FeatureVector(np.zeros(0, np.uint32), np.zeros(1, np.int32), np.zeros(0, np.uint32))
    A0 = dict(kp=A["kp"][:0], desc=A["desc"][:0], free=A["free"][:0], stereo=A["stereo"][:0], fv=empty)
    m, nm = batch(A0, nbs)
    assert m.shape == (3, 0) and (nm == 0).all()


def one_node(n):
    return orbx.FeatureVector(np.array([7], np.uint32), np.array([0, n], np.int32), np.arange(n, dtype=np.uint32))


def kps(xy, octave=0, angle=10.0):
    kp = np.zeros(len(xy), bow_synth.KP_DTYPE)
    kp["x"] = [p[0] for p in xy]; kp["y"] = [p[1] for p in xy]
    kp["octave"] = octave; kp["angle"] = angle; kp["size"] = 31; kp["class_id"] = -1
    return kp


def with_bits(nbits):
    """Descriptors with the first nbits[i] bits set: distance to the zero descriptor = nbits[i]."""
    d = np.zeros((len(nbits), 256), np.uint8)
    for i, b in enumerate(nbits):
        d[i, :b] = 1
    return np.packbits(d, axis=1)


def test_thresholds_ties_den_zero_and_epipole_edge(oracle):
    """Hand-built neighbours in one call: distance 50 accepted / 51 rejected; equal distances -> the later candidate wins;
    den == 0 rejects every candidate unless coarse; the epipole gate keeps a candidate at exactly 10 * sqrt(scale) and drops
    one just inside."""
    A = dict(kp=kps([(300.0, 200.0)]), desc=with_bits([0]), free=np.ones(1, np.uint8), stereo=np.zeros(1, np.uint8), fv=one_node(1))
    scale = np.ones(8, np.float32); sigma2 = np.full(8, 1e30, np.float32)
    F_line = np.zeros((3, 3), np.float32); F_line[0, 0] = 1.0                # la = x1, lb = lc = 0: the line x = 0 in image 2
    F_zero = np.zeros((3, 3), np.float32); F_zero[2, 2] = 1.0               # la = lb = 0: den == 0
    far = np.array([-5000.0, -5000.0], np.float32)

    def nb(xy, bits, F12=F_zero, ep=far, coarse=True, stereo=0):
        n = len(xy)
        return dict(kp=kps(xy), desc=with_bits(bits), free=np.ones(n, np.uint8), stereo=np.full(n, stereo, np.uint8), fv=one_node(n),
                    F12=F12, ep=ep, scale=scale, sigma2=sigma2, coarse=coarse)

    ep = np.array([100.0, 100.0], np.float32)
    nbs = [nb([(10.0, 10.0), (20.0, 20.0)], [51, 50]),                       # 0: 51 rejected, 50 accepted -> 1
           nb([(10.0, 10.0), (20.0, 20.0), (30.0, 30.0), (40.0, 40.0)], [12, 12, 30, 12]),   # 1: tie -> the last 12 (index 3)
           nb([(10.0, 10.0), (20.0, 20.0)], [5, 5], F12=F_zero, coarse=False),       # 2: den == 0 -> none
           nb([(10.0, 10.0), (20.0, 20.0)], [5, 5], F12=F_zero, coarse=True),        # 3: coarse skips the line test -> 1
           nb([(110.0, 100.0), (100.0, 109.99)], [3, 2], ep=ep),                     # 4: on the gate's edge kept, inside dropped -> 0
           nb([(100.0, 109.99)], [2], ep=ep, stereo=1),                              # 5: a stereo candidate skips the gate -> 0
           nb([(0.0, 50.0), (0.5, 60.0)], [4, 3], F12=F_line, coarse=False)]         # 6: on the line kept, 0.5 px off dropped -> 0
    nbs[6]["sigma2"] = np.full(8, 0.06, np.float32)                          # dsqr = 0.25 against 3.84 * 0.06 = 0.2304
    m, nm = check_rows(oracle, A, nbs, False, False)
    assert m[:, 0].tolist() == [1, 3, -1, 1, 0, 0, 0], m[:, 0]
    assert nm.tolist() == [1, 1, 0, 1, 1, 1, 1]


def bad_view(A, nbs, k, field, value):
    """The views of the wrapper, with field `field` of neighbour k replaced (None = a NULL pointer)."""
    views = (capi.TriangulationViewC * len(nbs))()
    keep = []
    for i, nb in enumerate(nbs):
        arrs = {f: np.ascontiguousarray(nb[f]) for f in ("kp", "desc", "free", "stereo", "scale", "sigma2")}
        keep.append(arrs)
        v = views[i]
        v.n = len(arrs["kp"]); v.kp = capi.ptr(arrs["kp"]); v.desc = capi.ptr(arrs["desc"]); v.free = capi.ptr(arrs["free"])
        v.stereo = capi.ptr(arrs["stereo"]); v.fv = nb["fv"].c_struct(); v.F12[:] = [float(x) for x in nb["F12"].reshape(9)]
        v.ep[:] = [float(x) for x in nb["ep"]]; v.scale = capi.ptr(arrs["scale"]); v.sigma2 = capi.ptr(arrs["sigma2"])
        v.n_levels = len(arrs["scale"])
        if i == k:
            setattr(v, field, value)
    n_a = len(A["kp"])
    m = np.zeros((len(nbs), n_a), np.int32); nm = np.zeros(len(nbs), np.int32)
    fa = A["fv"].c_struct()
    rc = orbx.lib().orbx_search_for_triangulation_batch(0, capi.ptr(A["kp"]), capi.ptr(A["desc"]), capi.ptr(A["free"]), capi.ptr(A["stereo"]),
                                                        n_a, C.addressof(fa), len(nbs), C.addressof(views), 0, 1, capi.ptr(m), capi.ptr(nm))
    return rc


def test_bad_arguments_rejected_per_neighbour(voc):
    """Each of the single call's rejections, on neighbour 2 of 4 (the earlier ones are fine)."""
    A, nbs = make_scene(voc, 61, 400, 4, 400)
    for field in ("kp", "desc", "free", "stereo", "scale", "sigma2"):
        assert bad_view(A, nbs, 2, field, None) == capi.ORBX_ERR_INVALID_ARG, field
    assert bad_view(A, nbs, 2, "n_levels", 0) == capi.ORBX_ERR_INVALID_ARG
    assert bad_view(A, nbs, 2, "n_levels", 17) == capi.ORBX_ERR_INVALID_ARG
    assert bad_view(A, nbs, 2, "n", -1) == capi.ORBX_ERR_INVALID_ARG
    assert bad_view(A, nbs, 2, "n_levels", 3) == capi.ORBX_ERR_INVALID_ARG          # octaves up to 3 and more now out of range
    rev = orbx.FeatureVector(nbs[2]["fv"].node_ids[::-1].copy(), nbs[2]["fv"].offsets, nbs[2]["fv"].indices)
    big = orbx.FeatureVector(nbs[2]["fv"].node_ids, nbs[2]["fv"].offsets, nbs[2]["fv"].indices + 10000)
    for fv in (rev, big):
        with pytest.raises(orbx.OrbxError):
            batch(A, nbs[:2] + [dict(nbs[2], fv=fv)] + nbs[3:])
    kp = nbs[2]["kp"].copy(); kp["octave"][5] = len(nbs[2]["scale"])
    with pytest.raises(orbx.OrbxError):
        batch(A, nbs[:2] + [dict(nbs[2], kp=kp)] + nbs[3:])
    kp["octave"][5] = -1
    with pytest.raises(orbx.OrbxError):
        batch(A, nbs[:2] + [dict(nbs[2], kp=kp)] + nbs[3:])
    with pytest.raises(orbx.OrbxError):                                              # KF1's own feature vector
        batch(dict(A, fv=orbx.FeatureVector(A["fv"].node_ids[::-1].copy(), A["fv"].offsets, A["fv"].indices)), nbs)
    assert orbx.lib().orbx_search_for_triangulation_batch(0, None, None, None, None, 0, None, -1, None, 0, 0, None, None) == \
        capi.ORBX_ERR_INVALID_ARG
    assert orbx.lib().orbx_search_for_triangulation_batch(0, None, None, None, None, 0, None, 0, None, 0, 0, None, None) == capi.ORBX_OK
    check_rows(None, A, nbs, False, True, with_oracle=False)                         # and the good call still works afterwards


def test_alongside_tracking_thread(oracle, voc):
    """A batched call on the local-mapping thread and orbx_search_by_projection_map on the tracking thread at once, 30 calls
    each: both bit-exact (their scratch arenas are separate)."""
    rng = np.random.default_rng(8)
    kp, desc, ur, occ, bounds = make_frame(rng, 2000)
    Pm = make_points(rng, kp, desc, ur, 1500)
    fv = orbx.FrameView(kp, desc, SCALE, bounds, u_right=ur, occupied=occ)
    margs = (Pm["in_view"], Pm["bad"], Pm["x"], Pm["y"], Pm["xr"], Pm["view_cos"], Pm["depth"], Pm["level"], Pm["n_obs"], Pm["desc"])
    want_m = oracle.search_by_projection_map(kp, desc, ur, occ, fv.bounds_grid(), SCALE, *margs, 1.0, False, 0.0, 0.8)
    A, nbs = make_scene(voc, 71, 1500, 20, 1500)
    want_t = [oracle_one(oracle, A, nb, False, True) for nb in nbs]
    errors = []

    def tracking():
        try:
            for _ in range(30):
                got = orbx.search_by_projection_map(fv, *margs, th=1.0, nnratio=0.8)
                assert got[1] == want_m[1] and np.array_equal(got[0], want_m[0])
        except BaseException as e:       # noqa: BLE001
            errors.append(e)

    def mapping():
        try:
            for _ in range(30):
                m, nm = batch(A, nbs)
                for k, (om, onm) in enumerate(want_t):
                    assert np.array_equal(m[k], om) and nm[k] == onm
        except BaseException as e:       # noqa: BLE001
            errors.append(e)

    ts = [threading.Thread(target=tracking), threading.Thread(target=mapping)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors
