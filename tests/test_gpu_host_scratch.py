"""The calls that take host buffers get their device scratch, pinned staging and stream from the arena of the ORB-SLAM3 thread
that makes them (tracking, local mapping, loop closing).  Three threads calling at once get exactly what each call returns alone;
an arena regrown under a new layout (small, large, then small inputs) still gives the oracle's answers; and orbx_extract_stereo
takes its matcher scratch from the left handle and checks every argument before it queues any work."""
import ctypes as C
import threading

import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import bow_synth
from tests.fuse_synth import BOUNDS, scene
from tests.loop_synth import sbp_scene
from tests.proj_synth import SCALE, make_frame, make_points
from tests.test_oracle_cv2 import _camera
from tests.tri_synth import make_scene
from wut_cuda_orb_slam3_b200 import capi, synth
from wut_cuda_orb_slam3_b200.capi import KP_DTYPE, lib, ptr

pytestmark = pytest.mark.gpu

BF, MAX_D = 47.9, 47.9 / 0.11
COLS, ROWS = 752, 480


def fv_tuple(fv):
    return (fv.node_ids, fv.offsets, fv.indices)


def same(got, want):
    """Results as tuples of arrays / ints, compared byte for byte."""
    assert len(got) == len(want)
    for g, w in zip(got, want):
        if isinstance(g, np.ndarray):
            assert g.shape == w.shape and g.tobytes() == np.ascontiguousarray(w, g.dtype).tobytes()
        else:
            assert g == w


@pytest.fixture(scope="module")
def vocab(oracle):
    parent, desc, weights = bow_synth.make_vocab(601, 10, 4)
    return dict(gpu=orbx.ORBVocabulary(parent, desc, weights, 10, 4), cpu=oracle.vocabulary(parent, desc, weights, 10, 4), desc=desc,
                parent=parent)


# ---- one case per converted call: (call, the oracle's answer), sized by `n` ----------------------------------------------------

def knn2_case(o, vocab, n):
    ndb = 50 * n
    db = synth.descriptors(3, ndb)
    q = synth.descriptors(3, n, is_query=True, ndb=ndb, plant_every=2)
    return (lambda: orbx.ORBmatcher(0.7).knn2(q, db)), o.knn2(q, db)


def stereo_match_case(o, vocab, n):
    imgL = synth.image(40 + n, COLS, ROWS, view=0, max_disp=40)
    imgR = synth.image(40 + n, COLS, ROWS, view=1, max_disp=40)
    exL, exR = orbx.ORBextractor(n, 1.2, 8, 20, 7), orbx.ORBextractor(n, 1.2, 8, 20, 7)
    exL(imgL, None, (0, 0)); exR(imgR, None, (0, 0))
    oL, oR = o.extractor(n, 1.2, 8, 20, 7), o.extractor(n, 1.2, 8, 20, 7)
    kL, dL, _ = oL.extract(imgL, (0, 0)); kR, dR, _ = oR.extract(imgR, (0, 0))
    u, d, _ = o.stereo_match(oL, oR, kL, dL, kR, dR, BF, MAX_D)
    return (lambda: orbx.compute_stereo_matches(exL, exR, kL, dL, kR, dR, BF, MAX_D)), (u, d)


def undistort_case(o, vocab, n):
    rng = np.random.default_rng(n)
    K, d, P = _camera(rng, 1)
    kps = np.zeros(n, KP_DTYPE)
    kps["x"] = rng.uniform(0, COLS, n); kps["y"] = rng.uniform(0, ROWS, n)
    kps["octave"] = rng.integers(0, 8, n); kps["angle"] = rng.uniform(0, 360, n); kps["size"] = 31; kps["class_id"] = -1
    return (lambda: (orbx.undistort_keypoints(kps, K, d, P),)), (o.undistort_keypoints(kps, K, d, P),)


def bow_case(o, vocab, n):
    feats = bow_synth.make_features(n, vocab["desc"], vocab["parent"], n)
    return (lambda: vocab["gpu"].transform_features(feats, 2)), vocab["cpu"].transform_features(feats, 2)


def bow_pair(vocab, n):
    P = bow_synth.make_pair(800 + n, vocab["desc"], vocab["parent"], n, n)
    return P, vocab["gpu"].transform(P["desc_a"], 2)[1], vocab["gpu"].transform(P["desc_b"], 2)[1]


def kf_frame_case(o, vocab, n):
    P, fva, fvb = bow_pair(vocab, n)
    want = o.search_by_bow_kf_frame(P["desc_a"], P["angle_a"], P["valid_a"], fv_tuple(fva), P["desc_b"], P["angle_b"], fv_tuple(fvb),
                                    -1, 0.6, True)

    def call():
        mb, _, nm = orbx.search_by_bow(P["desc_a"], P["angle_a"], P["valid_a"], fva, P["desc_b"], P["angle_b"], fvb, nnratio=0.6)
        return mb, nm
    return call, want


def kf_kf_case(o, vocab, n):
    P, fva, fvb = bow_pair(vocab, n)
    want = o.search_by_bow_kf_kf(P["desc_a"], P["angle_a"], P["valid_a"], fv_tuple(fva), P["desc_b"], P["angle_b"], P["valid_b"],
                                 fv_tuple(fvb), 0.8, True)

    def call():
        _, ma, nm = orbx.search_by_bow(P["desc_a"], P["angle_a"], P["valid_a"], fva, P["desc_b"], P["angle_b"], fvb, valid_b=P["valid_b"],
                                       kf_kf=True, nnratio=0.8)
        return ma, nm
    return call, want


def triangulation_case(o, vocab, n):
    A, (nb,) = make_scene((vocab["gpu"], vocab["desc"], vocab["parent"]), 70 + n, n, 1, n)
    args = (A["kp"], A["desc"], A["free"], A["stereo"])
    want = o.search_for_triangulation(*args, fv_tuple(A["fv"]), nb["kp"], nb["desc"], nb["free"], nb["stereo"], fv_tuple(nb["fv"]),
                                      nb["F12"], nb["ep"], nb["scale"], nb["sigma2"], False, False, True)
    return (lambda: orbx.search_for_triangulation(*args, A["fv"], nb["kp"], nb["desc"], nb["free"], nb["stereo"], nb["fv"], nb["F12"],
                                                  nb["ep"], nb["scale"], nb["sigma2"])), want


def distinctive_case(o, vocab, n):
    counts = np.random.default_rng(n).integers(0, 40, n)
    desc = synth.descriptors(5, int(counts.sum()) + 1)[:counts.sum()]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    want = np.array([o.distinctive_descriptor(desc[off[p]:off[p + 1]]) if counts[p] else -1 for p in range(n)], np.int32)
    return (lambda: (orbx.distinctive_descriptors(desc, off),)), (want,)


def grid_case(o, vocab, n):
    rng = np.random.default_rng(n)
    kp, desc, ur, occ, bounds = make_frame(rng, n)
    fv = orbx.FrameView(kp, desc, SCALE, bounds, u_right=ur, occupied=occ)
    cs, items = o.assign_features_to_grid(kp, fv.bounds_grid())
    area = o.get_features_in_area(kp, fv.bounds_grid(), 376.0, 240.0, 80.0)
    return (lambda: fv.assign_features_to_grid() + (fv.get_features_in_area(376.0, 240.0, 80.0),)), (cs, items, area)


# (case, small size, large size)
CASES = {"knn2": (knn2_case, 300, 4000), "stereo_match": (stereo_match_case, 300, 2000), "undistort": (undistort_case, 50, 20000),
         "bow_transform": (bow_case, 100, 5000), "search_by_bow_kf_frame": (kf_frame_case, 300, 2000),
         "search_by_bow_kf_kf": (kf_kf_case, 300, 2000), "search_for_triangulation": (triangulation_case, 200, 2000),
         "distinctive_descriptors": (distinctive_case, 20, 3000), "grid_and_area": (grid_case, 100, 6000)}


@pytest.mark.parametrize("name", list(CASES))
def test_arena_regrows_under_a_new_layout(oracle, vocab, name):
    """Small, large, small: the second call regrows its thread's arena, the third runs in the grown one with a smaller layout."""
    make, small, large = CASES[name]
    for n in (small, large, small):
        call, want = make(oracle, vocab, n)
        same(call(), want)


def test_three_slam_threads_at_once(oracle, vocab):
    """Tracking, local mapping and loop closing call their searches concurrently, many times each; every result equals what the
    same call returned alone."""
    rng = np.random.default_rng(16)
    kp, desc, ur, occ, bounds = make_frame(rng, 2000)
    Pm = make_points(rng, kp, desc, ur, 1500)
    fv = orbx.FrameView(kp, desc, SCALE, bounds, u_right=ur, occupied=occ)
    margs = (Pm["in_view"], Pm["bad"], Pm["x"], Pm["y"], Pm["xr"], Pm["view_cos"], Pm["depth"], Pm["level"], Pm["n_obs"], Pm["desc"])
    X, pd, kfs, P = scene(17, n_kf=10, n_points=1200)
    V = [orbx.KeyFrameView(k["kp"], k["desc"], k["scale"], BOUNDS, k["inv_sigma2"], k["bf"], u_right=k["ur"]) for k in kfs]
    K, socc, Ps, pds = sbp_scene(18, n_points=4000)
    sfv = orbx.FrameView(K["kp"], K["desc"], K["scale"], BOUNDS, occupied=socc)

    def case(name, n):
        return CASES[name][0](oracle, vocab, n)[0]

    threads = {
        "tracking": [lambda: orbx.search_by_projection_map(fv, *margs, th=1.0, nnratio=0.8), case("knn2", 2000), case("stereo_match", 1200),
                     case("undistort", 1200), case("bow_transform", 1200), case("search_by_bow_kf_frame", 1200)],
        "local mapping": [lambda: orbx.fuse(V, P["kf_offsets"], pd, P["point"], P["valid"], P["u"], P["v"], P["invz"], P["level"], 3.0),
                          case("search_for_triangulation", 1200), case("distinctive_descriptors", 1000)],
        "loop closing": [case("search_by_bow_kf_kf", 1500),
                         lambda: orbx.search_by_projection_sim3(sfv, Ps["valid"], Ps["u"], Ps["v"], Ps["level"], pds, 8, 1.5)],
    }
    alone = {t: [fn() for fn in fns] for t, fns in threads.items()}
    errors = []

    def run(t):
        try:
            for _ in range(30):
                for fn, want in zip(threads[t], alone[t]):
                    same(fn(), want)
        except BaseException as e:       # noqa: BLE001
            errors.append((t, e))

    ts = [threading.Thread(target=run, args=(t,)) for t in threads]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors


def extract_stereo_raw(exL, exR, imgL, imgR, cap, fill=0):
    """orbx_extract_stereo with `cap` rows per output, every output filled with `fill` bytes first; returns (rc, outputs)."""
    out = dict(kL=np.zeros(cap, KP_DTYPE), dL=np.zeros((cap, 32), np.uint8), kR=np.zeros(cap, KP_DTYPE), dR=np.zeros((cap, 32), np.uint8),
               u=np.zeros(cap, np.float32), d=np.zeros(cap, np.float32), nL=np.zeros(1, np.int32), nR=np.zeros(1, np.int32))
    for a in out.values():
        a.view(np.uint8)[...] = fill
    rc = lib().orbx_extract_stereo(exL._h, exR._h, ptr(imgL), ptr(imgR), ROWS, COLS, COLS, ptr(out["kL"]), ptr(out["dL"]), ptr(out["nL"]),
                                   ptr(out["kR"]), ptr(out["dR"]), ptr(out["nR"]), cap, C.c_float(BF), C.c_float(MAX_D), ptr(out["u"]),
                                   ptr(out["d"]))
    return rc, out


def test_extract_stereo_scratch_grows_with_capacity():
    """The matcher's outputs live in the left handle's stereo staging: a larger capacity on the same handles regrows it, and the
    pair still equals what orbx_extract_stereo_batch returns for it."""
    left = np.stack([synth.image(500 + i, COLS, ROWS, view=0, max_disp=40) for i in range(3)])
    right = np.stack([synth.image(500 + i, COLS, ROWS, view=1, max_disp=40) for i in range(3)])
    batch = orbx.ORBextractor(1200, 1.2, 8, 20, 7)
    nL, nR, kL, dL, kR, dR, u, d = batch.extract_stereo_batch(left, right, BF, MAX_D)
    exL, exR = orbx.ORBextractor(1200, 1.2, 8, 20, 7), orbx.ORBextractor(1200, 1.2, 8, 20, 7)
    cap = exL.max_keypoints(ROWS, COLS)
    for i, c in enumerate((cap, 3 * cap, 2 * cap)):
        rc, o = extract_stereo_raw(exL, exR, left[i], right[i], c)
        assert rc == capi.ORBX_OK
        a, b = o["nL"][0], o["nR"][0]
        assert a == nL[i] and b == nR[i] and a > 100
        assert o["kL"][:a].tobytes() == kL[i, :a].tobytes() and o["kR"][:b].tobytes() == kR[i, :b].tobytes()
        assert np.array_equal(o["dL"][:a], dL[i, :a]) and np.array_equal(o["dR"][:b], dR[i, :b])
        assert o["u"][:a].tobytes() == u[i, :a].tobytes() and o["d"][:a].tobytes() == d[i, :a].tobytes()


def test_extract_stereo_refuses_capacity_before_any_work():
    """capacity = 2^20 is past what the stereo kernels index: ORBX_ERR_UNSUPPORTED, and not one byte of the outputs is written."""
    img = synth.image(9, COLS, ROWS)
    exL, exR = orbx.ORBextractor(500, 1.2, 8, 20, 7), orbx.ORBextractor(500, 1.2, 8, 20, 7)
    rc, o = extract_stereo_raw(exL, exR, img, img, 1 << 20, fill=0xA5)
    assert rc == capi.ORBX_ERR_UNSUPPORTED
    for k, a in o.items():
        assert (a.view(np.uint8) == 0xA5).all(), k
    rc, o = extract_stereo_raw(exL, exR, img, img, exL.max_keypoints(ROWS, COLS))        # the handles are still good
    assert rc == capi.ORBX_OK and o["nL"][0] > 100
