"""CUDA path (through the C ABI) directly against the REFERENCE's own compiled functions (oracle/_ref/libref.so, built by
oracle/build_ref.sh where ORB_REFERENCE_ROOT names a reference checkout) — no oracle code between the two, except where an
OpenCV-owned primitive has to produce the input.  Where the library is not built, the CUDA path's answers are compared with the
stored CRCs of the reference's answers on the same inputs (tests/golden/ref_pin_golden.json, see ref_lib.Pin)."""
import numpy as np
import pytest

import wut_cuda_orb_slam3_b200 as orbx
from tests import bow_synth, ref_cases, ref_lib
from tests.proj_synth import SCALE, make_frame, make_points
from wut_cuda_orb_slam3_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ref():
    return ref_lib.load() if ref_lib.available() else None


@pytest.fixture
def pin(request):
    return ref_lib.Pin(request.node.name)


def test_tables_vs_reference_ctor(ref, pin):
    keys = ("scale", "inv", "sigma2", "invsigma2", "nfeat")
    for nf, sf, nl in [(1000, 1.2, 8), (1200, 1.2, 8), (2000, 1.2, 8), (500, 1.5, 5)]:
        t = orbx.compute_tables(nf, sf, nl); r = ref.tables(nf, sf, nl) if ref else None
        pin("%d_%g_%d" % (nf, sf, nl), [t[k] for k in keys], r and [r[k] for k in keys])


def test_octree_kernel_vs_reference_distribute_octree(ref, pin):
    got, want = [], []
    for case in range(120):
        xs, ys, sc, w, h, N = ref_cases.octree_inputs(case)
        idx = orbx.distribute_octree(xs, ys, sc, 16, 16 + w, 16, 16 + h, N)
        got += [xs[idx], ys[idx], sc[idx]]
        if ref:
            want += ref.distribute_octree(xs, ys, sc, 16, 16 + w, 16, 16 + h, N)
    pin("octree", got, want if ref else None)


@pytest.mark.parametrize("cols,rows,seed", [(752, 480, 1), (331, 277, 7)])
def test_fast_cells_vs_reference_tile_calc(ref, pin, cols, rows, seed):
    img = synth.image(seed, cols, rows)
    ex = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    ex(img, None, (0, 0))
    pin("cells", ex.candidates(0), ref and ref.tile_calc_keypoints(img, 1000, 20, 7))


def test_extract_levels_vs_reference_octree_and_descriptor(ref, pin):
    """Whole extraction: per level, the retained key points must be DistributeOctTree(tileCalcKeypoints(level)) and the
    descriptors computeOrbDescriptor on the blurred level, all by the reference's code."""
    img = synth.image(5, 752, 480)
    ex = orbx.ORBextractor(1000, 1.2, 8, 20, 7)
    ex(img, None, (0, 0))
    nfeat = orbx.compute_tables(1000, 1.2, 8)["nfeat"]
    for l in range(8):
        kps, desc = ex.level_keypoints(l)
        want = None
        if ref:
            lvl = ex.pyramid_level(l)
            h, w = lvl.shape
            rx, ry, rs = ref.tile_calc_keypoints(lvl, 1000, 20, 7)
            ox, oy, osc = ref.distribute_octree(rx, ry, rs, 16, w - 16, 16, h - 16, int(nfeat[l]), l)
            blurred = ex.blurred_level(l)
            # same angle in, same bits out
            rd = [ref.descriptor(blurred, int(kps["x"][i]), int(kps["y"][i]), float(kps["angle"][i])) for i in range(0, len(kps), 3)]
            want = [(ox + 16).astype(np.float32), (oy + 16).astype(np.float32), osc.astype(np.float32), np.array(rd, np.uint8).reshape(-1, 32)]
        pin("level%d" % l, [kps["x"], kps["y"], kps["response"], desc[::3]], want)


def test_stereo_vs_reference_compute_stereo_matches(ref, pin):
    left = synth.image(31, 752, 480, view=0); right = synth.image(31, 752, 480, view=1)
    exL = orbx.ORBextractor(1200, 1.2, 8, 20, 7); exR = orbx.ORBextractor(1200, 1.2, 8, 20, 7)
    _, kL, dL = exL(left, None, (0, 0)); _, kR, dR = exR(right, None, (0, 0))
    mbf, mb = np.float32(47.9), np.float32(0.11)
    u, d = orbx.compute_stereo_matches(exL, exR, kL, dL, kR, dR, mbf, np.float32(mbf / mb))
    pyrL = [exL.pyramid_level(l, with_border=True) for l in range(8)]; pyrR = [exR.pyramid_level(l, with_border=True) for l in range(8)]
    t = orbx.compute_tables(1200, 1.2, 8)
    want = ref and ref.compute_stereo_matches(kL, dL, kR, dR, pyrL, pyrR, t["scale"], t["inv"], mb, mbf)
    assert (u >= 0).sum() > 50
    pin("stereo", [u.view(np.uint32), d.view(np.uint32)], want and [a.view(np.uint32) for a in want])


def test_projection_searches_vs_reference(ref, pin):
    rng = np.random.default_rng(42)
    kp, desc, ur, occ, bounds = make_frame(rng, 900, crowd=8)
    P = make_points(rng, kp, desc, ur, 2200, dup_frac=0.6, max_flip=100)
    fv = orbx.FrameView(kp, desc, SCALE, bounds, u_right=ur, occupied=occ)
    bg = fv.bounds_grid()
    got, nm = orbx.search_by_projection_map(fv, P["in_view"], P["bad"], P["x"], P["y"], P["xr"], P["view_cos"], P["depth"], P["level"], P["n_obs"],
                                            P["desc"], th=4.0, far_points=True, th_far_points=25.0, nnratio=0.8)
    want = ref and ref.search_by_projection_map(kp, desc, ur, occ, bg, SCALE, P["in_view"], P["bad"], P["x"], P["y"], P["xr"], P["view_cos"],
                                                P["depth"], P["level"], P["n_obs"], P["desc"], th=4.0, far=True, th_far=25.0, nnratio=0.8)
    assert nm > 50
    pin("map", [got, np.int32(nm)], want and [want[0], np.int32(want[1])])
    invz = ref_lib.invz(P["depth"])
    for tz in (0.0, 2.0, -2.0):
        want = None
        if ref:
            rm, rnm, rinvz = ref.search_by_projection_last(kp, desc, ur, occ, bg, SCALE, 40.0, P["valid"], P["x"], P["y"], P["depth"], P["level"],
                                                           P["angle"], P["n_obs"], P["desc"], 15.0, last_tz=tz)
            assert rinvz.tobytes() == invz.tobytes()
            want = [rm, np.int32(rnm)]
        got, nm = orbx.search_by_projection_last(fv, 40.0, P["valid"], P["x"], P["y"], invz, P["level"], P["angle"], P["n_obs"], P["desc"], 15.0,
                                                 forward=tz > 1.0, backward=-tz > 1.0)
        assert nm > 50
        pin("last_tz=%g" % tz, [got, np.int32(nm)], want)
    found = (rng.random(len(P["x"])) < 0.1).astype(np.uint8)
    d3 = ref_lib.dist3d(P["x"], P["y"], P["depth"])
    want = None
    if ref:
        rm, rnm, rd3 = ref.search_by_projection_kf(kp, desc, occ, bg, SCALE, P["valid"], found, P["x"], P["y"], P["depth"], P["min_dist"] * 30,
                                                   P["max_dist"] * 30, P["level"], P["angle"], P["desc"], 10.0, 100)
        assert rd3.tobytes() == d3.tobytes()
        want = [rm, np.int32(rnm)]
    fv2 = orbx.FrameView(kp, desc, SCALE, bounds, occupied=occ)
    got, nm = orbx.search_by_projection_kf(fv2, P["valid"] & (1 - found), P["x"], P["y"], d3, P["min_dist"] * 30, P["max_dist"] * 30, P["level"],
                                           P["angle"], P["desc"], 10.0, 100)
    assert nm > 50
    pin("kf", [got, np.int32(nm)], want)


def test_search_by_bow_vs_reference(ref, pin, oracle):
    k, L = 10, 4
    parent, vdesc, weights = bow_synth.make_vocab(601, k, L)
    voc = orbx.ORBVocabulary(parent, vdesc, weights, k, L)
    B = bow_synth.make_pair(602, vdesc, parent, 1500, 1400)
    _, fva = voc.transform(B["desc_a"], 4); _, fvb = voc.transform(B["desc_b"], 4)
    t = lambda fv: (fv.node_ids, fv.offsets, fv.indices)   # noqa: E731
    mb, ma, nm = orbx.search_by_bow(B["desc_a"], B["angle_a"], B["valid_a"], fva, B["desc_b"], B["angle_b"], fvb, nnratio=0.7)
    want = ref and ref.search_by_bow_kf_frame(B["desc_a"], B["angle_a"], B["valid_a"], t(fva), B["desc_b"], B["angle_b"], t(fvb), -1, 0.7, True)
    assert nm > 50
    pin("kf_frame", [mb, np.int32(nm)], want and [want[0], np.int32(want[1])])
    mb, ma, nm = orbx.search_by_bow(B["desc_a"], B["angle_a"], B["valid_a"], fva, B["desc_b"], B["angle_b"], fvb, valid_b=B["valid_b"], kf_kf=True,
                                    nnratio=0.8)
    want = ref and ref.search_by_bow_kf_kf(B["desc_a"], B["angle_a"], B["valid_a"], t(fva), B["desc_b"], B["angle_b"], B["valid_b"], t(fvb), 0.8, True)
    assert nm > 50
    pin("kf_kf", [ma, np.int32(nm)], want and [want[0], np.int32(want[1])])


def test_bow_transform_vs_dbow2(ref, pin, tmp_path):
    """The CUDA vocabulary descent + host BowVector / FeatureVector assembly against DBoW2's own compiled transform, both
    loading the same ORBvoc-format file (no trailing newline: see tests/test_ref_pin.py)."""
    k, L = 10, 4
    parent, vdesc, weights = bow_synth.make_vocab(611, k, L)
    path = tmp_path / "voc.txt"
    bow_synth.write_vocab_text(path, parent, vdesc, weights, k, L, 0, 0)
    txt = open(path).read().rstrip()
    open(path, "w").write(txt)
    rv = ref and ref_lib.RefVocabulary(ref, path)
    voc = orbx.ORBVocabulary.loadFromTextFile(path)
    feats = bow_synth.make_features(612, vdesc, parent, 3000)
    pin("transform_features", voc.transform_features(feats, 4), rv and rv.transform_features(feats, 4))
    (ids, vals), fv = voc.transform(feats, 4)
    (ids2, vals2), _ = voc.transform(bow_synth.make_features(613, vdesc, parent, 2500), 4)
    got = [ids, vals.view(np.uint64), fv.node_ids, fv.offsets, fv.indices, np.float64(voc.score((ids, vals), (ids2, vals2))).view(np.uint64)]
    want = None
    if rv:
        (rid, rval), rfv = rv.transform(feats, 4)
        want = [rid, rval.view(np.uint64), *rfv, np.float64(rv.score((rid, rval), (ids2, vals2))).view(np.uint64)]
    pin("transform_score", got, want)
