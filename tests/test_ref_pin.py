"""PINS THE ORACLE AGAINST THE REFERENCE'S OWN COMPILED CODE (oracle/_ref/libref.so, built by oracle/build_ref.sh from the
reference sources where they lie): constructor tables, DistributeOctTree (with its std::sort tie behaviour), the CPU cell loop
tileCalcKeypoints, computeOrbDescriptor + bit_pattern_31_, the placement loop of operator(), DescriptorDistance,
ComputeThreeMaxima, the frame grid and the three SearchByProjection overloads.  CPU only.  Where the library is not built
(it is built only where ORB_REFERENCE_ROOT names a reference checkout), the oracle's answers are compared with the stored CRCs of
the reference's answers on the same inputs (tests/golden/ref_pin_golden.json, see ref_lib.Pin)."""
import numpy as np
import pytest

from tests import ref_lib
from tests import bow_synth
from tests.proj_synth import SCALE, make_frame, make_points
from wut_cuda_orb_slam3_b200 import synth



@pytest.fixture(scope="module")
def ref():
    return ref_lib.load() if ref_lib.available() else None


@pytest.fixture
def pin(request):
    return ref_lib.Pin(request.node.name)


@pytest.mark.parametrize("nf,sf,nl", [(1000, 1.2, 8), (1200, 1.2, 8), (2000, 1.2, 8), (5000, 1.2, 8), (500, 1.5, 5), (300, 2.0, 4), (1500, 1.1, 12)])
def test_tables_match_reference_ctor(oracle, ref, pin, nf, sf, nl):
    o = oracle.tables(nf, sf, nl)
    import os, re
    inc = open(os.path.join(os.path.dirname(ref_lib.ROOT + "/x"), "wut_cuda_orb_slam3_b200", "csrc", "brief_pattern.inc")).read()
    mine = np.array([int(t) for t in re.findall(r"-?\d+", re.sub(r"//.*", "", inc))], np.int32)
    keys = ("scale", "inv", "sigma2", "invsigma2", "nfeat", "umax")
    r = ref.tables(nf, sf, nl) if ref else None
    pin("tables", [o[k] for k in keys] + [mine], r and [r[k] for k in keys] + [r["pattern"]])


def random_candidates(rng, n, w, h, mode):
    if mode == 0:
        xs = rng.integers(0, w, n); ys = rng.integers(0, h, n)
    elif mode == 1:                       # clustered
        cx, cy = rng.integers(0, w, 6), rng.integers(0, h, 6)
        k = rng.integers(0, 6, n)
        xs = np.clip(cx[k] + rng.integers(-12, 13, n), 0, w - 1); ys = np.clip(cy[k] + rng.integers(-12, 13, n), 0, h - 1)
    else:                                 # lattice: many nodes with equal counts and equal UL.x => std::sort ties
        xs = (rng.integers(0, max(w // 8, 1), n) * 8) % w; ys = (rng.integers(0, max(h // 8, 1), n) * 8) % h
    pts = np.unique(np.stack([ys, xs], 1), axis=0)            # distinct pixels, (y, x) ascending like the cell loop's output
    sc = rng.integers(7, 60 if mode == 2 else 200, len(pts))
    return pts[:, 1].astype(np.int32), pts[:, 0].astype(np.int32), sc.astype(np.int32)


def test_distribute_octree_matches_reference(oracle, ref, pin):
    rng = np.random.default_rng(5)
    n_cases = 0
    got, want = [], []
    for case in range(1500):
        w, h = [(720, 448), (595, 368), (178, 102), (1209, 344), (1248, 688), (64, 40)][case % 6]
        n = int(rng.integers(1, 3000)) if case % 7 else int(rng.integers(1, 40))
        N = int(rng.choice([217, 60, 434, 1000, 25]))
        xs, ys, sc = random_candidates(rng, n, w, h, case % 3)
        idx = oracle.octree(xs, ys, sc, 16, 16 + w, 16, 16 + h, N)
        got += [xs[idx], ys[idx], sc[idx]]
        if ref:
            want += ref.distribute_octree(xs, ys, sc, 16, 16 + w, 16, 16 + h, N)
        n_cases += 1
    assert n_cases == 1500
    pin("octree", got, want if ref else None)


@pytest.mark.parametrize("cols,rows,seed", [(752, 480, 1), (627, 400, 2), (210, 134, 3), (1241, 376, 4), (346, 105, 5), (160, 120, 6), (331, 277, 7)])
def test_cell_loop_matches_reference_tile_calc(oracle, ref, pin, cols, rows, seed):
    img = synth.image(seed, cols, rows)
    x, y, s = oracle.cell_fast(img, 20, 7)
    assert len(x) > 10
    pin("20_7", [x, y, s], ref and ref.tile_calc_keypoints(img, 1000, 20, 7))
    x, y, s = oracle.cell_fast(img, 60, 30)                 # high thresholds: many cells take the minThFAST retry / stay empty
    pin("60_30", [x, y, s], ref and ref.tile_calc_keypoints(img, 1000, 60, 30))


def test_descriptor_matches_reference(oracle, ref, pin):
    rng = np.random.default_rng(9)
    img = synth.image(11, 400, 300)
    blurred = oracle.blur(img)
    got, want = [], []
    for _ in range(3000):
        x, y = int(rng.integers(19, 400 - 19)), int(rng.integers(19, 300 - 19))
        ang = float(np.float32(rng.uniform(0, 360)))
        if _ % 10 == 0:
            ang = float(rng.integers(0, 8) * 45)
        got.append(oracle.descriptor(blurred, x, y, ang))
        if ref:
            want.append(ref.descriptor(blurred, x, y, ang))
    pin("descriptors", got, want if ref else None)


@pytest.mark.parametrize("lap", [(0, 0), (0, 1000), (300, 450)])
def test_packing_matches_reference_loop(oracle, ref, pin, lap):
    img = synth.image(21, 752, 480)
    ex = oracle.extractor(1000, 1.2, 8, 20, 7)
    kps, desc, n_mono = ex.extract(img, lap)
    want = None
    if ref:
        lv = [ex.level_keypoints(l) for l in range(8)]
        rk, rd, rmono = ref.pack([k for k, _ in lv], [d for _, d in lv], ex.tables["scale"], lap, len(kps))
        want = [rk.view(np.uint8), rd, np.int32(rmono)]
    pin("pack", [kps.view(np.uint8), desc, np.int32(n_mono)], want)


def test_distance_and_three_maxima(oracle, ref, pin):
    rng = np.random.default_rng(3)
    d = rng.integers(0, 256, (400, 32), dtype=np.uint8)
    dist = []
    for i in range(0, 400, 2):
        assert oracle.hamming(d[i], d[i + 1], swar=True) == oracle.hamming(d[i], d[i + 1])
        dist.append(oracle.hamming(d[i], d[i + 1]))
    pin("distance", [np.array(dist, np.int32)], ref and [np.array([ref.descriptor_distance(d[i], d[i + 1]) for i in range(0, 400, 2)], np.int32)])
    got, want = [], []
    for _ in range(300):
        # bin = round(rot * 1/HISTO_LENGTH): only bins 0..12 of the 30 can fill (src/ORBmatcher1.cc:344-351); rot = 30 * bin
        counts = np.zeros(30, np.int64)
        counts[:12] = rng.integers(0, rng.choice([3, 12, 80]), 12)
        bins = np.repeat(np.arange(30), counts)
        keep = oracle.rotation_consistency(bins.astype(np.float32) * 30.0, np.zeros(len(bins), np.float32))
        got.append(keep)
        if ref:
            i1, i2, i3 = ref.three_maxima(counts)
            want.append(np.isin(bins, [i for i in (i1, i2, i3) if i >= 0]))
    pin("three_maxima", got, want if ref else None)


def bounds_grid(bounds):
    b = [np.float32(x) for x in bounds]
    return np.array(b + [np.float32(64) / (b[2] - b[0]), np.float32(48) / (b[3] - b[1])], np.float32)


def test_grid_and_area_match_reference(oracle, ref, pin):
    rng = np.random.default_rng(31)
    kp, desc, ur, occ, bounds = make_frame(rng, 2000)
    bg = bounds_grid(bounds)
    pin("grid", oracle.assign_features_to_grid(kp, bg), ref and ref.assign_features_to_grid(kp, bg))
    got, want = [], []
    for t in range(300):
        x, y = float(rng.uniform(-30, 780)), float(rng.uniform(-30, 510))
        r = float(rng.choice([2.5, 4.0, 10.0, 30.0, 80.0, 900.0]))
        lv = int(rng.integers(0, 8))
        mn, mx = [(-1, -1), (lv, -1), (0, lv), (lv - 1, lv + 1), (lv - 1, lv)][t % 5]
        got.append(oracle.get_features_in_area(kp, bg, x, y, r, mn, mx))
        if ref:
            want.append(ref.get_features_in_area(kp, bg, x, y, r, mn, mx))
    pin("area", got, want if ref else None)


@pytest.mark.parametrize("seed,n,n_pts,th,crowd,dup", [(41, 1000, 1500, 1.0, 0, 0.3), (42, 800, 2000, 5.0, 10, 0.7), (43, 60, 400, 8.0, 2, 0.9),
                                                      (44, 1200, 1200, 3.0, 0, 0.5)])
def test_search_by_projection_map_matches_reference(oracle, ref, pin, seed, n, n_pts, th, crowd, dup):
    rng = np.random.default_rng(seed)
    kp, desc, ur, occ, bounds = make_frame(rng, n, crowd=crowd)
    bg = bounds_grid(bounds)
    P = make_points(rng, kp, desc, ur, n_pts, dup_frac=dup, max_flip=100)
    for far, ratio in ((False, 0.8), (True, 0.6)):
        a = (kp, desc, ur, occ, bg, SCALE, P["in_view"], P["bad"], P["x"], P["y"], P["xr"], P["view_cos"], P["depth"], P["level"], P["n_obs"],
             P["desc"])
        got, nm = oracle.search_by_projection_map(*a, th=th, far=far, th_far=20.0, nnratio=ratio)
        want = ref and ref.search_by_projection_map(*a, th=th, far=far, th_far=20.0, nnratio=ratio)
        assert nm > 10
        pin("far=%d" % far, [got, np.int32(nm)], want and [want[0], np.int32(want[1])])


@pytest.mark.parametrize("seed,n,n_last,th,crowd,tz,mono", [(51, 1200, 1200, 15.0, 0, 0.0, False), (52, 1000, 1500, 30.0, 8, 0.0, False),
                                                           (53, 1000, 1000, 15.0, 0, 2.0, False), (54, 1000, 1000, 15.0, 0, -2.0, False),
                                                           (55, 800, 900, 7.0, 0, 2.0, True)])
def test_search_by_projection_last_matches_reference(oracle, ref, pin, seed, n, n_last, th, crowd, tz, mono):
    rng = np.random.default_rng(seed)
    kp, desc, ur, occ, bounds = make_frame(rng, n, crowd=crowd)
    if mono:
        ur = None
    bg = bounds_grid(bounds)
    P = make_points(rng, kp, desc, np.full(n, -1.0, np.float32) if ur is None else ur, n_last, dup_frac=0.4, jitter=4.0)
    z = np.where(rng.random(n_last) < 0.03, -5.0, P["depth"]).astype(np.float32)
    invz = ref_lib.invz(z)
    for ori in (True, False):
        want = None
        if ref:
            rm, rnm, rinvz = ref.search_by_projection_last(kp, desc, ur, occ, bg, SCALE, 40.0, P["valid"], P["x"], P["y"], z, P["level"],
                                                           P["angle"], P["n_obs"], P["desc"], th, last_tz=tz, mono=mono, check_ori=ori)
            assert rinvz.tobytes() == invz.tobytes()
            want = [rm, np.int32(rnm)]
        # bForward = tlc(2) > mb && !bMono with tlc = Tlw * twc = (0, 0, tz), mb = 1 (src/ORBmatcher3.cc:269-273)
        fwd = (tz > 1.0) and not mono; bwd = (-tz > 1.0) and not mono
        got, nm = oracle.search_by_projection_last(kp, desc, ur, occ, bg, SCALE, 40.0, P["valid"], P["x"], P["y"], invz, P["level"], P["angle"],
                                                   P["n_obs"], P["desc"], th, fwd, bwd, ori)
        assert nm > 10
        pin("ori=%d" % ori, [got, np.int32(nm)], want)


@pytest.mark.parametrize("seed,n,n_kf,th,orb_dist", [(61, 1000, 800, 10.0, 100), (62, 1000, 800, 3.0, 64), (63, 200, 2000, 10.0, 100)])
def test_search_by_projection_kf_matches_reference(oracle, ref, pin, seed, n, n_kf, th, orb_dist):
    rng = np.random.default_rng(seed)
    kp, desc, ur, occ, bounds = make_frame(rng, n, occupied_frac=0.4)
    bg = bounds_grid(bounds)
    P = make_points(rng, kp, desc, ur, n_kf, dup_frac=0.4)
    found = (rng.random(n_kf) < 0.1).astype(np.uint8)
    z = P["depth"]
    d3 = ref_lib.dist3d(P["x"], P["y"], z)
    for ori in (True, False):
        want = None
        if ref:
            rm, rnm, rd3 = ref.search_by_projection_kf(kp, desc, occ, bg, SCALE, P["valid"], found, P["x"], P["y"], z, P["min_dist"] * 30,
                                                       P["max_dist"] * 30, P["level"], P["angle"], P["desc"], th, orb_dist, ori)
            assert rd3.tobytes() == d3.tobytes()
            want = [rm, np.int32(rnm)]
        valid = P["valid"] & (1 - found)
        got, nm = oracle.search_by_projection_kf(kp, desc, occ, bg, SCALE, valid, P["x"], P["y"], d3, P["min_dist"] * 30, P["max_dist"] * 30,
                                                 P["level"], P["angle"], P["desc"], th, orb_dist, ori)
        pin("ori=%d" % ori, [got, np.int32(nm)], want)
    assert nm > 10


@pytest.mark.parametrize("cols,rows,nfeatures,seed", [(752, 480, 1200, 31), (1241, 376, 2000, 32), (400, 300, 500, 33)])
def test_compute_stereo_matches_matches_reference(oracle, ref, pin, cols, rows, nfeatures, seed):
    """Frame::ComputeStereoMatches (src/Frame.cc:841-1011) on a synthetic pair extracted by the oracle."""
    left = synth.image(seed, cols, rows, view=0); right = synth.image(seed, cols, rows, view=1)
    oL = oracle.extractor(nfeatures, 1.2, 8, 20, 7); oR = oracle.extractor(nfeatures, 1.2, 8, 20, 7)
    kL, dL, _ = oL.extract(left, (0, 0)); kR, dR, _ = oR.extract(right, (0, 0))
    pyrL = [oL.pyramid_level(l, with_border=True) for l in range(8)]; pyrR = [oR.pyramid_level(l, with_border=True) for l in range(8)]
    mbf, mb = np.float32(47.9), np.float32(0.11)
    max_d = np.float32(mbf / mb)                              # src/Frame.cc:873: maxD = mbf / minZ, minZ = mb
    ou, od, kept = oracle.stereo_match_raw(kL, dL, kR, dR, pyrL, pyrR, oL.tables["scale"], oL.tables["inv"], mbf, max_d)
    want = ref and ref.compute_stereo_matches(kL, dL, kR, dR, pyrL, pyrR, oL.tables["scale"], oL.tables["inv"], mb, mbf)
    assert kept > 30 and (ou >= 0).sum() == kept
    pin("stereo", [ou.view(np.uint32), od.view(np.uint32)], want and [w.view(np.uint32) for w in want])


@pytest.mark.parametrize("nleft,check_ori,ratio,seed", [(-1, True, 0.6, 71), (-1, False, 0.9, 72), (120, True, 0.75, 73), (-1, True, 0.75, 74)])
def test_search_by_bow_kf_frame_matches_reference(oracle, ref, pin, nleft, check_ori, ratio, seed):
    k, L = 4, 3
    parent, desc, weights = bow_synth.make_vocab(seed, k, L)
    voc = oracle.vocabulary(parent, desc, weights, k, L)
    P = bow_synth.make_pair(seed + 100, desc, parent, 600, 560)
    _, fva = voc.transform(P["desc_a"], 2); _, fvb = voc.transform(P["desc_b"], 2)
    a = (P["desc_a"], P["angle_a"], P["valid_a"], fva, P["desc_b"], P["angle_b"], fvb, nleft, ratio, check_ori)
    got, nm = oracle.search_by_bow_kf_frame(*a)
    want = ref and ref.search_by_bow_kf_frame(*a)
    assert nm > 20
    pin("bow", [got, np.int32(nm)], want and [want[0], np.int32(want[1])])


@pytest.mark.parametrize("check_ori,ratio,seed", [(True, 0.6, 81), (False, 0.9, 82), (True, 0.8, 83)])
def test_search_by_bow_kf_kf_matches_reference(oracle, ref, pin, check_ori, ratio, seed):
    k, L = 4, 3
    parent, desc, weights = bow_synth.make_vocab(seed, k, L)
    voc = oracle.vocabulary(parent, desc, weights, k, L)
    P = bow_synth.make_pair(seed + 100, desc, parent, 600, 560)
    _, fva = voc.transform(P["desc_a"], 2); _, fvb = voc.transform(P["desc_b"], 2)
    a = (P["desc_a"], P["angle_a"], P["valid_a"], fva, P["desc_b"], P["angle_b"], P["valid_b"], fvb, ratio, check_ori)
    got, nm = oracle.search_by_bow_kf_kf(*a)
    want = ref and ref.search_by_bow_kf_kf(*a)
    assert nm > 20
    pin("bow", [got, np.int32(nm)], want and [want[0], np.int32(want[1])])


@pytest.mark.parametrize("only_stereo,coarse,check_ori,seed", [(False, False, True, 91), (True, False, True, 92), (False, True, True, 93),
                                                               (False, False, False, 94)])
def test_search_for_triangulation_matches_reference(oracle, ref, pin, only_stereo, coarse, check_ori, seed):
    """ORBmatcher::SearchForTriangulation + the line test of Pinhole::epipolarConstrain (F12 and the epipole supplied)."""
    from tests import test_bow_cpu
    k, L = 4, 3
    parent, desc, weights = bow_synth.make_vocab(seed, k, L)
    voc = oracle.vocabulary(parent, desc, weights, k, L)
    P = bow_synth.make_pair(seed + 100, desc, parent, 900, 900)
    _, fva = voc.transform(P["desc_a"], 2); _, fvb = voc.transform(P["desc_b"], 2)
    kpa, kpb, F, ep, scale, sigma2, fa, fb, sa, sb = test_bow_cpu.tri_inputs(P, seed)
    a = (kpa, P["desc_a"], fa, sa, fva, kpb, P["desc_b"], fb, sb, fvb, F, ep, scale, sigma2, only_stereo, coarse, check_ori)
    got, nm = oracle.search_for_triangulation(*a)
    want = ref and ref.search_for_triangulation(*a)
    assert nm > (3 if not coarse else 30)
    pin("triangulation", [got, np.int32(nm)], want and [want[0], np.int32(want[1])])


def test_distinctive_descriptor_matches_reference(oracle, ref, pin):
    rng = np.random.default_rng(17)
    got, want = [], []
    for n in [1, 2, 3, 4, 7, 20, 61, 150]:
        for _ in range(20):
            base = rng.integers(0, 256, 32, dtype=np.uint8)
            d = np.stack([base ^ (rng.integers(0, 256, 32, dtype=np.uint8) & rng.integers(0, 256, 32, dtype=np.uint8) & rng.integers(0, 256, 32, dtype=np.uint8))
                          for _ in range(n)])
            if n > 3:
                d[n - 1] = d[0]                      # duplicates: equal medians, the first index must win
            got.append(oracle.distinctive_descriptor(d))
            if ref:
                want.append(ref.distinctive_descriptor(d))
    pin("distinctive", [np.array(got, np.int32)], ref and [np.array(want, np.int32)])


@pytest.mark.parametrize("k,L,levelsup,weighting,seed", [(10, 4, 4, 0, 5), (10, 4, 2, 0, 6), (4, 3, 1, 1, 7), (3, 6, 4, 2, 8), (5, 3, 2, 3, 9)])
def test_dbow2_transform_and_score_match_reference(oracle, ref, pin, tmp_path, k, L, levelsup, weighting, seed):
    """DBoW2's own loadFromTextFile / transform / L1 score on a synthetic ORBvoc-format file (written without a trailing newline:
    loadFromTextFile's `while(!f.eof())` loop turns a trailing empty line into a bogus root child with an uninitialised
    descriptor — undefined behaviour that the product loader does not reproduce, it skips the empty line)."""
    parent, desc, weights = bow_synth.make_vocab(seed, k, L)
    path = tmp_path / "voc.txt"
    bow_synth.write_vocab_text(path, parent, desc, weights, k, L, 0, weighting)
    txt = open(path).read().rstrip("\n")
    open(path, "w").write(txt)
    rv = ref and ref_lib.RefVocabulary(ref, path)
    ov = oracle.vocabulary(parent, desc, weights, k, L, 0, weighting)
    if rv:
        assert rv.info()["n_nodes"] == len(parent) and rv.info()["k"] == k and rv.info()["L"] == L
    feats = bow_synth.make_features(seed + 50, desc, parent, 1500)
    pin("transform_features", ov.transform_features(feats, levelsup), rv and rv.transform_features(feats, levelsup))
    (oid, oval), ofv = ov.transform(feats, levelsup)
    other = ov.transform(bow_synth.make_features(seed + 51, desc, parent, 1200), levelsup)[0]
    got = [oid, oval.view(np.uint64), *ofv, np.float64(oracle.bow_score_l1((oid, oval), other)).view(np.uint64)]   # identical doubles
    want = None
    if rv:
        (rid, rval), rfv = rv.transform(feats, levelsup)
        want = [rid, rval.view(np.uint64), *rfv, np.float64(rv.score((rid, rval), other)).view(np.uint64)]
    pin("transform_score", got, want)
