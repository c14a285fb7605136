"""Python mirror of the bag-of-words side of the reference over the C ABI: DBoW2::TemplatedVocabulary (ORBVocabulary,
reference include/ORBVocabulary.h, Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h), Frame::ComputeBoW (src/Frame.cc:768-775)
and the vocabulary-guided searches of ORBmatcher (src/ORBmatcher1.cc:225-427, src/ORBmatcher2.cc:36-471)."""
import ctypes as C

import numpy as np

from .capi import BowViewC, FeatureVectorC, KP_DTYPE, TriangulationViewC, check, lib, ptr

TF_IDF, TF, IDF, BINARY = 0, 1, 2, 3
L1_NORM, L2_NORM, CHI_SQUARE, KL, BHATTACHARYYA, DOT_PRODUCT = 0, 1, 2, 3, 4, 5


class FeatureVector:
    """DBoW2::FeatureVector (std::map<NodeId, std::vector<unsigned>>) in CSR form, node ids ascending."""

    def __init__(self, node_ids, offsets, indices):
        self.node_ids = np.ascontiguousarray(node_ids, np.uint32)
        self.offsets = np.ascontiguousarray(offsets, np.int32)
        self.indices = np.ascontiguousarray(indices, np.uint32)
        assert len(self.offsets) == len(self.node_ids) + 1

    def c_struct(self):
        return FeatureVectorC(len(self.node_ids), ptr(self.node_ids), ptr(self.offsets), ptr(self.indices))

    def as_dict(self):
        return {int(n): self.indices[self.offsets[i]:self.offsets[i + 1]].tolist() for i, n in enumerate(self.node_ids)}


class ORBVocabulary:
    """k-ary vocabulary tree of 256-bit descriptors with a device copy; `transform` runs the descent on the GPU."""

    def __init__(self, parent, descriptors, weights, k, L, scoring=L1_NORM, weighting=TF_IDF, device=0):
        parent = np.ascontiguousarray(parent, np.int32)
        descriptors = np.ascontiguousarray(descriptors, np.uint8).reshape(-1, 32)
        weights = np.ascontiguousarray(weights, np.float64)
        assert len(parent) == len(descriptors) == len(weights)
        h = C.c_void_p()
        check(lib().orbx_vocab_create(device, len(parent), ptr(parent), ptr(descriptors), ptr(weights), k, L, scoring, weighting,
                                      C.byref(h)))
        self._h = h
        self.k, self.L = k, L

    @classmethod
    def loadFromTextFile(cls, path, device=0):
        """TemplatedVocabulary::loadFromTextFile (the ORBvoc.txt format)."""
        self = cls.__new__(cls)
        h = C.c_void_p()
        check(lib().orbx_vocab_load_text(device, str(path).encode(), C.byref(h)))
        self._h = h
        info = self.info()
        self.k, self.L = info["k"], info["L"]
        return self

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                lib().orbx_vocab_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def info(self):
        v = [C.c_int(0) for _ in range(4)]
        check(lib().orbx_vocab_info(self._h, *[C.byref(x) for x in v]))
        return dict(n_nodes=v[0].value, n_words=v[1].value, k=v[2].value, L=v[3].value)

    def transform_features(self, descriptors, levelsup=4):
        """Per-feature (word id, weight, node id at level L - levelsup)."""
        d = np.ascontiguousarray(descriptors, np.uint8).reshape(-1, 32)
        n = len(d)
        word = np.zeros(n, np.uint32); weight = np.zeros(n, np.float64); node = np.zeros(n, np.uint32)
        check(lib().orbx_bow_transform(self._h, ptr(d), n, levelsup, ptr(word), ptr(weight), ptr(node)))
        return word, weight, node

    def transform(self, descriptors, levelsup=4):
        """transform(features, BowVector, FeatureVector, levelsup): returns ((word ids, values), FeatureVector)."""
        d = np.ascontiguousarray(descriptors, np.uint8).reshape(-1, 32)
        n = len(d)
        ids = np.zeros(max(n, 1), np.uint32); vals = np.zeros(max(n, 1), np.float64)
        nodes = np.zeros(max(n, 1), np.uint32); offs = np.zeros(n + 1, np.int32); idx = np.zeros(max(n, 1), np.uint32)
        nb = C.c_int(0); nf = C.c_int(0)
        check(lib().orbx_compute_bow(self._h, ptr(d), n, levelsup, ptr(ids), ptr(vals), C.byref(nb), ptr(nodes), ptr(offs), ptr(idx),
                                     C.byref(nf)))
        fv = FeatureVector(nodes[:nf.value].copy(), offs[:nf.value + 1].copy(), idx[:offs[nf.value]].copy())
        return (ids[:nb.value].copy(), vals[:nb.value].copy()), fv

    def score(self, bow_a, bow_b):
        ia = np.ascontiguousarray(bow_a[0], np.uint32); va = np.ascontiguousarray(bow_a[1], np.float64)
        ib = np.ascontiguousarray(bow_b[0], np.uint32); vb = np.ascontiguousarray(bow_b[1], np.float64)
        s = C.c_double(0)
        check(lib().orbx_bow_score(self._h, ptr(ia), ptr(va), len(ia), ptr(ib), ptr(vb), len(ib), C.byref(s)))
        return s.value


def search_by_bow(desc_a, angle_a, valid_a, fv_a, desc_b, angle_b, fv_b, valid_b=None, kf_kf=False, nleft_b=-1, nnratio=0.6,
                  check_orientation=True, device=0):
    """ORBmatcher::SearchByBoW: (KF, Frame) when kf_kf is False — returns (match_b, match_a, nmatches) with match_b the
    reference's vpMapPointMatches expressed as KF feature indices; (KF1, KF2) when kf_kf is True — match_a is vpMatches12
    expressed as KF2 feature indices."""
    da = np.ascontiguousarray(desc_a, np.uint8).reshape(-1, 32); db = np.ascontiguousarray(desc_b, np.uint8).reshape(-1, 32)
    aa = np.ascontiguousarray(angle_a, np.float32); ab = np.ascontiguousarray(angle_b, np.float32)
    va = np.ascontiguousarray(valid_a, np.uint8)
    vb = np.ascontiguousarray(valid_b, np.uint8) if valid_b is not None else None
    ma = np.full(len(da), -1, np.int32); mb = np.full(len(db), -1, np.int32)
    nm = C.c_int(0)
    fa, fb = fv_a.c_struct(), fv_b.c_struct()
    check(lib().orbx_search_by_bow(device, 1 if kf_kf else 0, ptr(da), ptr(aa), ptr(va), len(da), C.addressof(fa), ptr(db), ptr(ab),
                                   ptr(vb), len(db), C.addressof(fb), nleft_b, float(nnratio), int(check_orientation), ptr(ma), ptr(mb),
                                   C.byref(nm)))
    return mb, ma, nm.value


def search_by_bow_batch(desc, angle, valid, fv, kfs, kf_kf=False, nleft=-1, nnratio=0.6, check_orientation=True, device=0):
    """ORBmatcher::SearchByBoW of one fixed side against many key frames in one call (orbx_search_by_bow_batch).  `kfs` is a
    sequence of dicts with desc, angle, valid and fv.  kf_kf False (Tracking::Relocalization): the fixed side is the Frame
    (`valid` may be None) and each entry a candidate key frame; match[k, j] = feature of kfs[k] whose map point the Frame's
    feature j received.  kf_kf True (LoopClosing::DetectCommonRegionsFromBoW): the fixed side is KF1 and each entry a KF2;
    match[k, i] = feature of kfs[k] matched to KF1's feature i.  Returns (match [n_kf, n], nmatches [n_kf]); row k equals
    search_by_bow on kfs[k]."""
    d = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
    a = np.ascontiguousarray(angle, np.float32)
    v = np.ascontiguousarray(valid, np.uint8) if valid is not None else None
    n_kf = len(kfs)
    keep = []                                  # the arrays the views point into stay alive for the call
    views = (BowViewC * max(n_kf, 1))()
    for k, kf in enumerate(kfs):
        dk = np.ascontiguousarray(kf["desc"], np.uint8).reshape(-1, 32)
        ak = np.ascontiguousarray(kf["angle"], np.float32) if kf["angle"] is not None else None
        vk = np.ascontiguousarray(kf["valid"], np.uint8)
        keep += [dk, ak, vk, kf["fv"]]
        w = views[k]
        w.n = len(dk); w.desc = ptr(dk); w.angle = ptr(ak); w.valid = ptr(vk); w.fv = kf["fv"].c_struct()
    match = np.full((n_kf, len(d)), -1, np.int32)
    nm = np.zeros(n_kf, np.int32)
    f = fv.c_struct()
    check(lib().orbx_search_by_bow_batch(device, 1 if kf_kf else 0, ptr(d), ptr(a), ptr(v), len(d), C.addressof(f), nleft, n_kf,
                                         C.addressof(views), float(nnratio), int(check_orientation), ptr(match), ptr(nm)))
    return match, nm


def search_for_triangulation(kp_a, desc_a, free_a, stereo_a, fv_a, kp_b, desc_b, free_b, stereo_b, fv_b, F12, ep, scale_b, sigma2_b,
                             only_stereo=False, coarse=False, check_orientation=True, device=0):
    """ORBmatcher::SearchForTriangulation (single pinhole camera): returns (vMatches12 as KF2 indices, nmatches)."""
    ka = np.ascontiguousarray(kp_a, KP_DTYPE); kb = np.ascontiguousarray(kp_b, KP_DTYPE)
    da = np.ascontiguousarray(desc_a, np.uint8).reshape(-1, 32); db = np.ascontiguousarray(desc_b, np.uint8).reshape(-1, 32)
    fra = np.ascontiguousarray(free_a, np.uint8); frb = np.ascontiguousarray(free_b, np.uint8)
    sa = np.ascontiguousarray(stereo_a, np.uint8); sb = np.ascontiguousarray(stereo_b, np.uint8)
    F = np.ascontiguousarray(F12, np.float32).reshape(9); e = np.ascontiguousarray(ep, np.float32)
    sc = np.ascontiguousarray(scale_b, np.float32); sg = np.ascontiguousarray(sigma2_b, np.float32)
    ma = np.full(len(ka), -1, np.int32)
    nm = C.c_int(0)
    fa, fb = fv_a.c_struct(), fv_b.c_struct()
    check(lib().orbx_search_for_triangulation(device, ptr(ka), ptr(da), ptr(fra), ptr(sa), len(ka), C.addressof(fa), ptr(kb), ptr(db),
                                              ptr(frb), ptr(sb), len(kb), C.addressof(fb), ptr(F), ptr(e), ptr(sc), ptr(sg), len(sc),
                                              int(only_stereo), int(coarse), int(check_orientation), ptr(ma), C.byref(nm)))
    return ma, nm.value


def search_for_triangulation_batch(kp_a, desc_a, free_a, stereo_a, fv_a, neighbours, only_stereo=False, check_orientation=True,
                                   device=0):
    """ORBmatcher::SearchForTriangulation of KF1 against many neighbours in one call (orbx_search_for_triangulation_batch).
    `neighbours` is a sequence of dicts with the KF2 arguments of search_for_triangulation: kp, desc, free, stereo, fv, F12, ep,
    scale, sigma2 and optionally coarse (default False).  Returns (match [n_kf, n_a] as KF2 indices, nmatches [n_kf]); row k
    equals search_for_triangulation(KF1, neighbour k, ...)."""
    ka = np.ascontiguousarray(kp_a, KP_DTYPE)
    da = np.ascontiguousarray(desc_a, np.uint8).reshape(-1, 32)
    fra = np.ascontiguousarray(free_a, np.uint8); sa = np.ascontiguousarray(stereo_a, np.uint8)
    n_kf = len(neighbours)
    keep = []                                  # the arrays the views point into stay alive for the call
    views = (TriangulationViewC * max(n_kf, 1))()
    for k, nb in enumerate(neighbours):
        kb = np.ascontiguousarray(nb["kp"], KP_DTYPE); db = np.ascontiguousarray(nb["desc"], np.uint8).reshape(-1, 32)
        frb = np.ascontiguousarray(nb["free"], np.uint8); sb = np.ascontiguousarray(nb["stereo"], np.uint8)
        sc = np.ascontiguousarray(nb["scale"], np.float32); sg = np.ascontiguousarray(nb["sigma2"], np.float32)
        keep += [kb, db, frb, sb, sc, sg, nb["fv"]]
        v = views[k]
        v.n = len(kb); v.kp = ptr(kb); v.desc = ptr(db); v.free = ptr(frb); v.stereo = ptr(sb); v.fv = nb["fv"].c_struct()
        v.F12[:] = [float(x) for x in np.asarray(nb["F12"], np.float32).reshape(9)]
        v.ep[:] = [float(x) for x in np.asarray(nb["ep"], np.float32).reshape(2)]
        v.scale = ptr(sc); v.sigma2 = ptr(sg); v.n_levels = len(sc); v.coarse = int(bool(nb.get("coarse", False)))
    match = np.full((n_kf, len(ka)), -1, np.int32)
    nm = np.zeros(n_kf, np.int32)
    fa = fv_a.c_struct()
    check(lib().orbx_search_for_triangulation_batch(device, ptr(ka), ptr(da), ptr(fra), ptr(sa), len(ka), C.addressof(fa), n_kf,
                                                    C.addressof(views), int(only_stereo), int(check_orientation), ptr(match), ptr(nm)))
    return match, nm
