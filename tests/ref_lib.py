"""ctypes binding of oracle/_ref/libref.so — the REFERENCE's own functions of the hot path, compiled by oracle/build_ref.sh from
the reference checkout named by ORB_REFERENCE_ROOT — and Pin, which compares with the reference's answers: live when the library
is built, else with the CRCs of those answers stored in tests/golden/ref_pin_golden.json.  TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import json
import os
import subprocess
import zlib

import numpy as np

from tests.oracle_lib import KP_DTYPE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(ROOT, "oracle", "_ref", "libref.so")
_vp, _i, _f, _sz = C.c_void_p, C.c_int, C.c_float, C.c_size_t


def _p(a):
    return None if a is None else a.ctypes.data_as(_vp)


def available():
    if not os.path.exists(SO) and os.path.isdir(os.path.join(os.environ.get("ORB_REFERENCE_ROOT", ""), "src")):
        subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle")])
        subprocess.check_call(["sh", os.path.join(ROOT, "oracle", "build_ref.sh")])
    return os.path.exists(SO)


GOLDEN = os.path.join(ROOT, "tests", "golden", "ref_pin_golden.json")
_golden = None


def crc(arrays):
    c = 0
    for a in arrays:
        c = zlib.crc32(np.ascontiguousarray(a).tobytes(), c)
    return c & 0xFFFFFFFF


class Pin:
    """pin(part, got, want): `got` is a list of arrays computed by the oracle or the CUDA path, `want` the same list from the
    reference library, or None when libref.so is not built.  With `want`, every array must equal its counterpart (shape and
    values); without it, the CRC of `got` must equal the CRC stored for this test and part, which is the CRC of the
    reference's answer.  With ORBX_REF_PIN_RECORD=<file> set, each live comparison that passes records that CRC there (how
    tests/golden/ref_pin_golden.json is regenerated where the reference is built)."""

    def __init__(self, test_name):
        self.test_name = test_name

    def __call__(self, part, got, want):
        global _golden
        key = self.test_name + ":" + part
        got = [np.ascontiguousarray(a) for a in got]
        if want is None:
            if _golden is None:
                with open(GOLDEN) as f:
                    _golden = json.load(f)["crc32"]
            assert key in _golden, "no stored reference answer for " + key
            assert crc(got) == _golden[key], "differs from the reference's stored answer: " + key
            return
        assert len(got) == len(want), key
        for i, (a, b) in enumerate(zip(got, want)):
            b = np.ascontiguousarray(b)
            assert a.shape == b.shape and np.array_equal(a, b), (key, i)
        path = os.environ.get("ORBX_REF_PIN_RECORD")
        if path:
            rec = json.load(open(path)) if os.path.exists(path) else {}
            rec[key] = crc(got)
            with open(path, "w") as f:
                json.dump(rec, f, indent=1, sort_keys=True)


def invz(z):
    """1.0 / z as refc_search_by_projection_last hands it to the compared side (double division, stored as float)."""
    return (1.0 / np.asarray(z, np.float64)).astype(np.float32)


def dist3d(u, v, z):
    """|(u, v, z)| as refc_search_by_projection_kf hands it to the compared side (float, left-to-right, no contraction)."""
    u, v, z = (np.asarray(a, np.float32) for a in (u, v, z))
    return np.sqrt(u * u + v * v + z * z).astype(np.float32)


class Ref:
    def __init__(self):
        from tests import oracle_lib
        oracle_lib.load()                      # libref.so links against liborb_oracle.so (cv::FAST stand-in)
        self.lib = C.CDLL(SO)

    def tables(self, nfeatures, scale_factor, nlevels):
        sc = np.zeros(nlevels, np.float32); inv = sc.copy(); s2 = sc.copy(); is2 = sc.copy()
        nf = np.zeros(nlevels, np.int32); umax = np.zeros(16, np.int32); pat = np.zeros(1024, np.int32)
        self.lib.refc_tables(nfeatures, _f(scale_factor), nlevels, _p(sc), _p(inv), _p(s2), _p(is2), _p(nf), _p(umax), _p(pat))
        return dict(scale=sc, inv=inv, sigma2=s2, invsigma2=is2, nfeat=nf, umax=umax, pattern=pat)

    def distribute_octree(self, xs, ys, sc, min_x, max_x, min_y, max_y, N, level=0):
        xs = np.ascontiguousarray(xs, np.int32); ys = np.ascontiguousarray(ys, np.int32); sc = np.ascontiguousarray(sc, np.int32)
        cap = len(xs) + 8
        ox = np.zeros(cap, np.int32); oy = np.zeros(cap, np.int32); os_ = np.zeros(cap, np.int32)
        m = self.lib.refc_distribute_octree(_p(xs), _p(ys), _p(sc), len(xs), min_x, max_x, min_y, max_y, N, level, _p(ox), _p(oy), _p(os_), cap)
        return ox[:m].copy(), oy[:m].copy(), os_[:m].copy()

    def tile_calc_keypoints(self, img, nfeatures=1000, ini_th=20, min_th=7):
        img = np.ascontiguousarray(img, np.uint8)
        cap = img.size
        xs = np.zeros(cap, np.int32); ys = np.zeros(cap, np.int32); sc = np.zeros(cap, np.int32)
        n = self.lib.refc_tile_calc_keypoints(_p(img), img.shape[1], img.shape[0], _sz(img.strides[0]), nfeatures, ini_th, min_th, _p(xs),
                                              _p(ys), _p(sc), cap)
        return xs[:n].copy(), ys[:n].copy(), sc[:n].copy()

    def descriptor(self, blurred, x, y, angle_deg):
        blurred = np.ascontiguousarray(blurred, np.uint8)
        out = np.zeros(32, np.uint8)
        self.lib.refc_descriptor(_p(blurred), blurred.shape[1], blurred.shape[0], _sz(blurred.strides[0]), _f(x), _f(y), _f(angle_deg), _p(out))
        return out

    def pack(self, level_kps, level_desc, scale, lap, nkeypoints):
        """ORBextractor::operator()'s placement loop over all levels; level_kps[l] in level coordinates."""
        out_k = np.zeros(nkeypoints, KP_DTYPE); out_d = np.zeros((nkeypoints, 32), np.uint8)
        mono = C.c_int(0); stereo = C.c_int(nkeypoints - 1)
        for l, (k, d) in enumerate(zip(level_kps, level_desc)):
            if len(k) == 0:
                continue
            k = np.ascontiguousarray(k, KP_DTYPE).copy(); d = np.ascontiguousarray(d, np.uint8)
            self.lib.refc_pack_level(_p(k), _p(d), len(k), l, _f(scale[l]), int(lap[0]), int(lap[1]), _p(out_k), _p(out_d), nkeypoints,
                                     C.byref(mono), C.byref(stereo))
        return out_k, out_d, mono.value

    def descriptor_distance(self, a, b):
        a = np.ascontiguousarray(a, np.uint8); b = np.ascontiguousarray(b, np.uint8)
        return self.lib.refc_descriptor_distance(_p(a), _p(b))

    def distinctive_descriptor(self, desc):
        desc = np.ascontiguousarray(desc, np.uint8)
        return self.lib.refc_distinctive_descriptor(_p(desc), len(desc))

    def three_maxima(self, counts):
        c = np.ascontiguousarray(counts, np.int32); ind = np.zeros(3, np.int32)
        self.lib.refc_three_maxima(_p(c), len(c), _p(ind))
        return tuple(int(v) for v in ind)

    def assign_features_to_grid(self, kp, bounds_grid):
        kp = np.ascontiguousarray(kp, KP_DTYPE); bg = np.ascontiguousarray(bounds_grid, np.float32)
        cs = np.zeros(64 * 48 + 1, np.int32); items = np.zeros(max(len(kp), 1), np.int32)
        self.lib.refc_assign_features_to_grid(_p(kp), len(kp), _p(bg), _p(cs), _p(items))
        return cs, items[:cs[-1]]

    def get_features_in_area(self, kp, bounds_grid, x, y, r, min_level=-1, max_level=-1):
        kp = np.ascontiguousarray(kp, KP_DTYPE); bg = np.ascontiguousarray(bounds_grid, np.float32)
        out = np.zeros(max(len(kp), 1), np.int32)
        n = self.lib.refc_get_features_in_area(_p(kp), len(kp), _p(bg), _f(x), _f(y), _f(r), int(min_level), int(max_level), _p(out))
        return out[:n]

    def search_by_projection_map(self, kp, desc, uright, occupied, bounds_grid, scale, in_view, bad, projx, projy, projxr, viewcos, depth,
                                 level, nobs, mpdesc, th=1.0, far=False, th_far=0.0, nnratio=0.8):
        kp = np.ascontiguousarray(kp, KP_DTYPE); desc = np.ascontiguousarray(desc, np.uint8)
        ur = None if uright is None else np.ascontiguousarray(uright, np.float32)
        oc = None if occupied is None else np.ascontiguousarray(occupied, np.uint8)
        bg = np.ascontiguousarray(bounds_grid, np.float32); sc = np.ascontiguousarray(scale, np.float32)
        f32 = lambda a: np.ascontiguousarray(a, np.float32)   # noqa: E731
        iv = np.ascontiguousarray(in_view, np.uint8); bd = np.ascontiguousarray(bad, np.uint8)
        px, py, pxr, vc, dp = f32(projx), f32(projy), f32(projxr), f32(viewcos), f32(depth)
        lv = np.ascontiguousarray(level, np.int32); no = np.ascontiguousarray(nobs, np.int32); md = np.ascontiguousarray(mpdesc, np.uint8)
        out = np.full(max(len(kp), 1), -1, np.int32)
        nm = self.lib.refc_search_by_projection_map(_p(kp), _p(desc), _p(ur), _p(oc), len(kp), _p(bg), _p(sc), len(sc), _p(iv), _p(bd), _p(px),
                                                    _p(py), _p(pxr), _p(vc), _p(dp), _p(lv), _p(no), _p(md), len(iv), _f(th), int(far), _f(th_far),
                                                    _f(nnratio), _p(out))
        return out[:len(kp)], nm

    def search_by_projection_last(self, kp, desc, uright, occupied, bounds_grid, scale, mbf, valid, u, v, z, octave, angle, nobs, mpdesc, th,
                                  last_tz=0.0, mono=False, check_ori=True):
        """Returns (match_f, nmatches, invz) — invz is what the reference computed as 1.0 / x3Dc(2), for the oracle's input."""
        kp = np.ascontiguousarray(kp, KP_DTYPE); desc = np.ascontiguousarray(desc, np.uint8)
        ur = None if uright is None else np.ascontiguousarray(uright, np.float32)
        oc = None if occupied is None else np.ascontiguousarray(occupied, np.uint8)
        bg = np.ascontiguousarray(bounds_grid, np.float32); sc = np.ascontiguousarray(scale, np.float32)
        f32 = lambda a: np.ascontiguousarray(a, np.float32)   # noqa: E731
        va = np.ascontiguousarray(valid, np.uint8); uu, vv, zz, an = f32(u), f32(v), f32(z), f32(angle)
        oct_ = np.ascontiguousarray(octave, np.int32); no = np.ascontiguousarray(nobs, np.int32); md = np.ascontiguousarray(mpdesc, np.uint8)
        out = np.full(max(len(kp), 1), -1, np.int32); invz = np.zeros(len(va), np.float32)
        nm = self.lib.refc_search_by_projection_last(_p(kp), _p(desc), _p(ur), _p(oc), len(kp), _p(bg), _p(sc), len(sc), _f(mbf), _p(va), _p(uu),
                                                     _p(vv), _p(zz), _p(oct_), _p(an), _p(no), _p(md), len(va), _f(th), _f(last_tz), int(mono),
                                                     int(check_ori), _p(invz), _p(out))
        return out[:len(kp)], nm, invz

    def search_by_projection_kf(self, kp, desc, occupied, bounds_grid, scale, valid, found, u, v, z, mind, maxd, level, angle, mpdesc, th,
                                orb_dist, check_ori=True):
        kp = np.ascontiguousarray(kp, KP_DTYPE); desc = np.ascontiguousarray(desc, np.uint8)
        oc = None if occupied is None else np.ascontiguousarray(occupied, np.uint8)
        bg = np.ascontiguousarray(bounds_grid, np.float32); sc = np.ascontiguousarray(scale, np.float32)
        f32 = lambda a: np.ascontiguousarray(a, np.float32)   # noqa: E731
        va = np.ascontiguousarray(valid, np.uint8); fo = np.ascontiguousarray(found, np.uint8)
        uu, vv, zz, mn, mx, an = f32(u), f32(v), f32(z), f32(mind), f32(maxd), f32(angle)
        lv = np.ascontiguousarray(level, np.int32); md = np.ascontiguousarray(mpdesc, np.uint8)
        out = np.full(max(len(kp), 1), -1, np.int32); d3 = np.zeros(len(va), np.float32)
        nm = self.lib.refc_search_by_projection_kf(_p(kp), _p(desc), _p(oc), len(kp), _p(bg), _p(sc), len(sc), _p(va), _p(fo), _p(uu), _p(vv),
                                                   _p(zz), _p(mn), _p(mx), _p(lv), _p(an), _p(md), len(va), _f(th), int(orb_dist), int(check_ori),
                                                   _p(d3), _p(out))
        return out[:len(kp)], nm, d3


    def compute_stereo_matches(self, kpL, descL, kpR, descR, pyrL_bordered, pyrR_bordered, scale, inv, mb, mbf, border=19):
        nlev = len(pyrL_bordered)
        PL = (C.c_void_p * nlev)(); PR = (C.c_void_p * nlev)()
        steps = (C.c_size_t * nlev)(); widths = (C.c_int * nlev)(); heights = (C.c_int * nlev)()
        for l in range(nlev):
            a, b = pyrL_bordered[l], pyrR_bordered[l]
            PL[l] = a.ctypes.data; PR[l] = b.ctypes.data
            steps[l] = a.strides[0]; widths[l] = a.shape[1] - 2 * border; heights[l] = a.shape[0] - 2 * border
        kpL = np.ascontiguousarray(kpL, KP_DTYPE); kpR = np.ascontiguousarray(kpR, KP_DTYPE)
        descL = np.ascontiguousarray(descL, np.uint8); descR = np.ascontiguousarray(descR, np.uint8)
        scale = np.ascontiguousarray(scale, np.float32); inv = np.ascontiguousarray(inv, np.float32)
        u = np.zeros(len(kpL), np.float32); d = np.zeros(len(kpL), np.float32)
        self.lib.refc_compute_stereo_matches(_p(kpL), _p(descL), len(kpL), _p(kpR), _p(descR), len(kpR), PL, PR, steps, widths, heights, nlev,
                                             border, _p(scale), _p(inv), _f(mb), _f(mbf), _p(u), _p(d))
        return u, d

    @staticmethod
    def _fv(fv):
        return (np.ascontiguousarray(fv[0], np.uint32), np.ascontiguousarray(fv[1], np.int32), np.ascontiguousarray(fv[2], np.uint32))

    def search_by_bow_kf_frame(self, desc_kf, angle_kf, valid_kf, fv_kf, desc_f, angle_f, fv_f, nleft=-1, nnratio=0.6, check_ori=True):
        dk = np.ascontiguousarray(desc_kf, np.uint8); df = np.ascontiguousarray(desc_f, np.uint8)
        ak = np.ascontiguousarray(angle_kf, np.float32); af = np.ascontiguousarray(angle_f, np.float32)
        vk = np.ascontiguousarray(valid_kf, np.uint8)
        kn, ko, ki = self._fv(fv_kf); fn, fo, fi = self._fv(fv_f)
        out = np.full(len(df), -1, np.int32)
        nm = self.lib.refc_search_by_bow_kf_frame(_p(dk), _p(ak), _p(vk), len(dk), len(kn), _p(kn), _p(ko), _p(ki), _p(df), _p(af), len(df),
                                                  len(fn), _p(fn), _p(fo), _p(fi), int(nleft), _f(nnratio), int(check_ori), _p(out))
        return out, nm

    def search_by_bow_kf_kf(self, d1, a1, v1, fv1, d2, a2, v2, fv2, nnratio=0.6, check_ori=True):
        d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
        a1 = np.ascontiguousarray(a1, np.float32); a2 = np.ascontiguousarray(a2, np.float32)
        v1 = np.ascontiguousarray(v1, np.uint8); v2 = np.ascontiguousarray(v2, np.uint8)
        n1, o1, i1 = self._fv(fv1); n2, o2, i2 = self._fv(fv2)
        out = np.full(len(d1), -1, np.int32)
        nm = self.lib.refc_search_by_bow_kf_kf(_p(d1), _p(a1), _p(v1), len(d1), len(n1), _p(n1), _p(o1), _p(i1), _p(d2), _p(a2), _p(v2), len(d2),
                                               len(n2), _p(n2), _p(o2), _p(i2), _f(nnratio), int(check_ori), _p(out))
        return out, nm

    def search_for_triangulation(self, kp1, d1, free1, st1, fv1, kp2, d2, free2, st2, fv2, F12, ep, scale2, sigma2_2, only_stereo=False,
                                 coarse=False, check_ori=True):
        kp1 = np.ascontiguousarray(kp1, KP_DTYPE); kp2 = np.ascontiguousarray(kp2, KP_DTYPE)
        d1 = np.ascontiguousarray(d1, np.uint8); d2 = np.ascontiguousarray(d2, np.uint8)
        free1 = np.ascontiguousarray(free1, np.uint8); free2 = np.ascontiguousarray(free2, np.uint8)
        st1 = np.ascontiguousarray(st1, np.uint8); st2 = np.ascontiguousarray(st2, np.uint8)
        n1, o1, i1 = self._fv(fv1); n2, o2, i2 = self._fv(fv2)
        F = np.ascontiguousarray(F12, np.float32).reshape(9); e = np.ascontiguousarray(ep, np.float32)
        sc = np.ascontiguousarray(scale2, np.float32); sg = np.ascontiguousarray(sigma2_2, np.float32)
        out = np.full(len(d1), -1, np.int32)
        nm = self.lib.refc_search_for_triangulation(_p(kp1), _p(d1), _p(free1), _p(st1), len(d1), len(n1), _p(n1), _p(o1), _p(i1), _p(kp2), _p(d2),
                                                    _p(free2), _p(st2), len(d2), len(n2), _p(n2), _p(o2), _p(i2), _p(F), _p(e), _p(sc), _p(sg),
                                                    len(sc), int(only_stereo), int(coarse), int(check_ori), _p(out))
        return out, nm


class RefVocabulary:
    """DBoW2's own loadFromTextFile + transform + L1 score (Thirdparty/DBoW2/DBoW2, compiled by oracle/build_ref.sh)."""

    def __init__(self, ref, path):
        self.lib = ref.lib
        self.lib.refd_vocab_load_text.restype = _vp
        self.h = _vp(self.lib.refd_vocab_load_text(str(path).encode()))
        assert self.h.value, "loadFromTextFile failed"

    def __del__(self):
        try:
            self.lib.refd_vocab_destroy(self.h)
        except Exception:
            pass

    def info(self):
        v = [C.c_int(0) for _ in range(5)]
        self.lib.refd_vocab_info(self.h, *[C.byref(x) for x in v])
        return dict(n_nodes=v[0].value, n_words=v[1].value, k=v[2].value, L=v[3].value, weighting=v[4].value)

    def transform_features(self, desc, levelsup=4):
        d = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        n = len(d)
        word = np.zeros(n, np.uint32); weight = np.zeros(n, np.float64); node = np.zeros(n, np.uint32)
        self.lib.refd_transform_features(self.h, _p(d), n, levelsup, _p(word), _p(weight), _p(node))
        return word, weight, node

    def transform(self, desc, levelsup=4):
        d = np.ascontiguousarray(desc, np.uint8).reshape(-1, 32)
        n = len(d)
        ids = np.zeros(max(n, 1), np.uint32); vals = np.zeros(max(n, 1), np.float64)
        nodes = np.zeros(max(n, 1), np.uint32); offs = np.zeros(n + 1, np.int32); idx = np.zeros(max(n, 1), np.uint32)
        nb = C.c_int(0); nf = C.c_int(0)
        self.lib.refd_transform(self.h, _p(d), n, levelsup, _p(ids), _p(vals), C.byref(nb), _p(nodes), _p(offs), _p(idx), C.byref(nf))
        return (ids[:nb.value].copy(), vals[:nb.value].copy()), (nodes[:nf.value].copy(), offs[:nf.value + 1].copy(), idx[:offs[nf.value]].copy())

    def score(self, a, b):
        ia = np.ascontiguousarray(a[0], np.uint32); va = np.ascontiguousarray(a[1], np.float64)
        ib = np.ascontiguousarray(b[0], np.uint32); vb = np.ascontiguousarray(b[1], np.float64)
        self.lib.refd_score_l1.restype = C.c_double
        return self.lib.refd_score_l1(_p(ia), _p(va), len(ia), _p(ib), _p(vb), len(ib))


_cached = None


def load():
    global _cached
    if _cached is None:
        _cached = Ref()
    return _cached
