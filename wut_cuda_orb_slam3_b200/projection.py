"""Host mirror of the reference's frame grid and projection-guided searches (SURVEY.md §8(f)2) over the C ABI.

Reference interfaces: Frame::AssignFeaturesToGrid / GetFeaturesInArea (src/Frame.cc:387-418, 687-753) and the three
ORBmatcher::SearchByProjection overloads of the tracking thread (src/ORBmatcher1.cc:45-215, src/ORBmatcher3.cc:256-467,
469-578), ORBmatcher::SearchForInitialization (src/ORBmatcher1.cc:650-765), the search part of the local-mapping
ORBmatcher::Fuse (src/ORBmatcher2.cc:420-610), and loop closing's Sim3 SearchByProjection (src/ORBmatcher1.cc:429-648) and the
search part of its Sim3 Fuse (src/ORBmatcher2.cc:612-729).  Everything computes in liborbx.so on the GPU; there is no CPU
fallback.
"""
import ctypes as C

import numpy as np

from .capi import KP_DTYPE, FrameViewC, KeyFrameViewC, TrackPointsC, check, lib, ptr

GRID_COLS, GRID_ROWS = 64, 48


class FrameView:
    """The fields of ORB_SLAM3::Frame the searches read (Nleft == -1).  `bounds` = (mnMinX, mnMinY, mnMaxX, mnMaxY)."""

    def __init__(self, keys_un, descriptors, scale_factors, bounds, u_right=None, occupied=None):
        self.keys = np.ascontiguousarray(keys_un, KP_DTYPE)
        n = len(self.keys)
        self.desc = np.ascontiguousarray(descriptors, np.uint8).reshape(n, 32) if descriptors is not None else None
        self.scale = np.ascontiguousarray(scale_factors, np.float32)
        self.u_right = None if u_right is None else np.ascontiguousarray(u_right, np.float32)
        self.occupied = None if occupied is None else np.ascontiguousarray(occupied, np.uint8)
        self.bounds = tuple(np.float32(b) for b in bounds)
        mnx, mny, mxx, mxy = self.bounds
        # src/Frame.cc:161-162: static_cast<float>(FRAME_GRID_COLS) / (mnMaxX - mnMinX)
        self.grid_w_inv = np.float32(GRID_COLS) / np.float32(mxx - mnx)
        self.grid_h_inv = np.float32(GRID_ROWS) / np.float32(mxy - mny)
        self.c = FrameViewC(n, ptr(self.keys), ptr(self.desc), ptr(self.u_right), ptr(self.occupied), mnx, mny, mxx, mxy,
                            self.grid_w_inv, self.grid_h_inv, ptr(self.scale), len(self.scale))

    def __len__(self):
        return len(self.keys)

    def bounds_grid(self):
        return np.array(list(self.bounds) + [self.grid_w_inv, self.grid_h_inv], np.float32)

    def assign_features_to_grid(self, device=0):
        """Frame::AssignFeaturesToGrid -> (cell_start[3073], items) CSR over cell id = ix * 48 + iy."""
        cs = np.zeros(GRID_COLS * GRID_ROWS + 1, np.int32)
        items = np.zeros(max(len(self), 1), np.int32)
        check(lib().orbx_assign_features_to_grid(device, C.addressof(self.c), ptr(cs), ptr(items)))
        return cs, items[:cs[-1]]

    def get_features_in_area(self, x, y, r, min_level=-1, max_level=-1, device=0):
        out = np.zeros(max(len(self), 1), np.int32)
        n = C.c_int(0)
        check(lib().orbx_get_features_in_area(device, C.addressof(self.c), x, y, r, min_level, max_level, ptr(out), len(self), C.addressof(n)))
        return out[:n.value]


class KeyFrameView(FrameView):
    """The fields of ORB_SLAM3::KeyFrame that Fuse reads (NLeft == -1): a FrameView plus mvInvLevelSigma2 and mbf.  The Sim3
    Fuse (fuse_sim3) reads neither, so both may be left out for it."""

    def __init__(self, keys_un, descriptors, scale_factors, bounds, inv_level_sigma2=None, bf=0.0, u_right=None):
        super().__init__(keys_un, descriptors, scale_factors, bounds, u_right=u_right)
        self.inv_sigma2 = None if inv_level_sigma2 is None else np.ascontiguousarray(inv_level_sigma2, np.float32)
        self.bf = np.float32(bf)
        self.kc = KeyFrameViewC(self.c, ptr(self.inv_sigma2), self.bf)


def search_by_projection_map(frame, in_view, bad, proj_x, proj_y, proj_xr, view_cos, track_depth, scale_level, n_obs, descriptors,
                             th=1.0, far_points=False, th_far_points=0.0, nnratio=0.8, device=0):
    """ORBmatcher::SearchByProjection(F, vpMapPoints, th, bFarPoints, thFarPoints).  Returns (match_f[n], nmatches)."""
    a = dict(in_view=np.ascontiguousarray(in_view, np.uint8), bad=np.ascontiguousarray(bad, np.uint8),
             proj_x=np.ascontiguousarray(proj_x, np.float32), proj_y=np.ascontiguousarray(proj_y, np.float32),
             proj_xr=np.ascontiguousarray(proj_xr, np.float32), view_cos=np.ascontiguousarray(view_cos, np.float32),
             track_depth=np.ascontiguousarray(track_depth, np.float32), scale_level=np.ascontiguousarray(scale_level, np.int32),
             n_obs=np.ascontiguousarray(n_obs, np.int32), desc=np.ascontiguousarray(descriptors, np.uint8))
    n = len(a["in_view"])
    tp = TrackPointsC(n, ptr(a["in_view"]), ptr(a["bad"]), ptr(a["proj_x"]), ptr(a["proj_y"]), ptr(a["proj_xr"]), ptr(a["view_cos"]),
                      ptr(a["track_depth"]), ptr(a["scale_level"]), ptr(a["n_obs"]), ptr(a["desc"]))
    match_f = np.full(max(len(frame), 1), -1, np.int32)
    nm = C.c_int(0)
    check(lib().orbx_search_by_projection_map(device, C.addressof(frame.c), C.addressof(tp), th, int(far_points), th_far_points, nnratio,
                                              ptr(match_f), C.addressof(nm)))
    return match_f[:len(frame)], nm.value


def search_by_projection_last(cur, mbf, valid, u, v, invz, octave, angle, n_obs, descriptors, th, forward=False, backward=False,
                              check_orientation=True, device=0):
    """ORBmatcher::SearchByProjection(CurrentFrame, LastFrame, th, bMono) with the projection done by the caller."""
    valid = np.ascontiguousarray(valid, np.uint8); u = np.ascontiguousarray(u, np.float32); v = np.ascontiguousarray(v, np.float32)
    invz = np.ascontiguousarray(invz, np.float32); octave = np.ascontiguousarray(octave, np.int32)
    angle = np.ascontiguousarray(angle, np.float32); n_obs = np.ascontiguousarray(n_obs, np.int32)
    desc = np.ascontiguousarray(descriptors, np.uint8)
    match_f = np.full(max(len(cur), 1), -1, np.int32)
    nm = C.c_int(0)
    check(lib().orbx_search_by_projection_last(device, C.addressof(cur.c), mbf, len(valid), ptr(valid), ptr(u), ptr(v), ptr(invz), ptr(octave),
                                               ptr(angle), ptr(n_obs), ptr(desc), th, int(forward), int(backward), int(check_orientation),
                                               ptr(match_f), C.addressof(nm)))
    return match_f[:len(cur)], nm.value


def search_by_projection_kf(cur, valid, u, v, dist3d, min_dist, max_dist, level, angle, descriptors, th, orb_dist, check_orientation=True,
                            device=0):
    """ORBmatcher::SearchByProjection(CurrentFrame, pKF, sAlreadyFound, th, ORBdist) with the projection done by the caller."""
    valid = np.ascontiguousarray(valid, np.uint8); u = np.ascontiguousarray(u, np.float32); v = np.ascontiguousarray(v, np.float32)
    dist3d = np.ascontiguousarray(dist3d, np.float32); min_dist = np.ascontiguousarray(min_dist, np.float32)
    max_dist = np.ascontiguousarray(max_dist, np.float32); level = np.ascontiguousarray(level, np.int32)
    angle = np.ascontiguousarray(angle, np.float32); desc = np.ascontiguousarray(descriptors, np.uint8)
    match_f = np.full(max(len(cur), 1), -1, np.int32)
    nm = C.c_int(0)
    check(lib().orbx_search_by_projection_kf(device, C.addressof(cur.c), len(valid), ptr(valid), ptr(u), ptr(v), ptr(dist3d), ptr(min_dist),
                                             ptr(max_dist), ptr(level), ptr(angle), ptr(desc), th, int(orb_dist), int(check_orientation),
                                             ptr(match_f), C.addressof(nm)))
    return match_f[:len(cur)], nm.value


def search_for_initialization(kp1, desc1, frame2, prev_matched, window_size=100, nnratio=0.9, check_orientation=True, device=0):
    """ORBmatcher(nnratio, check_orientation).SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, window_size).

    kp1 / desc1 = F1.mvKeysUn / F1.mDescriptors, frame2 = a FrameView of F2, prev_matched = vbPrevMatched as [n1][2] (x, y).
    Returns (matches12[n1], nmatches, prev_matched_out); the input array is left as it is."""
    kp1 = np.ascontiguousarray(kp1, KP_DTYPE)
    n1 = len(kp1)
    desc1 = np.ascontiguousarray(desc1, np.uint8).reshape(n1, 32)
    prev = np.array(prev_matched, np.float32, copy=True).reshape(n1, 2)
    matches12 = np.full(max(n1, 1), -1, np.int32)
    nm = C.c_int(0)
    check(lib().orbx_search_for_initialization(device, ptr(kp1), ptr(desc1), n1, C.addressof(frame2.c), ptr(prev), int(window_size), nnratio,
                                               int(check_orientation), ptr(matches12), C.addressof(nm)))
    return matches12[:n1], nm.value, prev


def fuse(kfs, kf_offsets, point_desc, point, valid, u, v, invz, level, th=3.0, device=0):
    """The search part of ORBmatcher::Fuse(pKF, vpMapPoints, th) for many key frames in one call (orbx_fuse).

    kfs = KeyFrameViews; pairs [kf_offsets[k], kf_offsets[k + 1]) belong to kfs[k]; pair q is map point point[q] (a row of
    point_desc [n_desc][32]) at (u[q], v[q]) with invz[q] = 1 / z and level[q] = PredictScale; valid[q] = the caller's pre-checks.
    Returns (match[nq] = bestIdx or -1, n_fused[n_kf])."""
    n_kf = len(kfs)
    offs = np.ascontiguousarray(kf_offsets, np.int32)
    nq = int(offs[-1]) if len(offs) else 0
    pdesc = np.ascontiguousarray(point_desc, np.uint8).reshape(-1, 32)
    point = np.ascontiguousarray(point, np.int32); valid = np.ascontiguousarray(valid, np.uint8)
    u = np.ascontiguousarray(u, np.float32); v = np.ascontiguousarray(v, np.float32); invz = np.ascontiguousarray(invz, np.float32)
    level = np.ascontiguousarray(level, np.int32)
    arr = (KeyFrameViewC * max(n_kf, 1))(*[k.kc for k in kfs])
    match = np.full(max(nq, 1), -1, np.int32)
    n_fused = np.zeros(max(n_kf, 1), np.int32)
    check(lib().orbx_fuse(device, n_kf, C.addressof(arr), ptr(offs), len(pdesc), ptr(pdesc), ptr(point), ptr(valid), ptr(u), ptr(v), ptr(invz),
                          ptr(level), th, ptr(match), ptr(n_fused)))
    return match[:nq], n_fused[:n_kf]


def search_by_projection_sim3(kf, valid, u, v, level, descriptors, th, ratio_hamming=1.0, device=0):
    """ORBmatcher::SearchByProjection(pKF, Scw, vpPoints, vpMatched, th, ratioHamming) of loop closing, with the projection and
    the pre-checks done by the caller (valid).  kf = a FrameView of the key frame whose `occupied` marks vpMatched[idx] != NULL.
    Returns (match_f[n] = point index assigned to the feature by this call or -1, nmatches)."""
    valid = np.ascontiguousarray(valid, np.uint8); u = np.ascontiguousarray(u, np.float32); v = np.ascontiguousarray(v, np.float32)
    level = np.ascontiguousarray(level, np.int32); desc = np.ascontiguousarray(descriptors, np.uint8)
    match_f = np.full(max(len(kf), 1), -1, np.int32)
    nm = C.c_int(0)
    check(lib().orbx_search_by_projection_sim3(device, C.addressof(kf.c), len(valid), ptr(valid), ptr(u), ptr(v), ptr(level), ptr(desc),
                                               th, ratio_hamming, ptr(match_f), C.addressof(nm)))
    return match_f[:len(kf)], nm.value


def fuse_sim3(kfs, kf_offsets, point_desc, point, valid, u, v, level, th=4.0, device=0):
    """The search part of the Sim3 ORBmatcher::Fuse(pKF, Scw, vpPoints, th, vpReplacePoint) for many key frames in one call
    (orbx_fuse_sim3): the layout of fuse() without invz, and no reprojection gate.  Returns (match[nq], n_fused[n_kf])."""
    n_kf = len(kfs)
    offs = np.ascontiguousarray(kf_offsets, np.int32)
    nq = int(offs[-1]) if len(offs) else 0
    pdesc = np.ascontiguousarray(point_desc, np.uint8).reshape(-1, 32)
    point = np.ascontiguousarray(point, np.int32); valid = np.ascontiguousarray(valid, np.uint8)
    u = np.ascontiguousarray(u, np.float32); v = np.ascontiguousarray(v, np.float32); level = np.ascontiguousarray(level, np.int32)
    arr = (KeyFrameViewC * max(n_kf, 1))(*[k.kc for k in kfs])
    match = np.full(max(nq, 1), -1, np.int32)
    n_fused = np.zeros(max(n_kf, 1), np.int32)
    check(lib().orbx_fuse_sim3(device, n_kf, C.addressof(arr), ptr(offs), len(pdesc), ptr(pdesc), ptr(point), ptr(valid), ptr(u), ptr(v),
                               ptr(level), th, ptr(match), ptr(n_fused)))
    return match[:nq], n_fused[:n_kf]


def projection_rounds():
    """Speculation rounds the last search on this thread needed (diagnostics)."""
    return lib().orbx_projection_rounds()
