// ORBmatcherProjection.h — drop-in bodies for the tracking thread's projection-guided searches over the C ABI (include/orbx.h).
//
// Header-only templates over the reference's own types: `FrameT` = ORB_SLAM3::Frame, `MapPointT` = ORB_SLAM3::MapPoint (only the
// members the reference functions themselves read are touched, so the same code compiles against the reference headers and
// against the stand-ins of tests/cpp/matcher_adapter_test.cpp).  A maintainer replaces the bodies of
//   int ORBmatcher::SearchByProjection(Frame &F, const vector<MapPoint*> &vpMapPoints, const float th, const bool bFarPoints,
//                                      const float thFarPoints)                                     src/ORBmatcher1.cc:45-215
//   int ORBmatcher::SearchByProjection(Frame &CurrentFrame, const Frame &LastFrame, const float th, const bool bMono)
//                                                                                                   src/ORBmatcher3.cc:256-467
//   int ORBmatcher::SearchForInitialization(Frame &F1, Frame &F2, vector<cv::Point2f> &vbPrevMatched, vector<int> &vnMatches12,
//                                           int windowSize)                                        src/ORBmatcher1.cc:650-765
// by one-line calls of the functions below (Nleft == -1 rigs; a two-fisheye rig keeps the reference code).  FuseApply is the
// C ABI side and the bookkeeping of ORBmatcher::Fuse (src/ORBmatcher2.cc:420-610); SearchByProjectionSim3 and FuseSim3Apply are
// the same for loop closing's Sim3 SearchByProjection (src/ORBmatcher1.cc:429-648) and Sim3 Fuse (src/ORBmatcher2.cc:612-729).
// The class keeps the per-point Eigen lines.
#pragma once
#include <algorithm>
#include <cstring>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "orbx.h"

namespace ORB_SLAM3 {
namespace orbx_adapter {

inline void check(int rc, const char* what)
{
    if (rc != ORBX_OK) throw std::runtime_error(std::string(what) + ": " + orbx_last_error());
}

// The frame as the C ABI reads it.  `occupied` is filled by the caller-specific predicate.
template <class FrameT>
inline orbx_frame_view view_of(const FrameT& F, const std::vector<uint8_t>& occupied)
{
    static_assert(sizeof(F.mvKeysUn[0]) == sizeof(orbx_keypoint), "cv::KeyPoint must be the 28-byte POD");
    orbx_frame_view v{};
    v.n = F.N;
    v.keys_un = reinterpret_cast<const orbx_keypoint*>(F.mvKeysUn.data());
    v.descriptors = F.mDescriptors.ptr(0);
    v.u_right = F.mvuRight.empty() ? nullptr : F.mvuRight.data();
    v.occupied = occupied.data();
    v.min_x = FrameT::mnMinX; v.min_y = FrameT::mnMinY; v.max_x = FrameT::mnMaxX; v.max_y = FrameT::mnMaxY;
    v.grid_w_inv = FrameT::mfGridElementWidthInv; v.grid_h_inv = FrameT::mfGridElementHeightInv;
    v.scale_factors = F.mvScaleFactors.data();
    v.n_levels = (int)F.mvScaleFactors.size();
    return v;
}

// ORBmatcher::SearchByProjection(Frame&, const vector<MapPoint*>&, th, bFarPoints, thFarPoints) — src/ORBmatcher1.cc:45-215
template <class FrameT, class MapPointT>
inline int SearchByProjection(FrameT& F, const std::vector<MapPointT*>& vpMapPoints, const float th, const bool bFarPoints,
                              const float thFarPoints, const float mfNNratio, int device = 0)
{
    const int M = (int)vpMapPoints.size();
    std::vector<uint8_t> inView(M), bad(M), desc((size_t)32 * M), occ(F.N);
    std::vector<float> px(M), py(M), pxr(M), vc(M), depth(M);
    std::vector<int32_t> lvl(M), nobs(M), matchF(F.N);
    for (int i = 0; i < M; ++i) {
        MapPointT* p = vpMapPoints[i];
        inView[i] = p->mbTrackInView; bad[i] = p->isBad();
        px[i] = p->mTrackProjX; py[i] = p->mTrackProjY; pxr[i] = p->mTrackProjXR; vc[i] = p->mTrackViewCos; depth[i] = p->mTrackDepth;
        lvl[i] = p->mnTrackScaleLevel; nobs[i] = p->Observations();
        std::memcpy(&desc[(size_t)32 * i], p->GetDescriptor().ptr(0), 32);
    }
    for (int j = 0; j < F.N; ++j) occ[j] = F.mvpMapPoints[j] && F.mvpMapPoints[j]->Observations() > 0;   // :87-89
    const orbx_frame_view fv = view_of(F, occ);
    const orbx_track_points tp = {M, inView.data(), bad.data(), px.data(), py.data(), pxr.data(), vc.data(), depth.data(), lvl.data(),
                                  nobs.data(), desc.data()};
    int n = 0;
    check(orbx_search_by_projection_map(device, &fv, &tp, th, bFarPoints, thFarPoints, mfNNratio, matchF.data(), &n), "SearchByProjection");
    for (int j = 0; j < F.N; ++j)
        if (matchF[j] >= 0) F.mvpMapPoints[j] = vpMapPoints[matchF[j]];
    return n;
}

// ORBmatcher::SearchByProjection(Frame& CurrentFrame, const Frame& LastFrame, th, bMono) — src/ORBmatcher3.cc:256-467.  The
// Sophus / Eigen lines of the reference (:266-273, :284-296) stay in the caller, which hands over per last-frame feature i the
// projection `uv[i]` (mpCamera->project(Tcw * x3Dw)), `invz[i]` (1.0 / x3Dc(2)) and the flags bForward / bBackward.
template <class FrameT>
inline int SearchByProjectionLast(FrameT& CurrentFrame, const FrameT& LastFrame, const std::vector<float>& u, const std::vector<float>& v,
                                  const std::vector<float>& invz, const float th, const bool bForward, const bool bBackward,
                                  const bool mbCheckOrientation, int device = 0)
{
    const int M = LastFrame.N;
    std::vector<uint8_t> valid(M), desc((size_t)32 * M), occ(CurrentFrame.N);
    std::vector<int32_t> octave(M), nobs(M), matchF(CurrentFrame.N);
    std::vector<float> angle(M);
    for (int i = 0; i < M; ++i) {
        auto* pMP = LastFrame.mvpMapPoints[i];
        valid[i] = pMP && !LastFrame.mvbOutlier[i];                                                       // :278-281
        octave[i] = LastFrame.mvKeys[i].octave; angle[i] = LastFrame.mvKeysUn[i].angle;                  // :303, :358
        if (valid[i]) { nobs[i] = pMP->Observations(); std::memcpy(&desc[(size_t)32 * i], pMP->GetDescriptor().ptr(0), 32); }
    }
    for (int j = 0; j < CurrentFrame.N; ++j) occ[j] = CurrentFrame.mvpMapPoints[j] && CurrentFrame.mvpMapPoints[j]->Observations() > 0;
    const orbx_frame_view fv = view_of(CurrentFrame, occ);
    int n = 0;
    check(orbx_search_by_projection_last(device, &fv, CurrentFrame.mbf, M, valid.data(), u.data(), v.data(), invz.data(), octave.data(),
                                         angle.data(), nobs.data(), desc.data(), th, bForward, bBackward, mbCheckOrientation, matchF.data(), &n),
          "SearchByProjection");
    for (int j = 0; j < CurrentFrame.N; ++j)
        if (matchF[j] >= 0) CurrentFrame.mvpMapPoints[j] = LastFrame.mvpMapPoints[matchF[j]];
    return n;
}

// ORBmatcher::SearchForInitialization(Frame& F1, Frame& F2, vector<cv::Point2f>& vbPrevMatched, vector<int>& vnMatches12,
// windowSize) — src/ORBmatcher1.cc:650-765.  `PointT` = cv::Point2f, handed to the C ABI as its [n][2] floats.
template <class FrameT, class PointT>
inline int SearchForInitialization(FrameT& F1, FrameT& F2, std::vector<PointT>& vbPrevMatched, std::vector<int>& vnMatches12, int windowSize,
                                   const float mfNNratio, const bool mbCheckOrientation, int device = 0)
{
    static_assert(sizeof(PointT) == 8, "cv::Point2f must be two packed floats");
    static_assert(sizeof(F1.mvKeysUn[0]) == sizeof(orbx_keypoint), "cv::KeyPoint must be the 28-byte POD");
    const int n1 = (int)F1.mvKeysUn.size();
    if ((int)vbPrevMatched.size() < n1) throw std::runtime_error("SearchForInitialization: vbPrevMatched is shorter than F1.mvKeysUn");
    vnMatches12.assign(n1, -1);
    const std::vector<uint8_t> none;
    orbx_frame_view fv = view_of(F2, none);
    fv.occupied = nullptr; fv.u_right = nullptr;                                // not read by this search
    int n = 0;
    check(orbx_search_for_initialization(device, reinterpret_cast<const orbx_keypoint*>(F1.mvKeysUn.data()), n1 ? F1.mDescriptors.ptr(0) : nullptr,
                                         n1, &fv, reinterpret_cast<float*>(vbPrevMatched.data()), windowSize, mfNNratio, mbCheckOrientation,
                                         vnMatches12.data(), &n),
          "SearchForInitialization");
    return n;
}

// What the last Fuse on this thread re-searched because a Replace earlier in the call changed a point's descriptor: pairs
// re-searched and the extra orbx_fuse calls that took (diagnostics).
struct FuseDiagnostics { int researched_pairs = 0, extra_calls = 0; };
inline thread_local FuseDiagnostics fuse_diagnostics;

// The key frame as orbx_fuse reads it (KeyFrame stores the bounds as it stores them: the view takes them as floats).
template <class KF>
inline orbx_keyframe_view keyframe_view_of(const KF* pKF)
{
    static_assert(sizeof(pKF->mvKeysUn[0]) == sizeof(orbx_keypoint), "cv::KeyPoint must be the 28-byte POD");
    orbx_keyframe_view k{};
    orbx_frame_view& v = k.frame;
    v.n = (int)pKF->mvKeysUn.size();
    v.keys_un = reinterpret_cast<const orbx_keypoint*>(pKF->mvKeysUn.data());
    v.descriptors = v.n ? pKF->mDescriptors.ptr(0) : nullptr;
    v.u_right = pKF->mvuRight.empty() ? nullptr : pKF->mvuRight.data();
    v.min_x = (float)pKF->mnMinX; v.min_y = (float)pKF->mnMinY; v.max_x = (float)pKF->mnMaxX; v.max_y = (float)pKF->mnMaxY;
    v.grid_w_inv = pKF->mfGridElementWidthInv; v.grid_h_inv = pKF->mfGridElementHeightInv;
    v.scale_factors = pKF->mvScaleFactors.data();
    v.n_levels = (int)pKF->mvScaleFactors.size();
    k.inv_level_sigma2 = pKF->mvInvLevelSigma2.data();
    k.bf = pKF->mbf;
    return k;
}

// ORBmatcher::Fuse over the key frames vpKFs in order, each with all of vpMapPoints: pair q = k * M + i.  The caller has run the
// reference's per-point lines: valid[q] (pMP && !isBad() && !IsInKeyFrame(pKF), depth, distance window, viewing angle), the
// projection (u, v, invz) and level (PredictScale).  One orbx_fuse call searches every pair; then per key frame, in order:
// pairs whose point's live descriptor differs from the one searched with (a Replace in an earlier key frame of the call) are
// re-searched in one extra call, and the reference's tail is replayed with isBad() / IsInKeyFrame(pKF) re-evaluated live.
template <class KF, class MP>
inline int FuseApply(const std::vector<KF*>& vpKFs, const std::vector<MP*>& vpMapPoints, const float th, const std::vector<uint8_t>& valid,
                     const std::vector<float>& u, const std::vector<float>& v, const std::vector<float>& invz, const std::vector<int32_t>& level,
                     int device = 0)
{
    const int nK = (int)vpKFs.size(), M = (int)vpMapPoints.size();
    const size_t nq = (size_t)nK * M;
    fuse_diagnostics = FuseDiagnostics{};
    // descriptors the pairs were searched with: rows of `rows`, row_of[q]; the first M rows are the snapshot of the points
    std::vector<uint8_t> rows((size_t)M * 32, 0);
    for (int i = 0; i < M; ++i)
        if (vpMapPoints[i] && !vpMapPoints[i]->isBad()) std::memcpy(&rows[(size_t)32 * i], vpMapPoints[i]->GetDescriptor().ptr(0), 32);
    std::vector<int32_t> row_of(nq), point(nq), match(nq, -1), offs(nK + 1), nf(std::max(nK, 1));
    for (size_t q = 0; q < nq; ++q) row_of[q] = point[q] = (int32_t)(q % (size_t)std::max(M, 1));
    for (int k = 0; k <= nK; ++k) offs[k] = k * M;
    std::vector<orbx_keyframe_view> views(nK);
    for (int k = 0; k < nK; ++k) views[k] = keyframe_view_of(vpKFs[k]);
    check(orbx_fuse(device, nK, views.data(), offs.data(), M, rows.data(), point.data(), valid.data(), u.data(), v.data(), invz.data(),
                    level.data(), th, match.data(), nf.data()),
          "Fuse");
    // re-search pairs qs of key frame k with the points' live descriptors (appended to rows)
    auto research = [&](int k, const std::vector<size_t>& qs) {
        const int n = (int)qs.size();
        std::vector<uint8_t> d((size_t)n * 32), ok(n, 1);
        std::vector<int32_t> pt(n), lv(n), m(n), o = {0, n};
        std::vector<float> uu(n), vv(n), iz(n);
        for (int j = 0; j < n; ++j) {
            const size_t q = qs[j];
            std::memcpy(&d[(size_t)32 * j], vpMapPoints[point[q]]->GetDescriptor().ptr(0), 32);
            pt[j] = j; uu[j] = u[q]; vv[j] = v[q]; iz[j] = invz[q]; lv[j] = level[q];
        }
        int nfk = 0;
        check(orbx_fuse(device, 1, &views[k], o.data(), n, d.data(), pt.data(), ok.data(), uu.data(), vv.data(), iz.data(), lv.data(), th,
                        m.data(), &nfk),
              "Fuse");
        for (int j = 0; j < n; ++j) {
            row_of[qs[j]] = (int32_t)(rows.size() / 32);
            rows.insert(rows.end(), d.begin() + (size_t)32 * j, d.begin() + (size_t)32 * (j + 1));
            match[qs[j]] = m[j];
        }
        fuse_diagnostics.researched_pairs += n;
        fuse_diagnostics.extra_calls += 1;
    };
    auto live = [&](size_t q, KF* pKF) {
        MP* pMP = vpMapPoints[point[q]];
        return valid[q] && pMP && !pMP->isBad() && !pMP->IsInKeyFrame(pKF);
    };
    auto stale = [&](size_t q) { return std::memcmp(vpMapPoints[point[q]]->GetDescriptor().ptr(0), &rows[(size_t)32 * row_of[q]], 32) != 0; };
    int nFused = 0;
    for (int k = 0; k < nK; ++k) {
        KF* pKF = vpKFs[k];
        if (k > 0) {
            std::vector<size_t> qs;
            for (size_t q = (size_t)k * M; q < (size_t)(k + 1) * M; ++q)
                if (live(q, pKF) && stale(q)) qs.push_back(q);
            if (!qs.empty()) research(k, qs);
        }
        for (size_t q = (size_t)k * M; q < (size_t)(k + 1) * M; ++q) {
            if (!live(q, pKF)) continue;
            if (stale(q)) research(k, std::vector<size_t>(1, q));   // vpMapPoints holds the point twice (see DESIGN.md §5b)
            const int bestIdx = match[q];
            if (bestIdx < 0) continue;
            MP* pMP = vpMapPoints[point[q]];
            // If there is already a MapPoint replace otherwise add new measurement (src/ORBmatcher2.cc:420-610)
            MP* pMPinKF = pKF->GetMapPoint(bestIdx);
            if (pMPinKF) {
                if (!pMPinKF->isBad()) {
                    if (pMPinKF->Observations() > pMP->Observations())
                        pMP->Replace(pMPinKF);
                    else
                        pMPinKF->Replace(pMP);
                }
            } else {
                pMP->AddObservation(pKF, bestIdx);
                pKF->AddMapPoint(pMP, bestIdx);
            }
            nFused++;
        }
    }
    return nFused;
}

// Sim3 SearchByProjection (src/ORBmatcher1.cc:429-648): the caller has run the reference's per-point lines into valid[i]
// (!isBad(), not in spAlreadyFound, depth, distance window, viewing angle), (u, v) and level (PredictScale).  The key frame's
// slots are vpMatched: a non-NULL entry on entry is skipped.  matchF[idx] = index of the point this call assigned to idx, or -1.
template <class KF, class MP>
inline int SearchByProjectionSim3(KF* pKF, const std::vector<MP*>& vpPoints, const std::vector<MP*>& vpMatched, const std::vector<uint8_t>& valid,
                                  const std::vector<float>& u, const std::vector<float>& v, const std::vector<int32_t>& level, const int th,
                                  const float ratioHamming, std::vector<int32_t>& matchF, int device = 0)
{
    const int M = (int)vpPoints.size(), N = (int)vpMatched.size();
    std::vector<uint8_t> occ(N), desc((size_t)32 * M, 0);
    for (int j = 0; j < N; ++j) occ[j] = vpMatched[j] != nullptr;
    for (int i = 0; i < M; ++i)
        if (valid[i]) std::memcpy(&desc[(size_t)32 * i], vpPoints[i]->GetDescriptor().ptr(0), 32);
    orbx_frame_view fv = keyframe_view_of(pKF).frame;
    fv.occupied = occ.data();
    matchF.assign(N, -1);
    int n = 0;
    check(orbx_search_by_projection_sim3(device, &fv, M, valid.data(), u.data(), v.data(), level.data(), desc.data(), (float)th, ratioHamming,
                                         matchF.data(), &n),
          "SearchByProjection");
    return n;
}

// What the last Sim3 Fuse / SearchAndFuse on this thread re-searched because a Replace loop between two key frames changed a
// point's descriptor: pairs re-searched and the extra orbx_fuse_sim3 calls that took (diagnostics).
struct SearchAndFuseDiagnostics { int researched_pairs = 0, extra_calls = 0; };
inline thread_local SearchAndFuseDiagnostics search_and_fuse_diagnostics;

// The Sim3 Fuse (src/ORBmatcher2.cc:612-729) over the key frames vpKFs in order, each with all of vpPoints: pair q = k * M + i.
// The caller has run the reference's per-point lines into valid[q] (pMP && !isBad() on entry, depth, distance window, viewing
// angle), (u, v) and level.  One orbx_fuse_sim3 call searches every pair; then per key frame, in order:
//   1. spAlreadyFound = pKF->GetMapPoints() and isBad() are evaluated once, as the reference's snapshot at entry;
//   2. pairs still live whose point's descriptor differs from the one searched with (a Replace loop after an earlier key frame)
//      are re-searched in one extra call;
//   3. the reference's tail is replayed in point order into vpReplacePoint (AddObservation / AddMapPoint for an empty slot);
//   4. after(k) runs: SearchAndFuse's Replace loop, or nothing for a single Fuse.
// Nothing inside one key frame's Fuse changes a descriptor or a bad flag (Replace runs after it), so no per-pair re-check is
// needed inside step 3 (DESIGN.md §5b).  Returns the sum of the per-key-frame nFused.
template <class KF, class MP, class After>
inline int FuseSim3Apply(const std::vector<KF*>& vpKFs, const std::vector<MP*>& vpPoints, const float th, const std::vector<uint8_t>& valid,
                         const std::vector<float>& u, const std::vector<float>& v, const std::vector<int32_t>& level,
                         std::vector<MP*>& vpReplacePoint, After after, int device = 0)
{
    const int nK = (int)vpKFs.size(), M = (int)vpPoints.size();
    const size_t nq = (size_t)nK * M;
    search_and_fuse_diagnostics = SearchAndFuseDiagnostics{};
    // the descriptors every pair is first searched with: the points' at entry (each pair belongs to one key frame, so a pair is
    // re-searched at most once, at the start of its key frame)
    std::vector<uint8_t> rows((size_t)M * 32, 0);
    for (int i = 0; i < M; ++i)
        if (vpPoints[i] && !vpPoints[i]->isBad()) std::memcpy(&rows[(size_t)32 * i], vpPoints[i]->GetDescriptor().ptr(0), 32);
    std::vector<int32_t> point(nq), match(nq, -1), offs(nK + 1), nf(std::max(nK, 1));
    for (size_t q = 0; q < nq; ++q) point[q] = (int32_t)(q % (size_t)std::max(M, 1));
    for (int k = 0; k <= nK; ++k) offs[k] = k * M;
    std::vector<orbx_keyframe_view> views(nK);
    for (int k = 0; k < nK; ++k) views[k] = keyframe_view_of(vpKFs[k]);
    check(orbx_fuse_sim3(device, nK, views.data(), offs.data(), M, rows.data(), point.data(), valid.data(), u.data(), v.data(), level.data(), th,
                         match.data(), nf.data()),
          "Fuse");
    int nFused = 0;
    std::vector<uint8_t> live(M);
    for (int k = 0; k < nK; ++k) {
        KF* pKF = vpKFs[k];
        const size_t q0 = (size_t)k * M;
        // Set of MapPoints already found in the KeyFrame (src/ORBmatcher2.cc:612-729), and the isBad() test, at entry
        const auto spAlreadyFound = pKF->GetMapPoints();
        std::vector<size_t> stale;
        for (int i = 0; i < M; ++i) {
            MP* pMP = vpPoints[i];
            live[i] = valid[q0 + i] && !pMP->isBad() && !spAlreadyFound.count(pMP);
            if (live[i] && std::memcmp(pMP->GetDescriptor().ptr(0), &rows[(size_t)32 * i], 32) != 0) stale.push_back(q0 + i);
        }
        if (!stale.empty()) {
            const int n = (int)stale.size();
            std::vector<uint8_t> d((size_t)n * 32), ok(n, 1);
            std::vector<int32_t> pt(n), lv(n), m(n), o = {0, n};
            std::vector<float> uu(n), vv(n);
            for (int j = 0; j < n; ++j) {
                const size_t q = stale[j];
                std::memcpy(&d[(size_t)32 * j], vpPoints[point[q]]->GetDescriptor().ptr(0), 32);
                pt[j] = j; uu[j] = u[q]; vv[j] = v[q]; lv[j] = level[q];
            }
            int nfk = 0;
            check(orbx_fuse_sim3(device, 1, &views[k], o.data(), n, d.data(), pt.data(), ok.data(), uu.data(), vv.data(), lv.data(), th, m.data(), &nfk),
                  "Fuse");
            for (int j = 0; j < n; ++j) match[stale[j]] = m[j];
            search_and_fuse_diagnostics.researched_pairs += n;
            search_and_fuse_diagnostics.extra_calls += 1;
        }
        for (int iMP = 0; iMP < M; iMP++) {
            if (!live[iMP]) continue;
            const int bestIdx = match[q0 + iMP];
            if (bestIdx < 0) continue;
            MP* pMP = vpPoints[iMP];
            // If there is already a MapPoint replace otherwise add new measurement
            MP* pMPinKF = pKF->GetMapPoint(bestIdx);
            if (pMPinKF) {
                if (!pMPinKF->isBad()) vpReplacePoint[iMP] = pMPinKF;
            } else {
                pMP->AddObservation(pKF, bestIdx);
                pKF->AddMapPoint(pMP, bestIdx);
            }
            nFused++;
        }
        after(k);
    }
    return nFused;
}

// What the last batched SearchForTriangulation on this thread did besides delivering the batch: neighbours searched again because
// their map-point slots changed after entry, and matches dropped because their KF1 feature gained a map point (diagnostics).
struct TriangulationDiagnostics { int researched_kfs = 0, dropped = 0; };
inline thread_local TriangulationDiagnostics triangulation_diagnostics;

}  // namespace orbx_adapter
}  // namespace ORB_SLAM3
