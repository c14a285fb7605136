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
// by one-line calls of the functions below (Nleft == -1 rigs; a two-fisheye rig keeps the reference code).
#pragma once
#include <cstring>
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

}  // namespace orbx_adapter
}  // namespace ORB_SLAM3
