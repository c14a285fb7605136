// ORBmatcher.h — drop-in C++ adapter: `class ORB_SLAM3::ORBmatcher` with the reference's declarations
// (include/ORBmatcher.h:36-60) for the searches this library implements, over the C ABI (include/orbx.h).
//
// Include it where the reference's include/ORBmatcher.h was included, AFTER the headers that define the complete types
// ORB_SLAM3::Frame, KeyFrame and MapPoint (include/Frame.h, KeyFrame.h, MapPoint.h in ORB-SLAM3; the stand-ins of
// tests/cpp/matcher_adapter_test.cpp here): the bodies read exactly the members the reference functions read.
// Single-camera rigs (Nleft == -1, no mpCamera2): a two-fisheye rig keeps the reference code for these calls.
//
//   static int DescriptorDistance(a, b)                                              src/ORBmatcher3.cc:637-653
//   int SearchByProjection(Frame&, const vector<MapPoint*>&, th, bFarPoints, thFar)  src/ORBmatcher1.cc:45-215
//   int SearchByProjection(Frame& Current, const Frame& Last, th, bMono)             src/ORBmatcher3.cc:256-467
//   int SearchByBoW(KeyFrame*, Frame&, vector<MapPoint*>& vpMapPointMatches)         src/ORBmatcher1.cc:225-427
//   int SearchByBoW(KeyFrame*, KeyFrame*, vector<MapPoint*>& vpMatches12)            src/ORBmatcher2.cc:36-171
//   int SearchByBoW(const vector<KeyFrame*>&, Frame&, vector<vector<MapPoint*>>&, vector<int>&)
//                                     (added: the candidate loop of Tracking::Relocalization in one call)
//   int SearchByBoW(KeyFrame*, const vector<KeyFrame*>&, vector<vector<MapPoint*>>&, vector<int>&)
//                                     (added: the covisible loop of LoopClosing::DetectCommonRegionsFromBoW in one call)
//   int SearchForInitialization(Frame&, Frame&, vector<cv::Point2f>&, vector<int>&, windowSize)   src/ORBmatcher1.cc:650-765
//   int Fuse(KeyFrame*, const vector<MapPoint*>&, th, bRight)                        src/ORBmatcher2.cc:420-610
//   int Fuse(const vector<KeyFrame*>&, const vector<MapPoint*>&, th)  (added: the forward loop of SearchInNeighbors in one call)
//   int SearchByProjection(KeyFrame*, Sim3f&, vpPoints, vpMatched, th, ratioHamming)                    src/ORBmatcher1.cc:429-648
//   int SearchByProjection(KeyFrame*, Sim3f&, vpPoints, vpPointsKFs, vpMatched, vpMatchedKF, th, ratioHamming)
//   int Fuse(KeyFrame*, Sim3f&, const vector<MapPoint*>&, th, vector<MapPoint*>& vpReplacePoint)       src/ORBmatcher2.cc:612-729
//   int SearchAndFuse(const vector<KeyFrame*>&, const vector<Sim3f>&, const vector<MapPoint*>&, th)
//                                     (added: the loop body of both LoopClosing::SearchAndFuse overloads in one call)
//   int SearchForTriangulation(KeyFrame*, KeyFrame*, vector<pair<size_t, size_t>>&, bOnlyStereo, bCoarse)  src/ORBmatcher2.cc:173-471
//   int SearchForTriangulation(KeyFrame*, const vector<KeyFrame*>&, const vector<char>& vbCoarse, bOnlyStereo, body)
//                                     (added: the neighbour loop of LocalMapping::CreateNewMapPoints in one call)
// Not declared (no live caller / out of scope, DESIGN.md §8): SearchBySim3.
#ifndef ORBMATCHER_H
#define ORBMATCHER_H

#include <cstring>
#include <mutex>
#include <set>
#include <stdexcept>
#include <type_traits>
#include <utility>
#include <vector>

#include "ORBmatcherProjection.h"

namespace ORB_SLAM3 {

class ORBmatcher {
public:
    ORBmatcher(float nnratio = 0.6, bool checkOri = true, int cudaDevice = 0) : mfNNratio(nnratio), mbCheckOrientation(checkOri), device(cudaDevice) {}

    // Computes the Hamming distance between two ORB descriptors
    static int DescriptorDistance(const cv::Mat& a, const cv::Mat& b) { return orbx_descriptor_distance(a.ptr(0), b.ptr(0)); }

    // Search matches between Frame keypoints and projected MapPoints. Returns number of matches
    // Used to track the local map (Tracking)
    int SearchByProjection(Frame& F, const std::vector<MapPoint*>& vpMapPoints, const float th = 3, const bool bFarPoints = false,
                           const float thFarPoints = 50.0f)
    {
        return orbx_adapter::SearchByProjection(F, vpMapPoints, th, bFarPoints, thFarPoints, mfNNratio, device);
    }

    // Project MapPoints tracked in last frame into the current frame and search matches.
    // Used to track from previous frame (Tracking)
    int SearchByProjection(Frame& CurrentFrame, const Frame& LastFrame, const float th, const bool bMono)
    {
        // the Sophus / Eigen lines of the reference stay as they are (src/ORBmatcher3.cc:266-296): Eigen's own arithmetic
        const auto Tcw = CurrentFrame.GetPose();
        const auto twc = Tcw.inverse().translation();
        const auto Tlw = LastFrame.GetPose();
        const auto tlc = Tlw * twc;
        const bool bForward = tlc(2) > CurrentFrame.mb && !bMono;
        const bool bBackward = -tlc(2) > CurrentFrame.mb && !bMono;
        const int M = LastFrame.N;
        std::vector<float> u(M, 0.f), v(M, 0.f), invz(M, -1.f);            // invz < 0: the reference skips the point (:290-291)
        for (int i = 0; i < M; i++) {
            MapPoint* pMP = LastFrame.mvpMapPoints[i];
            if (pMP && !LastFrame.mvbOutlier[i]) {
                const auto x3Dw = pMP->GetWorldPos();
                const auto x3Dc = Tcw * x3Dw;
                invz[i] = 1.0 / x3Dc(2);
                if (invz[i] < 0) continue;
                const auto uv = CurrentFrame.mpCamera->project(x3Dc);
                u[i] = uv(0); v[i] = uv(1);
            }
        }
        return orbx_adapter::SearchByProjectionLast(CurrentFrame, LastFrame, u, v, invz, th, bForward, bBackward, mbCheckOrientation, device);
    }

    // Matching for the Map Initialization (only used in the monocular case)
    int SearchForInitialization(Frame& F1, Frame& F2, std::vector<cv::Point2f>& vbPrevMatched, std::vector<int>& vnMatches12, int windowSize = 10)
    {
        return orbx_adapter::SearchForInitialization(F1, F2, vbPrevMatched, vnMatches12, windowSize, mfNNratio, mbCheckOrientation, device);
    }

    // Project MapPoints into KeyFrame and search for duplicated MapPoints.  (Member templates: the body is compiled only where
    // Fuse is called, against the complete KeyFrame / MapPoint types.)
    template <class KF = KeyFrame, class MP = MapPoint>
    int Fuse(KF* pKF, const std::vector<MP*>& vpMapPoints, const float th = 3.0, const bool bRight = false)
    {
        if (bRight) throw std::invalid_argument("ORBmatcher::Fuse: bRight (two-camera rigs keep the reference code)");
        return Fuse(std::vector<KF*>(1, pKF), vpMapPoints, th);
    }

    // The same for several key frames: equal to the sum of Fuse(pKFi, vpMapPoints, th) over vpKFs in order (the forward loop of
    // LocalMapping::SearchInNeighbors), with one search call for all of them (orbx_adapter::FuseApply).
    template <class KF = KeyFrame, class MP = MapPoint>
    int Fuse(const std::vector<KF*>& vpKFs, const std::vector<MP*>& vpMapPoints, const float th = 3.0)
    {
        const int M = (int)vpMapPoints.size();
        const size_t nq = vpKFs.size() * (size_t)M;
        std::vector<uint8_t> valid(nq, 0);
        std::vector<float> u(nq, 0.f), v(nq, 0.f), invz(nq, 0.f);
        std::vector<int32_t> level(nq, 0);
        for (size_t k = 0; k < vpKFs.size(); ++k) {
            KF* pKF = vpKFs[k];
            if (pKF->NLeft != -1) throw std::invalid_argument("ORBmatcher::Fuse: NLeft != -1 (two-camera rigs keep the reference code)");
            // the reference's lines (src/ORBmatcher2.cc:420-610) with Eigen's / Sophus' own arithmetic; the search is orbx_fuse
            const auto Tcw = pKF->GetPose();
            const auto Ow = pKF->GetCameraCenter();
            auto* pCamera = pKF->mpCamera;
            for (int i = 0; i < M; i++) {
                MP* pMP = vpMapPoints[i];
                if (!pMP) continue;
                if (pMP->isBad()) continue;
                else if (pMP->IsInKeyFrame(pKF)) continue;
                using Vec3 = typename std::decay<decltype(pMP->GetWorldPos())>::type;
                const Vec3 p3Dw = pMP->GetWorldPos();
                const Vec3 p3Dc = Tcw * p3Dw;
                // Depth must be positive
                if (p3Dc(2) < 0.0f) continue;
                const float invzi = 1 / p3Dc(2);
                const auto uv = pCamera->project(p3Dc);
                const float maxDistance = pMP->GetMaxDistanceInvariance();
                const float minDistance = pMP->GetMinDistanceInvariance();
                const Vec3 PO = p3Dw - Ow;
                const float dist3D = PO.norm();
                // Depth must be inside the scale pyramid of the image
                if (dist3D < minDistance || dist3D > maxDistance) continue;
                // Viewing angle must be less than 60 deg
                const Vec3 Pn = pMP->GetNormal();
                if (PO.dot(Pn) < 0.5 * dist3D) continue;
                const size_t q = k * (size_t)M + i;
                valid[q] = 1; u[q] = uv(0); v[q] = uv(1); invz[q] = invzi;
                level[q] = pMP->PredictScale(dist3D, pKF);                  // IsInImage and the window: orbx_fuse
            }
        }
        return orbx_adapter::FuseApply(vpKFs, vpMapPoints, th, valid, u, v, invz, level, device);
    }

    // Project MapPoints using a Similarity Transformation and search matches.
    // Used in loop detection (Loop Closing)
    // (Member templates like Fuse: the Sim3 type is deduced from the argument, Sophus::Sim3f in ORB-SLAM3.)
    template <class KF = KeyFrame, class Sim3T, class MP = MapPoint>
    int SearchByProjection(KF* pKF, Sim3T& Scw, const std::vector<MP*>& vpPoints, std::vector<MP*>& vpMatched, int th, float ratioHamming = 1.0)
    {
        return SearchByProjectionSim3<KF, Sim3T, MP>(pKF, Scw, vpPoints, nullptr, vpMatched, nullptr, th, ratioHamming);
    }

    // Project MapPoints using a Similarity Transformation and search matches.
    // Used in Place Recognition (Loop Closing and Merging)
    template <class KF = KeyFrame, class Sim3T, class MP = MapPoint>
    int SearchByProjection(KF* pKF, Sim3T& Scw, const std::vector<MP*>& vpPoints, const std::vector<KF*>& vpPointsKFs, std::vector<MP*>& vpMatched,
                           std::vector<KF*>& vpMatchedKF, int th, float ratioHamming = 1.0)
    {
        if (vpPointsKFs.size() < vpPoints.size()) throw std::invalid_argument("ORBmatcher::SearchByProjection: vpPointsKFs is shorter than vpPoints");
        if ((int)vpMatchedKF.size() != pKF->N) throw std::invalid_argument("ORBmatcher::SearchByProjection: vpMatchedKF must have pKF->N entries");
        return SearchByProjectionSim3<KF, Sim3T, MP>(pKF, Scw, vpPoints, &vpPointsKFs, vpMatched, &vpMatchedKF, th, ratioHamming);
    }

    // Project MapPoints into KeyFrame using a given Sim3 and search for duplicated MapPoints.
    template <class KF = KeyFrame, class Sim3T, class MP = MapPoint>
    int Fuse(KF* pKF, Sim3T& Scw, const std::vector<MP*>& vpPoints, float th, std::vector<MP*>& vpReplacePoint)
    {
        if (vpReplacePoint.size() < vpPoints.size()) throw std::invalid_argument("ORBmatcher::Fuse: vpReplacePoint is shorter than vpPoints");
        return FuseSim3(std::vector<KF*>(1, pKF), std::vector<typename std::remove_const<Sim3T>::type>(1, Scw), vpPoints, th, vpReplacePoint, [](int) {});
    }

    // The loop body of both LoopClosing::SearchAndFuse overloads (loop correction and map merge) for the key frames vpKFs with
    // their corrected poses vScw, in order: per key frame, vpReplacePoints(M, NULL), Fuse(pKFi, Scw_i, vpMapPoints, th,
    // vpReplacePoints), then under pKFi->GetMap()->mMutexMapUpdate pRep->Replace(vpMapPoints[i]) for every non-NULL pRep.
    // One orbx_fuse_sim3 call for all key frames, plus one re-search call before a key frame whose points a Replace loop gave
    // new descriptors (orbx_adapter::FuseSim3Apply).  Returns the sum of the Fuse return values.
    template <class KF = KeyFrame, class Sim3T, class MP = MapPoint>
    int SearchAndFuse(const std::vector<KF*>& vpKFs, const std::vector<Sim3T>& vScw, const std::vector<MP*>& vpMapPoints, const float th = 4)
    {
        if (vScw.size() != vpKFs.size()) throw std::invalid_argument("ORBmatcher::SearchAndFuse: one Sim3 per key frame");
        std::vector<MP*> vpReplacePoints(vpMapPoints.size(), static_cast<MP*>(NULL));
        return FuseSim3(vpKFs, vScw, vpMapPoints, th, vpReplacePoints, [&](int k) {
            // Get Map Mutex
            std::unique_lock<std::mutex> lock(vpKFs[k]->GetMap()->mMutexMapUpdate);
            const int nLP = (int)vpMapPoints.size();
            for (int i = 0; i < nLP; i++) {
                MP* pRep = vpReplacePoints[i];
                if (pRep) pRep->Replace(vpMapPoints[i]);
            }
            std::fill(vpReplacePoints.begin(), vpReplacePoints.end(), static_cast<MP*>(NULL));   // the next key frame's vpReplacePoints
        });
    }

    // Search matches for triangulation of new MapPoints between two key frames; checks the epipolar constraint.  (Member
    // templates like Fuse.)  Equal to the batched overload below with the one neighbour pKF2.
    template <class KF = KeyFrame>
    int SearchForTriangulation(KF* pKF1, KF* pKF2, std::vector<std::pair<size_t, size_t>>& vMatchedPairs, const bool bOnlyStereo,
                               const bool bCoarse = false)
    {
        vMatchedPairs.clear();
        return SearchForTriangulation(pKF1, std::vector<KF*>(1, pKF2), std::vector<char>(1, (char)bCoarse), bOnlyStereo,
                                      [&](int, std::vector<std::pair<size_t, size_t>>& v) { vMatchedPairs.swap(v); return true; });
    }

    // The neighbour loop of LocalMapping::CreateNewMapPoints: for k = 0, 1, ... in order, body(k, vMatchedPairs) receives exactly
    // what SearchForTriangulation(pKF1, vpKF2[k], vMatchedPairs, bOnlyStereo, vbCoarse[k]) returns at that moment; body returns
    // false to stop (the CheckNewKeyFrames() return).  One orbx_search_for_triangulation_batch call searches every neighbour
    // against the KF1 features free at entry; before neighbour k is delivered its matches of KF1 features that gained a map point
    // since then are dropped, a neighbour whose own slots changed since entry is searched again (one extra call), and the
    // rotation filter runs on what is left (DESIGN.md §5d).  Poses are read at entry.  Returns the matches delivered.
    template <class KF = KeyFrame, class Body>
    int SearchForTriangulation(KF* pKF1, const std::vector<KF*>& vpKF2, const std::vector<char>& vbCoarse, const bool bOnlyStereo, Body body)
    {
        const int nK = (int)vpKF2.size();
        if ((int)vbCoarse.size() != nK) throw std::invalid_argument("ORBmatcher::SearchForTriangulation: one bCoarse per neighbour");
        auto single_camera = [](KF* pKF) {
            if (pKF->mpCamera2 || pKF->NLeft != -1)
                throw std::invalid_argument("ORBmatcher::SearchForTriangulation: two-camera key frame (two-camera rigs keep the reference code)");
        };
        single_camera(pKF1);
        for (KF* pKF2 : vpKF2) single_camera(pKF2);
        orbx_adapter::triangulation_diagnostics = orbx_adapter::TriangulationDiagnostics{};
        if (nK == 0) return 0;
        static_assert(sizeof(pKF1->mvKeysUn[0]) == sizeof(orbx_keypoint), "cv::KeyPoint must be the 28-byte POD");
        const int N1 = (int)pKF1->mvKeysUn.size();
        const orbx_keypoint* kp1 = reinterpret_cast<const orbx_keypoint*>(pKF1->mvKeysUn.data());
        std::vector<uint8_t> free1(N1), stereo1(N1);
        for (int i = 0; i < N1; ++i) { free1[i] = pKF1->GetMapPoint(i) == nullptr; stereo1[i] = pKF1->mvuRight[i] >= 0; }   // :246-258
        Csr fv1(pKF1->mFeatVec);
        const orbx_feature_vector va = fv1.view();
        std::vector<Csr> fv2;
        std::vector<std::vector<uint8_t>> free2(nK), stereo2(nK);
        std::vector<orbx_triangulation_view> views(nK);
        fv2.reserve(nK);
        for (int k = 0; k < nK; ++k) {
            KF* pKF2 = vpKF2[k];
            orbx_triangulation_view& V = views[k];
            // the reference's Sophus / Eigen lines (src/ORBmatcher2.cc:173-471) with the types' own arithmetic
            //Compute epipole in second image
            const auto T1w = pKF1->GetPose();
            const auto T2w = pKF2->GetPose();
            const auto Tw2 = pKF2->GetPoseInverse();
            const auto Cw = pKF1->GetCameraCenter();
            const auto C2 = T2w * Cw;
            const auto ep = pKF2->mpCamera->project(C2);
            const auto T12 = T1w * Tw2;
            const auto R12 = T12.rotationMatrix();
            const auto t12 = T12.translation();
            // Pinhole::epipolarConstrain (src/CameraModels/Pinhole.cpp:107-112): F12 = K1^-T [t12]x R12 K2^-1
            using SO3 = typename std::decay<decltype(T12.so3())>::type;
            const auto t12x = SO3::hat(t12);
            const auto K1 = pKF1->mpCamera->toK_();
            const auto K2 = pKF2->mpCamera->toK_();
            using Mat3 = typename std::decay<decltype(R12)>::type;
            const Mat3 F12 = K1.transpose().inverse() * t12x * R12 * K2.inverse();
            for (int r = 0; r < 3; ++r)
                for (int c = 0; c < 3; ++c) V.F12[r * 3 + c] = F12(r, c);
            V.ep[0] = ep(0); V.ep[1] = ep(1);
            const int N2 = (int)pKF2->mvKeysUn.size();
            free2[k].resize(N2); stereo2[k].resize(N2);
            for (int j = 0; j < N2; ++j) { free2[k][j] = pKF2->GetMapPoint(j) == nullptr; stereo2[k][j] = pKF2->mvuRight[j] >= 0; }   // :273-279
            fv2.emplace_back(pKF2->mFeatVec);
            V.n = N2;
            V.kp = reinterpret_cast<const orbx_keypoint*>(pKF2->mvKeysUn.data());
            V.desc = N2 ? pKF2->mDescriptors.ptr(0) : nullptr;
            V.free = free2[k].data(); V.stereo = stereo2[k].data();
            V.fv = fv2.back().view();
            V.scale = pKF2->mvScaleFactors.data(); V.sigma2 = pKF2->mvLevelSigma2.data();
            V.n_levels = (int)pKF2->mvScaleFactors.size();
            V.coarse = vbCoarse[k] != 0;
        }
        std::vector<int32_t> match((size_t)nK * N1, -1);
        std::vector<int> nm(nK, 0);
        orbx_adapter::check(orbx_search_for_triangulation_batch(device, kp1, N1 ? pKF1->mDescriptors.ptr(0) : nullptr, free1.data(), stereo1.data(), N1,
                                                                &va, nK, views.data(), bOnlyStereo, 0, match.data(), nm.data()),
                            "SearchForTriangulation");
        int total = 0;
        std::vector<std::pair<size_t, size_t>> vMatchedPairs;
        for (int k = 0; k < nK; ++k) {
            KF* pKF2 = vpKF2[k];
            int32_t* m = &match[(size_t)k * N1];
            orbx_triangulation_view& V = views[k];
            // a slot of pKF2 changed since entry (not by the loop itself: it adds map points to pKF1 and the searched neighbour
            // only): search this neighbour again with the live slots of both key frames
            bool changed = false;
            for (int j = 0; j < V.n && !changed; ++j) changed = (pKF2->GetMapPoint(j) == nullptr) != (free2[k][j] != 0);
            if (changed) {
                for (int j = 0; j < V.n; ++j) free2[k][j] = pKF2->GetMapPoint(j) == nullptr;
                for (int i = 0; i < N1; ++i) free1[i] = pKF1->GetMapPoint(i) == nullptr;
                int n = 0;
                orbx_adapter::check(orbx_search_for_triangulation(device, kp1, N1 ? pKF1->mDescriptors.ptr(0) : nullptr, free1.data(), stereo1.data(), N1,
                                                                  &va, V.kp, V.desc, V.free, V.stereo, V.n, &V.fv, V.F12, V.ep, V.scale, V.sigma2,
                                                                  V.n_levels, bOnlyStereo, V.coarse, 0, m, &n),
                                    "SearchForTriangulation");
                orbx_adapter::triangulation_diagnostics.researched_kfs += 1;
            }
            // KF1 features that gained a map point since entry: the reference skips them (pMP1 = pKF1->GetMapPoint(idx1); if (pMP1) continue;)
            for (int i = 0; i < N1; ++i)
                if (m[i] >= 0 && pKF1->GetMapPoint(i)) { m[i] = -1; orbx_adapter::triangulation_diagnostics.dropped += 1; }
            if (mbCheckOrientation) {                                       // :429-447, on the matches the reference would have made
                std::vector<int> idx;
                std::vector<float> a1, a2;
                for (int i = 0; i < N1; ++i)
                    if (m[i] >= 0) { idx.push_back(i); a1.push_back(pKF1->mvKeysUn[i].angle); a2.push_back(pKF2->mvKeysUn[m[i]].angle); }
                std::vector<uint8_t> keep(idx.size());
                orbx_adapter::check(orbx_rotation_consistency(a1.data(), a2.data(), (int)idx.size(), keep.data()), "SearchForTriangulation");
                for (size_t t = 0; t < idx.size(); ++t)
                    if (!keep[t]) m[idx[t]] = -1;
            }
            vMatchedPairs.clear();
            for (int i = 0; i < N1; ++i)
                if (m[i] >= 0) vMatchedPairs.push_back(std::make_pair((size_t)i, (size_t)m[i]));
            total += (int)vMatchedPairs.size();
            if (!body(k, vMatchedPairs)) break;
        }
        return total;
    }

    // Search matches between MapPoints in a KeyFrame and ORB in a Frame.
    // Brute force constrained to ORB that belong to the same vocabulary node (at a certain level)
    // Used in Relocalisation and Loop Detection
    int SearchByBoW(KeyFrame* pKF, Frame& F, std::vector<MapPoint*>& vpMapPointMatches)
    {
        const std::vector<MapPoint*> vpMapPointsKF = pKF->GetMapPointMatches();
        vpMapPointMatches = std::vector<MapPoint*>(F.N, static_cast<MapPoint*>(NULL));
        const int nA = (int)vpMapPointsKF.size();
        std::vector<uint8_t> validA(nA);
        std::vector<float> angA(nA), angB(F.N);
        for (int i = 0; i < nA; ++i) { validA[i] = vpMapPointsKF[i] && !vpMapPointsKF[i]->isBad(); angA[i] = pKF->mvKeysUn[i].angle; }   // :252-258, :335
        for (int j = 0; j < F.N; ++j) angB[j] = F.mvKeys[j].angle;                                                                 // :343
        Csr fa(pKF->mFeatVec), fb(F.mFeatVec);
        const orbx_feature_vector va = fa.view(), vb = fb.view();
        std::vector<int32_t> matchB(F.N, -1);
        int n = 0;
        orbx_adapter::check(orbx_search_by_bow(device, 0, pKF->mDescriptors.ptr(0), angA.data(), validA.data(), nA, &va, F.mDescriptors.ptr(0),
                                               angB.data(), nullptr, F.N, &vb, -1, mfNNratio, mbCheckOrientation, nullptr, matchB.data(), &n),
                            "SearchByBoW");
        for (int j = 0; j < F.N; ++j)
            if (matchB[j] >= 0) vpMapPointMatches[j] = vpMapPointsKF[matchB[j]];
        return n;
    }

    // Matching for the loop detection / place recognition between two key frames
    int SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, std::vector<MapPoint*>& vpMatches12)
    {
        const std::vector<MapPoint*> vpMapPoints1 = pKF1->GetMapPointMatches();
        const std::vector<MapPoint*> vpMapPoints2 = pKF2->GetMapPointMatches();
        const int nA = (int)vpMapPoints1.size(), nB = (int)vpMapPoints2.size();
        vpMatches12 = std::vector<MapPoint*>(nA, static_cast<MapPoint*>(NULL));
        std::vector<uint8_t> validA(nA), validB(nB);
        std::vector<float> angA(nA), angB(nB);
        for (int i = 0; i < nA; ++i) { validA[i] = vpMapPoints1[i] && !vpMapPoints1[i]->isBad(); angA[i] = pKF1->mvKeysUn[i].angle; }   // :73-82, :129
        for (int j = 0; j < nB; ++j) { validB[j] = vpMapPoints2[j] && !vpMapPoints2[j]->isBad(); angB[j] = pKF2->mvKeysUn[j].angle; }   // :95-103
        Csr fa(pKF1->mFeatVec), fb(pKF2->mFeatVec);
        const orbx_feature_vector va = fa.view(), vb = fb.view();
        std::vector<int32_t> matchA(nA, -1);
        int n = 0;
        orbx_adapter::check(orbx_search_by_bow(device, 1, pKF1->mDescriptors.ptr(0), angA.data(), validA.data(), nA, &va, pKF2->mDescriptors.ptr(0),
                                               angB.data(), validB.data(), nB, &vb, -1, mfNNratio, mbCheckOrientation, matchA.data(), nullptr, &n),
                            "SearchByBoW");
        for (int i = 0; i < nA; ++i)
            if (matchA[i] >= 0) vpMatches12[i] = vpMapPoints2[matchA[i]];
        return n;
    }

    // The candidate loop of Tracking::Relocalization: for every i, vnMatches[i] = SearchByBoW(vpKFs[i], F, vvpMapPointMatches[i]),
    // except that a NULL or isBad() candidate is not searched (vnMatches[i] = 0, vvpMapPointMatches[i] empty), as the loop
    // discards it.  One orbx_search_by_bow_batch call.  Every key frame's GetMapPointMatches() is read at entry: the loop changes
    // no map state between its searches, and a change made by another thread between two of the reference's searches is a race
    // the reference has too.  Returns the sum of vnMatches.  (Member templates like Fuse.)
    template <class KF = KeyFrame, class FrameT = Frame, class MP = MapPoint>
    int SearchByBoW(const std::vector<KF*>& vpKFs, FrameT& F, std::vector<std::vector<MP*>>& vvpMapPointMatches, std::vector<int>& vnMatches)
    {
        const int nK = (int)vpKFs.size();
        vvpMapPointMatches.assign(nK, std::vector<MP*>());
        vnMatches.assign(nK, 0);
        std::vector<int> live;                                          // positions in vpKFs that are searched
        std::vector<std::vector<MP*>> vpMPs;
        std::vector<std::vector<uint8_t>> valid;
        std::vector<std::vector<float>> ang;
        std::vector<Csr> fv;
        for (int i = 0; i < nK; ++i) {
            KF* pKF = vpKFs[i];
            if (!pKF || pKF->isBad()) continue;
            live.push_back(i);
            vpMPs.push_back(pKF->GetMapPointMatches());
            const std::vector<MP*>& mp = vpMPs.back();
            const int nA = (int)mp.size();
            valid.emplace_back(nA); ang.emplace_back(nA);
            for (int a = 0; a < nA; ++a) { valid.back()[a] = mp[a] && !mp[a]->isBad(); ang.back()[a] = pKF->mvKeysUn[a].angle; }   // :252-258, :335
            fv.emplace_back(pKF->mFeatVec);
        }
        const int nL = (int)live.size();
        if (nL == 0) return 0;
        std::vector<orbx_bow_view> views(nL);
        for (int k = 0; k < nL; ++k) {
            KF* pKF = vpKFs[live[k]];
            views[k] = orbx_bow_view{(int)vpMPs[k].size(), pKF->mDescriptors.ptr(0), ang[k].data(), valid[k].data(), fv[k].view()};
        }
        std::vector<float> angB(F.N);
        for (int j = 0; j < F.N; ++j) angB[j] = F.mvKeys[j].angle;                                                               // :343
        Csr fb(F.mFeatVec);
        const orbx_feature_vector vb = fb.view();
        std::vector<int32_t> match((size_t)nL * F.N, -1);
        std::vector<int> nm(nL, 0);
        orbx_adapter::check(orbx_search_by_bow_batch(device, 0, F.mDescriptors.ptr(0), angB.data(), nullptr, F.N, &vb, -1, nL, views.data(), mfNNratio,
                                                     mbCheckOrientation, match.data(), nm.data()),
                            "SearchByBoW");
        int total = 0;
        for (int k = 0; k < nL; ++k) {
            std::vector<MP*>& out = vvpMapPointMatches[live[k]];
            out.assign(F.N, static_cast<MP*>(NULL));
            const int32_t* m = &match[(size_t)k * F.N];
            for (int j = 0; j < F.N; ++j)
                if (m[j] >= 0) out[j] = vpMPs[k][m[j]];
            vnMatches[live[k]] = nm[k];
            total += nm[k];
        }
        return total;
    }

    // The covisible loop of LoopClosing::DetectCommonRegionsFromBoW: for every j, vnMatches[j] = SearchByBoW(pKF1, vpKF2[j],
    // vvpMatches12[j]), except that a NULL or isBad() entry is not searched (vnMatches[j] = 0, vvpMatches12[j] empty), as the
    // loop skips it.  One orbx_search_by_bow_batch call; map points are read at entry, as in the overload above.  Returns the sum
    // of vnMatches.
    template <class KF = KeyFrame, class MP = MapPoint>
    int SearchByBoW(KF* pKF1, const std::vector<KF*>& vpKF2, std::vector<std::vector<MP*>>& vvpMatches12, std::vector<int>& vnMatches)
    {
        const int nK = (int)vpKF2.size();
        vvpMatches12.assign(nK, std::vector<MP*>());
        vnMatches.assign(nK, 0);
        const std::vector<MP*> vpMapPoints1 = pKF1->GetMapPointMatches();
        const int nA = (int)vpMapPoints1.size();
        std::vector<uint8_t> validA(nA);
        std::vector<float> angA(nA);
        for (int i = 0; i < nA; ++i) { validA[i] = vpMapPoints1[i] && !vpMapPoints1[i]->isBad(); angA[i] = pKF1->mvKeysUn[i].angle; }   // :73-82, :129
        std::vector<int> live;
        std::vector<std::vector<MP*>> vpMPs;
        std::vector<std::vector<uint8_t>> valid;
        std::vector<std::vector<float>> ang;
        std::vector<Csr> fv;
        for (int j = 0; j < nK; ++j) {
            KF* pKF2 = vpKF2[j];
            if (!pKF2 || pKF2->isBad()) continue;
            live.push_back(j);
            vpMPs.push_back(pKF2->GetMapPointMatches());
            const std::vector<MP*>& mp = vpMPs.back();
            const int nB = (int)mp.size();
            valid.emplace_back(nB); ang.emplace_back(nB);
            for (int b = 0; b < nB; ++b) { valid.back()[b] = mp[b] && !mp[b]->isBad(); ang.back()[b] = pKF2->mvKeysUn[b].angle; }   // :95-103
            fv.emplace_back(pKF2->mFeatVec);
        }
        const int nL = (int)live.size();
        if (nL == 0) return 0;
        std::vector<orbx_bow_view> views(nL);
        for (int k = 0; k < nL; ++k) {
            KF* pKF2 = vpKF2[live[k]];
            views[k] = orbx_bow_view{(int)vpMPs[k].size(), pKF2->mDescriptors.ptr(0), ang[k].data(), valid[k].data(), fv[k].view()};
        }
        Csr fa(pKF1->mFeatVec);
        const orbx_feature_vector va = fa.view();
        std::vector<int32_t> match((size_t)nL * nA, -1);
        std::vector<int> nm(nL, 0);
        orbx_adapter::check(orbx_search_by_bow_batch(device, 1, pKF1->mDescriptors.ptr(0), angA.data(), validA.data(), nA, &va, -1, nL, views.data(),
                                                     mfNNratio, mbCheckOrientation, match.data(), nm.data()),
                            "SearchByBoW");
        int total = 0;
        for (int k = 0; k < nL; ++k) {
            std::vector<MP*>& out = vvpMatches12[live[k]];
            out.assign(nA, static_cast<MP*>(NULL));
            const int32_t* m = &match[(size_t)k * nA];
            for (int i = 0; i < nA; ++i)
                if (m[i] >= 0) out[i] = vpMPs[k][m[i]];
            vnMatches[live[k]] = nm[k];
            total += nm[k];
        }
        return total;
    }

public:
    static const int TH_LOW = 50;          // src/ORBmatcher1.cc:37-39
    static const int TH_HIGH = 100;
    static const int HISTO_LENGTH = 30;

protected:
    // The per-point lines of the Sim3 searches (src/ORBmatcher1.cc:429-648, ORBmatcher2.cc:612-729) after the isBad() /
    // spAlreadyFound test `keep`, with Eigen's / Sophus' own arithmetic: Tcw = SE3(R, t / s), depth, projection, distance window,
    // viewing angle, PredictScale.  IsInImage and the window are the C ABI's.  Fills entries [0, M) of valid / u / v / level.
    template <class KF, class Sim3T, class MP, class Keep>
    static void Sim3Project(KF* pKF, const Sim3T& Scw, const std::vector<MP*>& vpPoints, Keep keep, uint8_t* valid, float* u, float* v, int32_t* level)
    {
        if (pKF->NLeft != -1) throw std::invalid_argument("ORBmatcher: NLeft != -1 (two-camera rigs keep the reference code)");
        // Decompose Scw
        using SE3 = typename std::decay<decltype(pKF->GetPose())>::type;
        const SE3 Tcw = SE3(Scw.rotationMatrix(), Scw.translation() / Scw.scale());
        const auto Ow = Tcw.inverse().translation();
        for (int iMP = 0, iendMP = (int)vpPoints.size(); iMP < iendMP; iMP++) {
            MP* pMP = vpPoints[iMP];
            if (!pMP) continue;                                             // (the reference dereferences it)
            // Discard Bad MapPoints and already found
            if (pMP->isBad() || !keep(pMP)) continue;
            using Vec3 = typename std::decay<decltype(pMP->GetWorldPos())>::type;
            // Get 3D Coords.
            const Vec3 p3Dw = pMP->GetWorldPos();
            // Transform into Camera Coords.
            const Vec3 p3Dc = Tcw * p3Dw;
            // Depth must be positive
            if (p3Dc(2) < 0.0f) continue;
            // Project into Image
            const auto uv = pKF->mpCamera->project(p3Dc);
            // Depth must be inside the scale invariance region of the point
            const float maxDistance = pMP->GetMaxDistanceInvariance();
            const float minDistance = pMP->GetMinDistanceInvariance();
            const Vec3 PO = p3Dw - Ow;
            const float dist = PO.norm();
            if (dist < minDistance || dist > maxDistance) continue;
            // Viewing angle must be less than 60 deg
            const Vec3 Pn = pMP->GetNormal();
            if (PO.dot(Pn) < 0.5 * dist) continue;
            valid[iMP] = 1; u[iMP] = uv(0); v[iMP] = uv(1);
            level[iMP] = pMP->PredictScale(dist, pKF);                     // IsInImage and the window: the C ABI
        }
    }

    template <class KF, class Sim3T, class MP>
    int SearchByProjectionSim3(KF* pKF, Sim3T& Scw, const std::vector<MP*>& vpPoints, const std::vector<KF*>* vpPointsKFs,
                               std::vector<MP*>& vpMatched, std::vector<KF*>* vpMatchedKF, int th, float ratioHamming)
    {
        if ((int)vpMatched.size() != pKF->N) throw std::invalid_argument("ORBmatcher::SearchByProjection: vpMatched must have pKF->N entries");
        const int M = (int)vpPoints.size();
        std::vector<uint8_t> valid(M, 0);
        std::vector<float> u(M, 0.f), v(M, 0.f);
        std::vector<int32_t> level(M, 0), matchF;
        // Set of MapPoints already found in the KeyFrame
        std::set<MP*> spAlreadyFound(vpMatched.begin(), vpMatched.end());
        spAlreadyFound.erase(static_cast<MP*>(NULL));
        Sim3Project(pKF, Scw, vpPoints, [&](MP* pMP) { return !spAlreadyFound.count(pMP); }, valid.data(), u.data(), v.data(), level.data());
        const int nmatches = orbx_adapter::SearchByProjectionSim3(pKF, vpPoints, vpMatched, valid, u, v, level, th, ratioHamming, matchF, device);
        for (int idx = 0; idx < pKF->N; ++idx) {
            if (matchF[idx] < 0) continue;
            vpMatched[idx] = vpPoints[matchF[idx]];
            if (vpMatchedKF) (*vpMatchedKF)[idx] = (*vpPointsKFs)[matchF[idx]];
        }
        return nmatches;
    }

    // The Sim3 Fuse of vpPoints into each of vpKFs with its Sim3, in order; after(k) runs once key frame k is applied.
    template <class KF, class Sim3T, class MP, class After>
    int FuseSim3(const std::vector<KF*>& vpKFs, const std::vector<Sim3T>& vScw, const std::vector<MP*>& vpPoints, const float th,
                 std::vector<MP*>& vpReplacePoint, After after)
    {
        const size_t M = vpPoints.size(), nq = vpKFs.size() * M;
        std::vector<uint8_t> valid(nq, 0);
        std::vector<float> u(nq, 0.f), v(nq, 0.f);
        std::vector<int32_t> level(nq, 0);
        // spAlreadyFound = pKF->GetMapPoints() is taken at the start of each key frame, by FuseSim3Apply
        for (size_t k = 0; k < vpKFs.size(); ++k)
            Sim3Project(vpKFs[k], vScw[k], vpPoints, [](MP*) { return true; }, valid.data() + k * M, u.data() + k * M, v.data() + k * M,
                        level.data() + k * M);
        return orbx_adapter::FuseSim3Apply(vpKFs, vpPoints, th, valid, u, v, level, vpReplacePoint, after, device);
    }

    // DBoW2::FeatureVector (std::map<NodeId, std::vector<unsigned int>>, Thirdparty/DBoW2/DBoW2/FeatureVector.h:23-25) -> CSR
    struct Csr {
        std::vector<uint32_t> nodes, indices;
        std::vector<int32_t> offsets;
        template <class FeatVecT> explicit Csr(const FeatVecT& fv)
        {
            offsets.push_back(0);
            for (auto it = fv.begin(); it != fv.end(); ++it) {
                nodes.push_back((uint32_t)it->first);
                for (unsigned int idx : it->second) indices.push_back((uint32_t)idx);
                offsets.push_back((int32_t)indices.size());
            }
        }
        orbx_feature_vector view() const { return orbx_feature_vector{(int)nodes.size(), nodes.data(), offsets.data(), indices.data()}; }
    };

    float mfNNratio;
    bool mbCheckOrientation;
    int device;
};

}  // namespace ORB_SLAM3

#endif  // ORBMATCHER_H
