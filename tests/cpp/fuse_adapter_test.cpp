// Compiles csrc/adapter/ORBmatcher.h — `class ORB_SLAM3::ORBmatcher` with the reference's declaration of
//   int Fuse(KeyFrame* pKF, const vector<MapPoint*>& vpMapPoints, const float th = 3.0, const bool bRight = false)
// and the added batched overload Fuse(const vector<KeyFrame*>&, const vector<MapPoint*>&, th) — against stand-ins of
// ORB_SLAM3::KeyFrame / MapPoint that implement the members Fuse reads and changes (observations, nObs with the stereo-counts-2
// rule, Replace, a real ComputeDistinctiveDescriptors, PredictScale).  The driver builds identical worlds for one scene, runs the
// reference's Fuse loop (src/ORBmatcher2.cc:420-610, restated below over the same stand-ins) key frame by key frame on the first,
// the batched overload on the second and the single-key-frame overload in a loop on the third, and compares the whole final
// state: every key frame's slots, every point's bad flag, observations, nObs and descriptor, and the return values.
//   usage: fuse_adapter_test SCENE [ref]   (SCENE = 0..5; prints "researched=<pairs> calls=<extra calls>" of the batched run;
//                                          with "ref" only the reference loop runs and its final state is printed)
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <tuple>
#include <vector>

#include <opencv2/core.hpp>

#include "orbx.h"

namespace ORB_SLAM3 {
struct Vec2 { float d[2]; float operator()(int i) const { return d[i]; } };
struct Vec3 {
    float d[3];
    float operator()(int i) const { return d[i]; }
    Vec3 operator-(const Vec3& o) const { return Vec3{{d[0] - o.d[0], d[1] - o.d[1], d[2] - o.d[2]}}; }
    float dot(const Vec3& o) const { return d[0] * o.d[0] + d[1] * o.d[1] + d[2] * o.d[2]; }
    float norm() const { return std::sqrt(dot(*this)); }
};
struct SE3f {                                     // translation-only pose: p_c = p_w - t
    float t[3] = {0, 0, 0};
    Vec3 operator*(const Vec3& p) const { return Vec3{{p.d[0] - t[0], p.d[1] - t[1], p.d[2] - t[2]}}; }
};
struct Pinhole {
    float fx = 435.f, fy = 435.f, cx = 376.f, cy = 240.f;
    Vec2 project(const Vec3& p) const { return Vec2{{fx * p(0) / p(2) + cx, fy * p(1) / p(2) + cy}}; }
};
static const std::vector<float> kScale = {1.0f, 1.2f, 1.44f, 1.728f, 2.0736f, 2.48832f, 2.985984f, 3.5831808f};

class MapPoint;
class KeyFrame {
public:
    long unsigned int mnId = 0;
    int NLeft = -1;
    std::vector<cv::KeyPoint> mvKeysUn;
    std::vector<unsigned char> descBuf;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvScaleFactors = kScale, mvInvLevelSigma2;
    float mbf = 40.f, mfLogScaleFactor = std::log(1.2f);
    int mnScaleLevels = 8;
    int mnMinX = 0, mnMinY = 0, mnMaxX = 752, mnMaxY = 480;     // KeyFrame keeps the image bounds as int
    float mfGridElementWidthInv = 64.f / 752.f, mfGridElementHeightInv = 48.f / 480.f;
    SE3f pose;
    Vec3 centre{{0, 0, 0}};
    std::map<unsigned int, std::vector<unsigned int>> mFeatVec;
    std::vector<MapPoint*> GetMapPointMatches() { return mvpMapPoints; }
    Pinhole cam;
    Pinhole* mpCamera = &cam;
    std::vector<MapPoint*> mvpMapPoints;
    KeyFrame() { for (float s : kScale) mvInvLevelSigma2.push_back(1.0f / (s * s)); }
    SE3f GetPose() const { return pose; }
    Vec3 GetCameraCenter() const { return centre; }
    bool isBad() const { return false; }
    MapPoint* GetMapPoint(const size_t& idx) { return mvpMapPoints[idx]; }
    void AddMapPoint(MapPoint* pMP, const size_t& idx) { mvpMapPoints[idx] = pMP; }
    void ReplaceMapPointMatch(const int& idx, MapPoint* pMP) { mvpMapPoints[idx] = pMP; }
    void EraseMapPointMatch(const int& idx) { mvpMapPoints[idx] = nullptr; }
};
struct ById { bool operator()(const KeyFrame* a, const KeyFrame* b) const { return a->mnId < b->mnId; } };

class MapPoint {
public:
    long unsigned int mnId = 0;
    bool mbBad = false, mbTrackInView = false;                                 // (the tracking-thread members the class reads)
    float mTrackProjX = 0, mTrackProjY = 0, mTrackProjXR = 0, mTrackViewCos = 0, mTrackDepth = 0;
    int mnTrackScaleLevel = 0;
    int nObs = 0;
    unsigned char desc[32] = {};
    Vec3 pos{{0, 0, 5}}, normal{{0, 0, 1}};
    float mfMinDistance = 0.5f, mfMaxDistance = 20.f;
    std::map<KeyFrame*, std::tuple<int, int>, ById> mObservations;
    bool isBad() { return mbBad; }
    int Observations() { return nObs; }
    bool IsInKeyFrame(KeyFrame* pKF) { return mObservations.count(pKF) > 0; }
    cv::Mat GetDescriptor() { return cv::Mat(1, 32, CV_8U, desc); }
    Vec3 GetWorldPos() { return pos; }
    Vec3 GetNormal() { return normal; }
    float GetMinDistanceInvariance() { return 0.8f * mfMinDistance; }
    float GetMaxDistanceInvariance() { return 1.2f * mfMaxDistance; }
    int PredictScale(const float& currentDist, KeyFrame* pKF)                  // MapPoint::PredictScale
    {
        const float ratio = mfMaxDistance / currentDist;
        int nScale = (int)std::ceil(std::log(ratio) / pKF->mfLogScaleFactor);
        if (nScale < 0) nScale = 0;
        else if (nScale >= pKF->mnScaleLevels) nScale = pKF->mnScaleLevels - 1;
        return nScale;
    }
    void AddObservation(KeyFrame* pKF, int idx)                                // MapPoint::AddObservation
    {
        std::tuple<int, int> indexes = mObservations.count(pKF) ? mObservations[pKF] : std::tuple<int, int>(-1, -1);
        std::get<0>(indexes) = idx;
        mObservations[pKF] = indexes;
        if (pKF->mvuRight[idx] >= 0) nObs += 2;
        else nObs++;
    }
    void ComputeDistinctiveDescriptors()                                       // MapPoint::ComputeDistinctiveDescriptors
    {
        if (mbBad) return;
        std::vector<const unsigned char*> vDescriptors;
        for (auto& o : mObservations)
            if (!o.first->isBad() && std::get<0>(o.second) != -1) vDescriptors.push_back(o.first->mDescriptors.ptr(std::get<0>(o.second)));
        if (vDescriptors.empty()) return;
        const size_t N = vDescriptors.size();
        std::vector<std::vector<int>> D(N, std::vector<int>(N, 0));
        for (size_t i = 0; i < N; i++)
            for (size_t j = i + 1; j < N; j++) D[i][j] = D[j][i] = orbx_descriptor_distance(vDescriptors[i], vDescriptors[j]);
        int BestMedian = INT_MAX, BestIdx = 0;
        for (size_t i = 0; i < N; i++) {
            std::vector<int> vDists(D[i]);
            std::sort(vDists.begin(), vDists.end());
            const int median = vDists[(size_t)(0.5 * (N - 1))];
            if (median < BestMedian) { BestMedian = median; BestIdx = (int)i; }
        }
        std::memcpy(desc, vDescriptors[BestIdx], 32);
    }
    void Replace(MapPoint* pMP)                                                // MapPoint::Replace
    {
        if (pMP->mnId == this->mnId) return;
        auto obs = mObservations;
        mObservations.clear();
        mbBad = true;
        for (auto& o : obs) {
            KeyFrame* pKF = o.first;
            const int leftIndex = std::get<0>(o.second);
            if (!pMP->IsInKeyFrame(pKF)) {
                if (leftIndex != -1) { pKF->ReplaceMapPointMatch(leftIndex, pMP); pMP->AddObservation(pKF, leftIndex); }
            } else {
                if (leftIndex != -1) pKF->EraseMapPointMatch(leftIndex);
            }
        }
        pMP->ComputeDistinctiveDescriptors();
    }
};
typedef std::map<unsigned int, std::vector<unsigned int>> FeatureVector;      // DBoW2::FeatureVector
struct SE3Frame {
    Vec3 operator*(const Vec3& p) const { return p; }
    SE3Frame inverse() const { return *this; }
    Vec3 translation() const { return Vec3{{0, 0, 0}}; }
};
class Frame {                                     // what the tracking-thread overloads of the class read (not called here)
public:
    int N = 0, Nleft = -1;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn;
    std::vector<float> mvuRight, mvScaleFactors;
    std::vector<MapPoint*> mvpMapPoints;
    std::vector<bool> mvbOutlier;
    cv::Mat mDescriptors;
    FeatureVector mFeatVec;
    float mbf = 0, mb = 0;
    Pinhole* mpCamera = nullptr;
    SE3Frame GetPose() const { return SE3Frame(); }
    static float mnMinX, mnMaxX, mnMinY, mnMaxY, mfGridElementWidthInv, mfGridElementHeightInv;
};
float Frame::mnMinX, Frame::mnMaxX, Frame::mnMinY, Frame::mnMaxY, Frame::mfGridElementWidthInv, Frame::mfGridElementHeightInv;
}  // namespace ORB_SLAM3

#include "ORBmatcher.h"

using namespace ORB_SLAM3;

// ---- the reference loop over the stand-ins (src/ORBmatcher2.cc:420-610, NLeft == -1, bRight == false) ----------------------
static int RefFuse(KeyFrame* pKF, const std::vector<MapPoint*>& vpMapPoints, const float th)
{
    const SE3f Tcw = pKF->GetPose();
    const Vec3 Ow = pKF->GetCameraCenter();
    Pinhole* pCamera = pKF->mpCamera;
    const float& bf = pKF->mbf;
    int nFused = 0;
    const int nMPs = (int)vpMapPoints.size();
    for (int i = 0; i < nMPs; i++) {
        MapPoint* pMP = vpMapPoints[i];
        if (!pMP) continue;
        if (pMP->isBad()) continue;
        else if (pMP->IsInKeyFrame(pKF)) continue;
        Vec3 p3Dw = pMP->GetWorldPos();
        Vec3 p3Dc = Tcw * p3Dw;
        if (p3Dc(2) < 0.0f) continue;
        const float invz = 1 / p3Dc(2);
        const Vec2 uv = pCamera->project(p3Dc);
        const float x = uv(0), y = uv(1);
        if (!(x >= pKF->mnMinX && x < pKF->mnMaxX && y >= pKF->mnMinY && y < pKF->mnMaxY)) continue;   // KeyFrame::IsInImage
        const float ur = uv(0) - bf * invz;
        const float maxDistance = pMP->GetMaxDistanceInvariance();
        const float minDistance = pMP->GetMinDistanceInvariance();
        Vec3 PO = p3Dw - Ow;
        const float dist3D = PO.norm();
        if (dist3D < minDistance || dist3D > maxDistance) continue;
        Vec3 Pn = pMP->GetNormal();
        if (PO.dot(Pn) < 0.5 * dist3D) continue;
        int nPredictedLevel = pMP->PredictScale(dist3D, pKF);
        const float radius = th * pKF->mvScaleFactors[nPredictedLevel];
        // KeyFrame::GetFeaturesInArea (the grid: Frame::AssignFeaturesToGrid, then cell column, cell row, index)
        std::vector<size_t> vIndices;
        {
            const float r = radius;
            const int nMinCellX = std::max(0, (int)floor((x - pKF->mnMinX - r) * pKF->mfGridElementWidthInv));
            const int nMaxCellX = std::min(63, (int)ceil((x - pKF->mnMinX + r) * pKF->mfGridElementWidthInv));
            const int nMinCellY = std::max(0, (int)floor((y - pKF->mnMinY - r) * pKF->mfGridElementHeightInv));
            const int nMaxCellY = std::min(47, (int)ceil((y - pKF->mnMinY + r) * pKF->mfGridElementHeightInv));
            if (nMinCellX < 64 && nMaxCellX >= 0 && nMinCellY < 48 && nMaxCellY >= 0)
                for (int ix = nMinCellX; ix <= nMaxCellX; ix++)
                    for (int iy = nMinCellY; iy <= nMaxCellY; iy++)
                        for (size_t j = 0; j < pKF->mvKeysUn.size(); j++) {
                            const cv::KeyPoint& kp = pKF->mvKeysUn[j];
                            const int px = (int)round((kp.pt.x - pKF->mnMinX) * pKF->mfGridElementWidthInv);
                            const int py = (int)round((kp.pt.y - pKF->mnMinY) * pKF->mfGridElementHeightInv);
                            if (px != ix || py != iy) continue;
                            if (fabs(kp.pt.x - x) < r && fabs(kp.pt.y - y) < r) vIndices.push_back(j);
                        }
        }
        if (vIndices.empty()) continue;
        int bestDist = 256, bestIdx = -1;
        for (size_t idx : vIndices) {
            const cv::KeyPoint& kp = pKF->mvKeysUn[idx];
            const int& kpLevel = kp.octave;
            if (kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel) continue;
            if (pKF->mvuRight[idx] >= 0) {
                const float ex = uv(0) - kp.pt.x, ey = uv(1) - kp.pt.y, er = ur - pKF->mvuRight[idx];
                const float e2 = ex * ex + ey * ey + er * er;
                if (e2 * pKF->mvInvLevelSigma2[kpLevel] > 7.8) continue;
            } else {
                const float ex = uv(0) - kp.pt.x, ey = uv(1) - kp.pt.y;
                const float e2 = ex * ex + ey * ey;
                if (e2 * pKF->mvInvLevelSigma2[kpLevel] > 5.99) continue;
            }
            const int dist = orbx_descriptor_distance(pMP->desc, pKF->mDescriptors.ptr((int)idx));
            if (dist < bestDist) { bestDist = dist; bestIdx = (int)idx; }
        }
        if (bestDist <= ORBmatcher::TH_LOW) {
            MapPoint* pMPinKF = pKF->GetMapPoint(bestIdx);
            if (pMPinKF) {
                if (!pMPinKF->isBad()) {
                    if (pMPinKF->Observations() > pMP->Observations()) pMP->Replace(pMPinKF);
                    else pMPinKF->Replace(pMP);
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

// ---- worlds --------------------------------------------------------------------------------------------------------------
struct World {
    std::vector<std::unique_ptr<KeyFrame>> kfs;
    std::vector<std::unique_ptr<MapPoint>> mps;
    std::vector<KeyFrame*> targets;        // the key frames Fuse runs on, in order
    std::vector<MapPoint*> points;         // vpMapPoints (may hold NULL and duplicates)
    float th = 3.0f;
};

static void flip(unsigned char* d, int b0, int b1) { for (int b = b0; b < b1; ++b) d[b >> 3] ^= (unsigned char)(1u << (b & 7)); }

struct Builder {
    World& W;
    unsigned char base[32];
    explicit Builder(World& w, unsigned seed) : W(w) { for (int i = 0; i < 32; ++i) base[i] = (unsigned char)((seed * 131u + i * 29u) & 0xff); }
    // descriptor = base with bit ranges flipped
    void desc(unsigned char* d, std::initializer_list<std::pair<int, int>> ranges) { std::memcpy(d, base, 32); for (auto r : ranges) flip(d, r.first, r.second); }
    KeyFrame* kf(float tx, bool stereo)
    {
        W.kfs.emplace_back(new KeyFrame());
        KeyFrame* K = W.kfs.back().get();
        K->mnId = W.kfs.size() - 1;
        K->pose.t[0] = tx; K->centre = Vec3{{tx, 0, 0}};
        K->mvuRight.clear();
        (void)stereo;
        return K;
    }
    MapPoint* mp(float x, float y, float z, std::initializer_list<std::pair<int, int>> d)
    {
        W.mps.emplace_back(new MapPoint());
        MapPoint* P = W.mps.back().get();
        P->mnId = W.mps.size() - 1;
        P->pos = Vec3{{x, y, z}};
        desc(P->desc, d);
        return P;
    }
    // a feature of K at the projection of P (+ dx), level = P's predicted level in K, descriptor from ranges
    int feature(KeyFrame* K, MapPoint* P, float dx, std::initializer_list<std::pair<int, int>> d, bool stereo, int level = -1)
    {
        const Vec3 pc = K->pose * P->pos;
        const Vec2 uv = K->mpCamera->project(pc);
        cv::KeyPoint kp{};
        kp.pt.x = uv(0) + dx; kp.pt.y = uv(1);
        kp.octave = level >= 0 ? level : P->PredictScale((P->pos - K->centre).norm(), K);
        kp.size = 31.f; kp.class_id = -1;
        K->mvKeysUn.push_back(kp);
        K->mvuRight.push_back(stereo ? kp.pt.x - K->mbf / pc(2) : -1.0f);
        const size_t n = K->descBuf.size();
        K->descBuf.resize(n + 32);
        desc(&K->descBuf[n], d);
        K->mvpMapPoints.push_back(nullptr);
        return (int)K->mvKeysUn.size() - 1;
    }
    void observe(MapPoint* P, KeyFrame* K, int idx) { P->AddObservation(K, idx); K->mvpMapPoints[idx] = P; }
    void seal() { for (auto& K : W.kfs) K->mDescriptors = cv::Mat((int)K->mvKeysUn.size(), 32, CV_8U, K->descBuf.data()); }
};

static void build(World& W, int scene)
{
    Builder B(W, 7u + scene);
    switch (scene) {
    case 0: {   // two points on one empty slot; both Replace directions; the observation-count tie
        KeyFrame* A = B.kf(0.f, true); KeyFrame* O = B.kf(0.3f, false);
        MapPoint* p0 = B.mp(0.0f, 0.0f, 5.f, {{0, 10}}); MapPoint* p1 = B.mp(0.01f, 0.0f, 5.f, {{0, 12}});
        B.feature(A, p0, 0.2f, {{0, 11}}, true);                                       // p0 takes it, p1 then meets p0 in the slot
        MapPoint* q = B.mp(1.f, 0.5f, 6.f, {{40, 50}}); MapPoint* p2 = B.mp(1.f, 0.5f, 6.f, {{40, 52}});   // slot q (3 obs) > p2 (1)
        int f = B.feature(A, q, 0.f, {{40, 51}}, false); int g = B.feature(O, q, 0.f, {{40, 49}}, true);
        MapPoint* r = B.mp(-1.f, -0.5f, 7.f, {{60, 70}}); MapPoint* p3 = B.mp(-1.f, -0.5f, 7.f, {{60, 72}});  // slot r (1) < p3 (2)
        int f2 = B.feature(A, r, 0.f, {{60, 71}}, false); int g2 = B.feature(O, p3, 0.f, {{60, 73}}, true);
        MapPoint* s = B.mp(0.5f, -1.f, 8.f, {{80, 90}}); MapPoint* p4 = B.mp(0.5f, -1.f, 8.f, {{80, 92}});   // tie 2 = 2: s->Replace(p4)
        int f3 = B.feature(A, s, 0.f, {{80, 91}}, true); int g3 = B.feature(O, p4, 0.f, {{80, 93}}, true);
        B.seal();
        B.observe(q, A, f); B.observe(q, O, g); B.observe(r, A, f2); B.observe(p3, O, g2); B.observe(s, A, f3); B.observe(p4, O, g3);
        W.targets = {A}; W.points = {p0, p1, p2, p3, p4, nullptr};
        break;
    }
    case 1: {   // the slot holds a bad point: nothing changes, nFused still counts
        KeyFrame* A = B.kf(0.f, false);
        MapPoint* z = B.mp(0.f, 0.f, 5.f, {{0, 5}}); MapPoint* p = B.mp(0.f, 0.f, 5.f, {{0, 6}});
        int f = B.feature(A, z, 0.f, {{0, 7}}, false);
        B.seal(); B.observe(z, A, f); z->mbBad = true;
        W.targets = {A}; W.points = {p};
        break;
    }
    case 2: {   // a point replaced in A (the slot's point has more observations) and then skipped in B
        KeyFrame* A = B.kf(0.f, true); KeyFrame* Bk = B.kf(0.2f, true); KeyFrame* O = B.kf(-0.2f, true);
        MapPoint* m = B.mp(0.f, 0.f, 5.f, {{0, 5}}); MapPoint* p = B.mp(0.f, 0.f, 5.f, {{0, 8}});
        int f = B.feature(A, m, 0.f, {{0, 6}}, true); int g = B.feature(O, m, 0.f, {{0, 4}}, true);
        B.feature(Bk, p, 0.3f, {{0, 9}}, true);
        B.seal(); B.observe(m, A, f); B.observe(m, O, g);
        W.targets = {A, Bk}; W.points = {p};
        break;
    }
    case 3: {   // p survives in A (tie: the slot's point is replaced), takes a new descriptor that matches a different feature in B
        KeyFrame* C = B.kf(-0.3f, false); KeyFrame* C2 = B.kf(-0.4f, false); KeyFrame* A = B.kf(0.f, false); KeyFrame* Bk = B.kf(0.25f, false);
        KeyFrame* D = B.kf(0.35f, false);
        MapPoint* p = B.mp(0.f, 0.f, 5.f, {});                              // Dp = base
        MapPoint* m = B.mp(0.f, 0.f, 5.f, {{0, 40}});                       // Dm = bits [0, 40)
        int c = B.feature(C, p, 0.f, {}, false); int c2 = B.feature(C2, p, 0.f, {{0, 38}}, false);
        int a = B.feature(A, m, 0.f, {{0, 40}}, false); int d = B.feature(D, m, 0.f, {{0, 40}}, false);
        B.feature(Bk, p, 0.3f, {{100, 130}}, false);                        // g1: 30 from Dp, 70 from Dm
        B.feature(Bk, p, -0.3f, {{0, 40}, {200, 210}}, false);              // g2: 50 from Dp, 10 from Dm
        B.seal();
        B.observe(p, C, c); B.observe(p, C2, c2); B.observe(m, A, a); B.observe(m, D, d);
        W.targets = {A, Bk}; W.points = {p};
        break;
    }
    case 4: {   // p gains an observation of B through Replace, so B skips it
        KeyFrame* A = B.kf(0.f, true); KeyFrame* Bk = B.kf(0.2f, true);
        MapPoint* m = B.mp(0.f, 0.f, 5.f, {{0, 5}}); MapPoint* p = B.mp(0.f, 0.f, 5.f, {{0, 7}});
        int a = B.feature(A, m, 0.f, {{0, 6}}, false); int b = B.feature(Bk, m, 0.f, {{0, 5}}, false);
        B.feature(Bk, p, 0.4f, {{0, 7}}, false);
        B.seal(); B.observe(m, A, a); B.observe(m, Bk, b); p->nObs = 5;    // p outnumbers m: m->Replace(p) moves B's slot to p
        W.targets = {A, Bk}; W.points = {p};
        break;
    }
    case 5: {   // vpMapPoints holds p twice; A's slot holds m, which does not observe A: the in-loop check re-searches
        KeyFrame* A = B.kf(0.f, false); KeyFrame* D = B.kf(0.3f, false); KeyFrame* D2 = B.kf(0.4f, false);
        MapPoint* p = B.mp(0.f, 0.f, 5.f, {});
        MapPoint* m = B.mp(0.f, 0.f, 5.f, {{0, 30}});
        int a = B.feature(A, p, 0.f, {{0, 20}}, false);
        B.feature(A, p, 0.5f, {{0, 30}, {120, 130}}, false);               // 30 from Dp (loses to a at 20), 10 from Dm
        int d = B.feature(D, m, 0.f, {{0, 30}}, false); int d2 = B.feature(D2, m, 0.f, {{0, 30}}, false);
        B.seal();
        A->mvpMapPoints[a] = m;                                            // slot without an observation of A
        B.observe(m, D, d); B.observe(m, D2, d2);
        p->nObs = 2;                                                        // tie with m: m->Replace(p), p takes Dm
        W.targets = {A}; W.points = {p, p};
        break;
    }
    default: std::fprintf(stderr, "unknown scene %d\n", scene); std::exit(2);
    }
}

static bool same_state(World& X, World& Y, const char* what)
{
    bool ok = true;
    for (size_t k = 0; k < X.kfs.size(); ++k)
        for (size_t j = 0; j < X.kfs[k]->mvpMapPoints.size(); ++j) {
            MapPoint* a = X.kfs[k]->mvpMapPoints[j]; MapPoint* b = Y.kfs[k]->mvpMapPoints[j];
            if ((a ? (long)a->mnId : -1L) != (b ? (long)b->mnId : -1L)) { std::printf("%s: key frame %zu slot %zu differs\n", what, k, j); ok = false; }
        }
    for (size_t i = 0; i < X.mps.size(); ++i) {
        MapPoint* a = X.mps[i].get(); MapPoint* b = Y.mps[i].get();
        if (a->mbBad != b->mbBad || a->nObs != b->nObs || std::memcmp(a->desc, b->desc, 32) != 0) { std::printf("%s: point %zu differs\n", what, i); ok = false; }
        std::vector<std::pair<long, int>> oa, ob;
        for (auto& o : a->mObservations) oa.push_back({(long)o.first->mnId, std::get<0>(o.second)});
        for (auto& o : b->mObservations) ob.push_back({(long)o.first->mnId, std::get<0>(o.second)});
        if (oa != ob) { std::printf("%s: point %zu observations differ\n", what, i); ok = false; }
    }
    return ok;
}

int main(int argc, char** argv)
{
    if (argc < 2) { std::fprintf(stderr, "usage: %s SCENE\n", argv[0]); return 2; }
    const int scene = std::atoi(argv[1]);
    World R, G, S;
    build(R, scene); build(G, scene); build(S, scene);
    int nRef = 0;
    for (KeyFrame* K : R.targets) nRef += RefFuse(K, R.points, R.th);
    if (argc > 2) {                               // "ref": the reference run alone (no device needed), its final state printed
        std::printf("scene %d: nFused ref=%d\n", scene, nRef);
        for (auto& p : R.mps) {
            std::printf("point %lu bad=%d nObs=%d obs:", p->mnId, (int)p->mbBad, p->nObs);
            for (auto& o : p->mObservations) std::printf(" kf%lu/%d", o.first->mnId, std::get<0>(o.second));
            std::printf(" desc0=%02x%02x%02x%02x%02x\n", p->desc[0], p->desc[1], p->desc[2], p->desc[3], p->desc[15]);
        }
        return 0;
    }
    ORBmatcher matcher;
    const int nBatch = matcher.Fuse(G.targets, G.points, G.th);
    const orbx_adapter::FuseDiagnostics diag = orbx_adapter::fuse_diagnostics;
    int nSingle = 0;
    for (KeyFrame* K : S.targets) nSingle += matcher.Fuse(K, S.points, S.th);
    std::printf("scene %d: nFused ref=%d batched=%d single=%d researched=%d calls=%d\n", scene, nRef, nBatch, nSingle, diag.researched_pairs,
                diag.extra_calls);
    bool ok = nRef == nBatch && nRef == nSingle;
    ok = same_state(R, G, "batched") && ok;
    ok = same_state(R, S, "single") && ok;
    // the reference itself: the scene does what it says
    std::printf("bad:");
    for (auto& p : R.mps) std::printf(" %d", (int)p->mbBad);
    std::printf("\n");
    bool threw = false;
    try { matcher.Fuse(S.targets[0], S.points, 3.0f, true); } catch (const std::invalid_argument&) { threw = true; }
    ok = ok && threw;
    std::printf(ok ? "OK\n" : "MISMATCH\n");
    return ok ? 0 : 1;
}
