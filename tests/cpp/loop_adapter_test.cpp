// Compiles csrc/adapter/ORBmatcher.h — `class ORB_SLAM3::ORBmatcher` with the reference's declarations of the loop-closing searches
//   int SearchByProjection(KeyFrame*, Sim3f& Scw, vpPoints, [vpPointsKFs,] vpMatched, [vpMatchedKF,] int th, float ratioHamming)
//   int Fuse(KeyFrame* pKF, Sim3f& Scw, const vector<MapPoint*>& vpPoints, float th, vector<MapPoint*>& vpReplacePoint)
// and the added SearchAndFuse(vector<KeyFrame*>, vector<Sim3f>, vector<MapPoint*>, th) — against stand-ins of its own: a Sim3
// with rotationMatrix / translation / scale, an SE3 built from (R, t), a Map holding mMutexMapUpdate, and KeyFrame / MapPoint
// with the members the searches and MapPoint::Replace read and change (GetMapPoints, GetMap, observations, nObs, a real
// ComputeDistinctiveDescriptors, PredictScale).  The reference loops (upstream ORB-SLAM3 v1.0: src/ORBmatcher1.cc:429-648,
// src/ORBmatcher2.cc:612-729, the loop body of LoopClosing::SearchAndFuse) are restated below over the same stand-ins.
//   usage: loop_adapter_test SCENE [ref]   SCENE 0..5: SearchAndFuse.  Builds three identical worlds and runs the reference
//            loop on the first, the batched SearchAndFuse on the second and the single-key-frame Sim3 Fuse in the reference's
//            loop on the third, then compares the whole final state; prints "researched=<pairs> calls=<extra calls>" of the
//            batched run.  SCENE 6: both SearchByProjection overloads against the reference loop, vpMatched and vpMatchedKF.
//            With "ref" only the reference runs (no device needed) and its final state is printed.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <set>
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
    Vec3 operator+(const Vec3& o) const { return Vec3{{d[0] + o.d[0], d[1] + o.d[1], d[2] + o.d[2]}}; }
    Vec3 operator/(float s) const { return Vec3{{d[0] / s, d[1] / s, d[2] / s}}; }
    float dot(const Vec3& o) const { return d[0] * o.d[0] + d[1] * o.d[1] + d[2] * o.d[2]; }
    float norm() const { return std::sqrt(dot(*this)); }
};
struct Mat3 {
    float m[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
    Vec3 operator*(const Vec3& p) const
    {
        return Vec3{{m[0] * p.d[0] + m[1] * p.d[1] + m[2] * p.d[2], m[3] * p.d[0] + m[4] * p.d[1] + m[5] * p.d[2],
                     m[6] * p.d[0] + m[7] * p.d[1] + m[8] * p.d[2]}};
    }
    Mat3 transpose() const { Mat3 r; for (int i = 0; i < 3; ++i) for (int j = 0; j < 3; ++j) r.m[3 * i + j] = m[3 * j + i]; return r; }
};
struct SE3f {                                     // p_c = R p_w + t
    Mat3 R;
    Vec3 t{{0, 0, 0}};
    SE3f() = default;
    SE3f(const Mat3& r, const Vec3& tr) : R(r), t(tr) {}
    Vec3 operator*(const Vec3& p) const { return R * p + t; }
    SE3f inverse() const { const Mat3 Rt = R.transpose(); const Vec3 c = Rt * t; return SE3f(Rt, Vec3{{-c.d[0], -c.d[1], -c.d[2]}}); }
    Vec3 translation() const { return t; }
};
struct Sim3f {                                    // Sophus::Sim3f: p_c = s R p_w + t
    Mat3 R;
    Vec3 t{{0, 0, 0}};
    float s = 1.f;
    Mat3 rotationMatrix() const { return R; }
    Vec3 translation() const { return t; }
    float scale() const { return s; }
};
struct Pinhole {
    float fx = 435.f, fy = 435.f, cx = 376.f, cy = 240.f;
    Vec2 project(const Vec3& p) const { return Vec2{{fx * p(0) / p(2) + cx, fy * p(1) / p(2) + cy}}; }
};
static const std::vector<float> kScale = {1.0f, 1.2f, 1.44f, 1.728f, 2.0736f, 2.48832f, 2.985984f, 3.5831808f};

struct Map { std::mutex mMutexMapUpdate; };

class MapPoint;
class KeyFrame {
public:
    long unsigned int mnId = 0;
    int N = 0, NLeft = -1;
    std::vector<cv::KeyPoint> mvKeysUn;
    std::vector<unsigned char> descBuf;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvScaleFactors = kScale, mvInvLevelSigma2;
    float mbf = 40.f, mfLogScaleFactor = std::log(1.2f);
    int mnScaleLevels = 8;
    int mnMinX = 0, mnMinY = 0, mnMaxX = 752, mnMaxY = 480;
    float mfGridElementWidthInv = 64.f / 752.f, mfGridElementHeightInv = 48.f / 480.f;
    SE3f pose;                                    // the corrected pose the scene's Sim3 decomposes to
    Map* mpMap = nullptr;
    std::map<unsigned int, std::vector<unsigned int>> mFeatVec;
    std::vector<MapPoint*> GetMapPointMatches() { return mvpMapPoints; }
    Pinhole cam;
    Pinhole* mpCamera = &cam;
    std::vector<MapPoint*> mvpMapPoints;
    KeyFrame() { for (float s : kScale) mvInvLevelSigma2.push_back(1.0f / (s * s)); }
    SE3f GetPose() const { return pose; }
    Map* GetMap() { return mpMap; }
    bool isBad() const { return false; }
    std::set<MapPoint*> GetMapPoints();           // KeyFrame::GetMapPoints: the non-NULL, non-bad slots
    MapPoint* GetMapPoint(const size_t& idx) { return mvpMapPoints[idx]; }
    void AddMapPoint(MapPoint* pMP, const size_t& idx) { mvpMapPoints[idx] = pMP; }
    void ReplaceMapPointMatch(const int& idx, MapPoint* pMP) { mvpMapPoints[idx] = pMP; }
    void EraseMapPointMatch(const int& idx) { mvpMapPoints[idx] = nullptr; }
};
struct ById { bool operator()(const KeyFrame* a, const KeyFrame* b) const { return a->mnId < b->mnId; } };

class MapPoint {
public:
    long unsigned int mnId = 0;
    bool mbBad = false, mbTrackInView = false;
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
    int PredictScale(const float& currentDist, KeyFrame* pKF)
    {
        const float ratio = mfMaxDistance / currentDist;
        int nScale = (int)std::ceil(std::log(ratio) / pKF->mfLogScaleFactor);
        if (nScale < 0) nScale = 0;
        else if (nScale >= pKF->mnScaleLevels) nScale = pKF->mnScaleLevels - 1;
        return nScale;
    }
    void AddObservation(KeyFrame* pKF, int idx)
    {
        std::tuple<int, int> indexes = mObservations.count(pKF) ? mObservations[pKF] : std::tuple<int, int>(-1, -1);
        std::get<0>(indexes) = idx;
        mObservations[pKF] = indexes;
        if (pKF->mvuRight[idx] >= 0) nObs += 2;
        else nObs++;
    }
    void ComputeDistinctiveDescriptors()
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
    void Replace(MapPoint* pMP)                   // MapPoint::Replace
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
std::set<MapPoint*> KeyFrame::GetMapPoints()
{
    std::set<MapPoint*> s;
    for (MapPoint* p : mvpMapPoints)
        if (p && !p->isBad()) s.insert(p);
    return s;
}
typedef std::map<unsigned int, std::vector<unsigned int>> FeatureVector;
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
    SE3f GetPose() const { return SE3f(); }
    static float mnMinX, mnMaxX, mnMinY, mnMaxY, mfGridElementWidthInv, mfGridElementHeightInv;
};
float Frame::mnMinX, Frame::mnMaxX, Frame::mnMinY, Frame::mnMaxY, Frame::mfGridElementWidthInv, Frame::mfGridElementHeightInv;
}  // namespace ORB_SLAM3

#include "ORBmatcher.h"

using namespace ORB_SLAM3;

// ---- the reference loops over the stand-ins ---------------------------------------------------------------------------------
// KeyFrame::GetFeaturesInArea(x, y, r): cells of Frame::AssignFeaturesToGrid in (column, row) order, the cell's index order.
static std::vector<size_t> GetFeaturesInArea(KeyFrame* pKF, float x, float y, float r)
{
    std::vector<size_t> vIndices;
    const int nMinCellX = std::max(0, (int)floor((x - pKF->mnMinX - r) * pKF->mfGridElementWidthInv));
    const int nMaxCellX = std::min(63, (int)ceil((x - pKF->mnMinX + r) * pKF->mfGridElementWidthInv));
    const int nMinCellY = std::max(0, (int)floor((y - pKF->mnMinY - r) * pKF->mfGridElementHeightInv));
    const int nMaxCellY = std::min(47, (int)ceil((y - pKF->mnMinY + r) * pKF->mfGridElementHeightInv));
    if (nMinCellX >= 64 || nMaxCellX < 0 || nMinCellY >= 48 || nMaxCellY < 0) return vIndices;
    for (int ix = nMinCellX; ix <= nMaxCellX; ix++)
        for (int iy = nMinCellY; iy <= nMaxCellY; iy++)
            for (size_t j = 0; j < pKF->mvKeysUn.size(); j++) {
                const cv::KeyPoint& kp = pKF->mvKeysUn[j];
                const int px = (int)round((kp.pt.x - pKF->mnMinX) * pKF->mfGridElementWidthInv);
                const int py = (int)round((kp.pt.y - pKF->mnMinY) * pKF->mfGridElementHeightInv);
                if (px != ix || py != iy) continue;
                if (fabs(kp.pt.x - x) < r && fabs(kp.pt.y - y) < r) vIndices.push_back(j);
            }
    return vIndices;
}
static bool IsInImage(KeyFrame* pKF, float x, float y) { return x >= pKF->mnMinX && x < pKF->mnMaxX && y >= pKF->mnMinY && y < pKF->mnMaxY; }

// SearchByProjection(pKF, Scw, vpPoints, vpPointsKFs, vpMatched, vpMatchedKF, th, ratioHamming) — src/ORBmatcher1.cc:429-648
// (vpPointsKFs / vpMatchedKF null: the first overload)
static int RefSearchByProjection(KeyFrame* pKF, Sim3f& Scw, const std::vector<MapPoint*>& vpPoints, const std::vector<KeyFrame*>* vpPointsKFs,
                                 std::vector<MapPoint*>& vpMatched, std::vector<KeyFrame*>* vpMatchedKF, int th, float ratioHamming)
{
    SE3f Tcw = SE3f(Scw.rotationMatrix(), Scw.translation() / Scw.scale());
    Vec3 Ow = Tcw.inverse().translation();
    std::set<MapPoint*> spAlreadyFound(vpMatched.begin(), vpMatched.end());
    spAlreadyFound.erase(static_cast<MapPoint*>(NULL));
    int nmatches = 0;
    for (int iMP = 0, iendMP = (int)vpPoints.size(); iMP < iendMP; iMP++) {
        MapPoint* pMP = vpPoints[iMP];
        if (!pMP) continue;                       // (the reference dereferences NULL; the scenes hold one)
        if (pMP->isBad() || spAlreadyFound.count(pMP)) continue;
        Vec3 p3Dw = pMP->GetWorldPos();
        Vec3 p3Dc = Tcw * p3Dw;
        if (p3Dc(2) < 0.0) continue;
        const Vec2 uv = pKF->mpCamera->project(p3Dc);
        if (!IsInImage(pKF, uv(0), uv(1))) continue;
        const float maxDistance = pMP->GetMaxDistanceInvariance();
        const float minDistance = pMP->GetMinDistanceInvariance();
        Vec3 PO = p3Dw - Ow;
        const float dist = PO.norm();
        if (dist < minDistance || dist > maxDistance) continue;
        Vec3 Pn = pMP->GetNormal();
        if (PO.dot(Pn) < 0.5 * dist) continue;
        int nPredictedLevel = pMP->PredictScale(dist, pKF);
        const float radius = th * pKF->mvScaleFactors[nPredictedLevel];
        const std::vector<size_t> vIndices = GetFeaturesInArea(pKF, uv(0), uv(1), radius);
        if (vIndices.empty()) continue;
        int bestDist = 256;
        int bestIdx = -1;
        for (size_t idx : vIndices) {
            if (vpMatched[idx]) continue;
            const int& kpLevel = pKF->mvKeysUn[idx].octave;
            if (kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel) continue;
            const int dist = orbx_descriptor_distance(pMP->desc, pKF->mDescriptors.ptr((int)idx));
            if (dist < bestDist) { bestDist = dist; bestIdx = (int)idx; }
        }
        if (bestDist <= ORBmatcher::TH_LOW * ratioHamming) {
            vpMatched[bestIdx] = pMP;
            if (vpMatchedKF) (*vpMatchedKF)[bestIdx] = (*vpPointsKFs)[iMP];
            nmatches++;
        }
    }
    return nmatches;
}

// Fuse(pKF, Scw, vpPoints, th, vpReplacePoint) — src/ORBmatcher2.cc:612-729
static int RefFuse(KeyFrame* pKF, Sim3f& Scw, const std::vector<MapPoint*>& vpPoints, float th, std::vector<MapPoint*>& vpReplacePoint)
{
    SE3f Tcw = SE3f(Scw.rotationMatrix(), Scw.translation() / Scw.scale());
    Vec3 Ow = Tcw.inverse().translation();
    const std::set<MapPoint*> spAlreadyFound = pKF->GetMapPoints();
    int nFused = 0;
    const int nPoints = (int)vpPoints.size();
    for (int iMP = 0; iMP < nPoints; iMP++) {
        MapPoint* pMP = vpPoints[iMP];
        if (pMP->isBad() || spAlreadyFound.count(pMP)) continue;
        Vec3 p3Dw = pMP->GetWorldPos();
        Vec3 p3Dc = Tcw * p3Dw;
        if (p3Dc(2) < 0.0f) continue;
        const Vec2 uv = pKF->mpCamera->project(p3Dc);
        if (!IsInImage(pKF, uv(0), uv(1))) continue;
        const float maxDistance = pMP->GetMaxDistanceInvariance();
        const float minDistance = pMP->GetMinDistanceInvariance();
        Vec3 PO = p3Dw - Ow;
        const float dist3D = PO.norm();
        if (dist3D < minDistance || dist3D > maxDistance) continue;
        Vec3 Pn = pMP->GetNormal();
        if (PO.dot(Pn) < 0.5 * dist3D) continue;
        const int nPredictedLevel = pMP->PredictScale(dist3D, pKF);
        const float radius = th * pKF->mvScaleFactors[nPredictedLevel];
        const std::vector<size_t> vIndices = GetFeaturesInArea(pKF, uv(0), uv(1), radius);
        if (vIndices.empty()) continue;
        int bestDist = INT_MAX;
        int bestIdx = -1;
        for (size_t idx : vIndices) {
            const int& kpLevel = pKF->mvKeysUn[idx].octave;
            if (kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel) continue;
            int dist = orbx_descriptor_distance(pMP->desc, pKF->mDescriptors.ptr((int)idx));
            if (dist < bestDist) { bestDist = dist; bestIdx = (int)idx; }
        }
        if (bestDist <= ORBmatcher::TH_LOW) {
            MapPoint* pMPinKF = pKF->GetMapPoint(bestIdx);
            if (pMPinKF) {
                if (!pMPinKF->isBad()) vpReplacePoint[iMP] = pMPinKF;
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
    std::vector<KeyFrame*> targets;        // the corrected key frames, in order
    std::vector<Sim3f> scw;                // their Sim3
    std::vector<MapPoint*> points;         // vpMapPoints / vpPoints (may hold NULL and duplicates)
    std::vector<KeyFrame*> pointKFs;       // vpPointsKFs (scene 6)
    std::vector<MapPoint*> matched;        // vpMatched on entry (scene 6)
    Map map;
};

// The loop body of LoopClosing::SearchAndFuse (both overloads), with the Fuse given.
template <class FuseFn>
static int SearchAndFuseLoop(World& W, FuseFn fuse)
{
    int total = 0;
    for (size_t k = 0; k < W.targets.size(); ++k) {
        KeyFrame* pKFi = W.targets[k];
        Map* pMap = pKFi->GetMap();
        std::vector<MapPoint*> vpReplacePoints(W.points.size(), static_cast<MapPoint*>(NULL));
        total += fuse(pKFi, W.scw[k], W.points, 4.f, vpReplacePoints);
        std::unique_lock<std::mutex> lock(pMap->mMutexMapUpdate);
        const int nLP = (int)W.points.size();
        for (int i = 0; i < nLP; i++) {
            MapPoint* pRep = vpReplacePoints[i];
            if (pRep) pRep->Replace(W.points[i]);
        }
    }
    return total;
}

static void flip(unsigned char* d, int b0, int b1) { for (int b = b0; b < b1; ++b) d[b >> 3] ^= (unsigned char)(1u << (b & 7)); }

struct Builder {
    World& W;
    unsigned char base[32];
    explicit Builder(World& w, unsigned seed) : W(w) { for (int i = 0; i < 32; ++i) base[i] = (unsigned char)((seed * 131u + i * 29u) & 0xff); }
    void desc(unsigned char* d, std::initializer_list<std::pair<int, int>> ranges) { std::memcpy(d, base, 32); for (auto r : ranges) flip(d, r.first, r.second); }
    // a key frame whose corrected pose is a translation by -tx, given as a Sim3 of scale 2 (t / s is exact)
    KeyFrame* kf(float tx, bool target)
    {
        W.kfs.emplace_back(new KeyFrame());
        KeyFrame* K = W.kfs.back().get();
        K->mnId = W.kfs.size() - 1;
        K->pose.t = Vec3{{-tx, 0, 0}};
        K->mpMap = &W.map;
        if (target) {
            Sim3f S;
            S.s = 2.f; S.t = Vec3{{-2.f * tx, 0, 0}};
            W.targets.push_back(K); W.scw.push_back(S);
        }
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
    int feature(KeyFrame* K, MapPoint* P, float dx, std::initializer_list<std::pair<int, int>> d)
    {
        const Vec3 pc = K->pose * P->pos;
        const Vec2 uv = K->mpCamera->project(pc);
        cv::KeyPoint kp{};
        kp.pt.x = uv(0) + dx; kp.pt.y = uv(1);
        kp.octave = P->PredictScale((P->pos - K->pose.inverse().translation()).norm(), K);
        kp.size = 31.f; kp.class_id = -1;
        K->mvKeysUn.push_back(kp);
        K->mvuRight.push_back(-1.0f);
        const size_t n = K->descBuf.size();
        K->descBuf.resize(n + 32);
        desc(&K->descBuf[n], d);
        K->mvpMapPoints.push_back(nullptr);
        K->N = (int)K->mvKeysUn.size();
        return K->N - 1;
    }
    void observe(MapPoint* P, KeyFrame* K, int idx) { P->AddObservation(K, idx); K->mvpMapPoints[idx] = P; }
    void seal() { for (auto& K : W.kfs) K->mDescriptors = cv::Mat((int)K->mvKeysUn.size(), 32, CV_8U, K->descBuf.data()); }
};

static void build(World& W, int scene)
{
    Builder B(W, 11u + scene);
    switch (scene) {
    case 0: {   // p survives the Replace loop of A with m's descriptor, which matches a different feature of Bk
        KeyFrame* C = B.kf(-0.3f, false); KeyFrame* C2 = B.kf(-0.4f, false); KeyFrame* A = B.kf(0.f, true); KeyFrame* Bk = B.kf(0.25f, true);
        KeyFrame* D = B.kf(0.35f, false);
        MapPoint* p = B.mp(0.f, 0.f, 5.f, {});                              // Dp = base
        MapPoint* m = B.mp(0.f, 0.f, 5.f, {{0, 40}});                       // Dm = bits [0, 40)
        int c = B.feature(C, p, 0.f, {}); int c2 = B.feature(C2, p, 0.f, {{0, 38}});
        int a = B.feature(A, m, 0.f, {{0, 40}}); int d = B.feature(D, m, 0.f, {{0, 40}});
        B.feature(Bk, p, 0.3f, {{100, 130}});                               // g1: 30 from Dp, 70 from Dm
        B.feature(Bk, p, -0.3f, {{0, 40}, {200, 210}});                     // g2: 50 from Dp, 10 from Dm
        B.seal();
        B.observe(p, C, c); B.observe(p, C2, c2); B.observe(m, A, a); B.observe(m, D, d);
        W.points = {p};
        break;
    }
    case 1: {   // p takes over m's slots in A and Bk through the Replace loop of A, so Bk's snapshot holds p and skips it
        KeyFrame* A = B.kf(0.f, true); KeyFrame* Bk = B.kf(0.2f, true);
        MapPoint* m = B.mp(0.f, 0.f, 5.f, {{0, 5}}); MapPoint* p = B.mp(0.f, 0.f, 5.f, {});
        int a = B.feature(A, m, 0.f, {{0, 6}}); int b = B.feature(Bk, m, 0.f, {{0, 5}});
        B.feature(Bk, p, 0.4f, {{0, 2}});                                   // the closest feature of Bk, had p not been skipped
        B.seal(); B.observe(m, A, a); B.observe(m, Bk, b);
        W.points = {p};
        break;
    }
    case 2: {   // q is a loop point and A's slot: p's pRep is q, which turns bad and is skipped in Bk
        KeyFrame* A = B.kf(0.f, true); KeyFrame* Bk = B.kf(0.2f, true);
        MapPoint* q = B.mp(0.5f, 0.f, 5.f, {{60, 70}}); MapPoint* p = B.mp(0.f, 0.f, 5.f, {});
        int a = B.feature(A, p, 0.f, {{0, 8}});                             // q's slot, at p's projection
        B.feature(Bk, q, 0.f, {{60, 72}});                                  // q would take it, were it not bad
        B.feature(Bk, p, 0.f, {{0, 9}});
        B.seal(); B.observe(q, A, a);
        W.points = {q, p};
        break;
    }
    case 3: {   // two loop points on one empty slot: p0 is added, then becomes p1's vpReplacePoint and is replaced by it
        KeyFrame* A = B.kf(0.f, true);
        MapPoint* p0 = B.mp(0.f, 0.f, 5.f, {{0, 10}}); MapPoint* p1 = B.mp(0.01f, 0.f, 5.f, {{0, 12}});
        B.feature(A, p0, 0.2f, {{0, 11}});
        B.seal();
        W.points = {p0, p1};
        break;
    }
    case 4: {   // the slot holds a bad point: nothing changes, nFused still counts
        KeyFrame* A = B.kf(0.f, true);
        MapPoint* z = B.mp(0.f, 0.f, 5.f, {{0, 5}}); MapPoint* p = B.mp(0.f, 0.f, 5.f, {{0, 6}});
        int f = B.feature(A, z, 0.f, {{0, 7}});
        B.seal(); B.observe(z, A, f); z->mbBad = true;
        W.points = {p};
        break;
    }
    case 5: {   // vpMapPoints holds p twice: the snapshot misses the first acceptance, so the second entry matches p's own slot
        KeyFrame* A = B.kf(0.f, true); KeyFrame* Bk = B.kf(0.2f, true);
        MapPoint* p = B.mp(0.f, 0.f, 5.f, {});
        B.feature(A, p, 0.f, {{0, 20}});
        B.feature(Bk, p, 0.3f, {{0, 15}});
        B.seal();
        W.points = {p, p};
        break;
    }
    case 6: {   // SearchByProjection: an occupied slot, two points competing, a duplicate, an already found point, NULL, a bad one
        KeyFrame* K = B.kf(0.f, true); KeyFrame* O1 = B.kf(0.5f, false); KeyFrame* O2 = B.kf(-0.5f, false);
        MapPoint* p0 = B.mp(0.f, 0.f, 5.f, {}); MapPoint* p1 = B.mp(0.002f, 0.f, 5.f, {{0, 1}});
        MapPoint* p2 = B.mp(0.6f, 0.2f, 6.f, {{40, 45}}); MapPoint* p3 = B.mp(-0.6f, 0.2f, 6.f, {{80, 90}});
        MapPoint* p4 = B.mp(0.3f, -0.4f, 7.f, {{120, 130}}); MapPoint* p5 = B.mp(-0.3f, -0.4f, 7.f, {{160, 170}});
        MapPoint* o = B.mp(0.f, 0.f, 5.f, {{200, 210}});
        B.feature(K, p0, 0.f, {{0, 3}}); B.feature(K, p0, 0.5f, {{0, 9}});  // p0 takes the first, p1 the second
        int f2 = B.feature(K, p2, 0.f, {{40, 46}});                          // occupied on entry by o
        B.feature(K, p2, 0.4f, {{40, 60}});                                  // p2's only free candidate
        B.feature(K, p3, 0.f, {{80, 91}}); B.feature(K, p3, -0.3f, {{80, 95}});   // p3, then its duplicate
        B.feature(K, p4, 0.f, {{120, 131}});                                 // p4 is already found: skipped
        B.feature(K, p5, 0.f, {{160, 171}});                                 // p5 is bad: skipped
        B.seal();
        p5->mbBad = true;
        W.matched.assign(K->N, nullptr);
        W.matched[f2] = o;
        W.matched[6] = p4;                                                   // p4 holds a slot already (its own feature)
        W.points = {p0, p1, p2, p3, p3, nullptr, p4, p5};
        W.pointKFs = {O1, O2, O1, O2, O1, nullptr, O2, O1};
        break;
    }
    default: std::fprintf(stderr, "unknown scene %d\n", scene); std::exit(2);
    }
}

static long idOf(MapPoint* p) { return p ? (long)p->mnId : -1L; }
static long idOf(KeyFrame* k) { return k ? (long)k->mnId : -1L; }

static bool same_state(World& X, World& Y, const char* what)
{
    bool ok = true;
    for (size_t k = 0; k < X.kfs.size(); ++k)
        for (size_t j = 0; j < X.kfs[k]->mvpMapPoints.size(); ++j)
            if (idOf(X.kfs[k]->mvpMapPoints[j]) != idOf(Y.kfs[k]->mvpMapPoints[j])) { std::printf("%s: key frame %zu slot %zu differs\n", what, k, j); ok = false; }
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

static void print_state(World& W)
{
    for (auto& p : W.mps) {
        std::printf("point %lu bad=%d nObs=%d obs:", p->mnId, (int)p->mbBad, p->nObs);
        for (auto& o : p->mObservations) std::printf(" kf%lu/%d", o.first->mnId, std::get<0>(o.second));
        std::printf("\n");
    }
}

static int run_sbp(bool ref_only)
{
    World R, G;
    build(R, 6); build(G, 6);
    KeyFrame* K = R.targets[0];
    std::vector<MapPoint*> m1 = R.matched, m2 = R.matched;
    std::vector<KeyFrame*> kf2(K->N, nullptr);
    const int n1 = RefSearchByProjection(K, R.scw[0], R.points, nullptr, m1, nullptr, 4, 1.0f);
    const int n2 = RefSearchByProjection(K, R.scw[0], R.points, &R.pointKFs, m2, &kf2, 4, 1.0f);
    std::printf("scene 6: nmatches ref=%d,%d matched:", n1, n2);
    for (size_t j = 0; j < m2.size(); ++j) std::printf(" %ld/%ld", idOf(m2[j]), idOf(kf2[j]));
    std::printf("\n");
    if (ref_only) return 0;
    ORBmatcher matcher;
    KeyFrame* GK = G.targets[0];
    std::vector<MapPoint*> g1 = G.matched, g2 = G.matched;
    std::vector<KeyFrame*> gkf2(GK->N, nullptr);
    const int a1 = matcher.SearchByProjection(GK, G.scw[0], G.points, g1, 4, 1.0f);
    const int a2 = matcher.SearchByProjection(GK, G.scw[0], G.points, G.pointKFs, g2, gkf2, 4, 1.0f);
    bool ok = a1 == n1 && a2 == n2;
    for (int j = 0; j < K->N; ++j)
        ok = ok && idOf(g1[j]) == idOf(m1[j]) && idOf(g2[j]) == idOf(m2[j]) && idOf(gkf2[j]) == idOf(kf2[j]);
    std::vector<MapPoint*> shortv(GK->N - 1);
    bool threw = false;
    try { matcher.SearchByProjection(GK, G.scw[0], G.points, shortv, 4, 1.0f); } catch (const std::invalid_argument&) { threw = true; }
    ok = ok && threw;
    std::printf("adapter nmatches=%d,%d\n%s\n", a1, a2, ok ? "OK" : "MISMATCH");
    return ok ? 0 : 1;
}

int main(int argc, char** argv)
{
    if (argc < 2) { std::fprintf(stderr, "usage: %s SCENE [ref]\n", argv[0]); return 2; }
    const int scene = std::atoi(argv[1]);
    const bool ref_only = argc > 2;
    if (scene == 6) return run_sbp(ref_only);
    World R, G, S;
    build(R, scene); build(G, scene); build(S, scene);
    const int nRef = SearchAndFuseLoop(R, [](KeyFrame* pKF, Sim3f& Scw, const std::vector<MapPoint*>& vp, float th, std::vector<MapPoint*>& rep) {
        return RefFuse(pKF, Scw, vp, th, rep);
    });
    if (ref_only) {                               // the reference run alone (no device needed), its final state printed
        std::printf("scene %d: nFused ref=%d\n", scene, nRef);
        print_state(R);
        return 0;
    }
    ORBmatcher matcher;
    const int nBatch = matcher.SearchAndFuse(G.targets, G.scw, G.points, 4.f);
    const orbx_adapter::SearchAndFuseDiagnostics diag = orbx_adapter::search_and_fuse_diagnostics;
    const int nSingle = SearchAndFuseLoop(S, [&](KeyFrame* pKF, Sim3f& Scw, const std::vector<MapPoint*>& vp, float th, std::vector<MapPoint*>& rep) {
        return matcher.Fuse(pKF, Scw, vp, th, rep);
    });
    std::printf("scene %d: nFused ref=%d batched=%d single=%d researched=%d calls=%d\n", scene, nRef, nBatch, nSingle, diag.researched_pairs,
                diag.extra_calls);
    bool ok = nRef == nBatch && nRef == nSingle;
    ok = same_state(R, G, "batched") && ok;
    ok = same_state(R, S, "single") && ok;
    bool threw = false;
    S.targets[0]->NLeft = 0;
    std::vector<MapPoint*> rep(S.points.size());
    try { matcher.Fuse(S.targets[0], S.scw[0], S.points, 4.f, rep); } catch (const std::invalid_argument&) { threw = true; }
    ok = ok && threw;
    std::printf(ok ? "OK\n" : "MISMATCH\n");
    return ok ? 0 : 1;
}
