// Compiles csrc/adapter/ORBmatcher.h — `class ORB_SLAM3::ORBmatcher` with the reference's declaration of
//   int SearchForTriangulation(KeyFrame* pKF1, KeyFrame* pKF2, vector<pair<size_t, size_t>>& vMatchedPairs, const bool bOnlyStereo,
//                              const bool bCoarse = false)
// and the added batched overload SearchForTriangulation(pKF1, vpKF2, vbCoarse, bOnlyStereo, body) — against stand-ins of
// ORB_SLAM3::KeyFrame / MapPoint with a rotation + translation pose, a pinhole camera with toK_(), mFeatVec and map-point slots.
// The driver builds identical worlds for one scene (3-D points seen by KF1 and its neighbours, projected exactly), runs a
// CreateNewMapPoints-shaped loop three times — over the reference's SearchForTriangulation (src/ORBmatcher2.cc:173-471 with
// Pinhole::epipolarConstrain, restated below over the same stand-ins), over the single overload of the class, and as the
// batched overload — and compares the per-neighbour vMatchedPairs, the return values and every key frame's final slots.  The
// loop adds one new map point to KF1 and to the neighbour for every match, as CreateNewMapPoints does after triangulating.
//   usage: triangulation_adapter_test SCENE [ref]   (SCENE = 0..5; prints "researched=<neighbours> dropped=<matches>" of the
//                                                    batched run; with "ref" only the reference loop runs and prints its counts)
#include <algorithm>
#include <array>
#include <cassert>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <random>
#include <stdexcept>
#include <utility>
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
struct Mat3 {
    float m[3][3];
    float operator()(int r, int c) const { return m[r][c]; }
    Mat3 operator*(const Mat3& o) const
    {
        Mat3 p{};
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) p.m[r][c] = m[r][0] * o.m[0][c] + m[r][1] * o.m[1][c] + m[r][2] * o.m[2][c];
        return p;
    }
    Vec3 operator*(const Vec3& v) const
    {
        Vec3 p{};
        for (int r = 0; r < 3; ++r) p.d[r] = m[r][0] * v.d[0] + m[r][1] * v.d[1] + m[r][2] * v.d[2];
        return p;
    }
    Mat3 transpose() const
    {
        Mat3 t{};
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) t.m[r][c] = m[c][r];
        return t;
    }
    Mat3 inverse() const                          // adjugate / determinant
    {
        const float det = m[0][0] * (m[1][1] * m[2][2] - m[1][2] * m[2][1]) - m[0][1] * (m[1][0] * m[2][2] - m[1][2] * m[2][0]) +
                          m[0][2] * (m[1][0] * m[2][1] - m[1][1] * m[2][0]);
        Mat3 a{};
        a.m[0][0] = (m[1][1] * m[2][2] - m[1][2] * m[2][1]) / det; a.m[0][1] = (m[0][2] * m[2][1] - m[0][1] * m[2][2]) / det;
        a.m[0][2] = (m[0][1] * m[1][2] - m[0][2] * m[1][1]) / det; a.m[1][0] = (m[1][2] * m[2][0] - m[1][0] * m[2][2]) / det;
        a.m[1][1] = (m[0][0] * m[2][2] - m[0][2] * m[2][0]) / det; a.m[1][2] = (m[0][2] * m[1][0] - m[0][0] * m[1][2]) / det;
        a.m[2][0] = (m[1][0] * m[2][1] - m[1][1] * m[2][0]) / det; a.m[2][1] = (m[0][1] * m[2][0] - m[0][0] * m[2][1]) / det;
        a.m[2][2] = (m[0][0] * m[1][1] - m[0][1] * m[1][0]) / det;
        return a;
    }
};
struct SO3f {
    static Mat3 hat(const Vec3& t) { return Mat3{{{0, -t(2), t(1)}, {t(2), 0, -t(0)}, {-t(1), t(0), 0}}}; }
};
struct SE3f {                                     // p_c = R p_w + t
    Mat3 R{{{1, 0, 0}, {0, 1, 0}, {0, 0, 1}}};
    Vec3 t{{0, 0, 0}};
    Vec3 operator*(const Vec3& p) const { const Vec3 q = R * p; return Vec3{{q.d[0] + t.d[0], q.d[1] + t.d[1], q.d[2] + t.d[2]}}; }
    SE3f operator*(const SE3f& o) const { SE3f s; s.R = R * o.R; s.t = (*this) * o.t; return s; }
    SE3f inverse() const { SE3f s; s.R = R.transpose(); const Vec3 q = s.R * t; s.t = Vec3{{-q.d[0], -q.d[1], -q.d[2]}}; return s; }
    Mat3 rotationMatrix() const { return R; }
    Vec3 translation() const { return t; }
    SO3f so3() const { return SO3f(); }
};
struct Pinhole {
    float fx = 435.f, fy = 435.f, cx = 376.f, cy = 240.f;
    Vec2 project(const Vec3& p) const { return Vec2{{fx * p(0) / p(2) + cx, fy * p(1) / p(2) + cy}}; }
    Mat3 toK_() const { return Mat3{{{fx, 0.f, cx}, {0.f, fy, cy}, {0.f, 0.f, 1.f}}}; }
};
static const std::vector<float> kScale = {1.0f, 1.2f, 1.44f, 1.728f, 2.0736f, 2.48832f, 2.985984f, 3.5831808f};

class MapPoint {
public:
    long unsigned int mnId = 0;
    bool mbTrackInView = false;                                                // (the tracking-thread members the class reads)
    float mTrackProjX = 0, mTrackProjY = 0, mTrackProjXR = 0, mTrackViewCos = 0, mTrackDepth = 0;
    int mnTrackScaleLevel = 0;
    unsigned char desc[32] = {};
    bool isBad() { return false; }
    int Observations() { return 1; }
    cv::Mat GetDescriptor() { return cv::Mat(1, 32, CV_8U, desc); }
    Vec3 GetWorldPos() { return Vec3{{0, 0, 1}}; }
};
typedef std::map<unsigned int, std::vector<unsigned int>> FeatureVector;      // DBoW2::FeatureVector
class KeyFrame {
public:
    long unsigned int mnId = 0;
    int N = 0, NLeft = -1;
    std::vector<cv::KeyPoint> mvKeysUn;
    std::vector<unsigned char> descBuf;
    cv::Mat mDescriptors;
    std::vector<float> mvuRight, mvScaleFactors = kScale, mvLevelSigma2;
    FeatureVector mFeatVec;
    SE3f Tcw;
    Pinhole cam;
    Pinhole* mpCamera = &cam;
    Pinhole* mpCamera2 = nullptr;
    std::vector<MapPoint*> mvpMapPoints;
    KeyFrame() { for (float s : kScale) mvLevelSigma2.push_back(s * s); }
    SE3f GetPose() const { return Tcw; }
    SE3f GetPoseInverse() const { return Tcw.inverse(); }
    Vec3 GetCameraCenter() const { return Tcw.inverse().translation(); }
    MapPoint* GetMapPoint(const size_t& idx) { return mvpMapPoints[idx]; }
    void AddMapPoint(MapPoint* pMP, const size_t& idx) { mvpMapPoints[idx] = pMP; }
    std::vector<MapPoint*> GetMapPointMatches() { return mvpMapPoints; }
};
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
typedef std::vector<std::pair<size_t, size_t>> Pairs;

// ---- the reference over the stand-ins (src/ORBmatcher2.cc:173-471 single camera; Pinhole.cpp:107-129) -----------------------
static bool RefEpipolarConstrain(Pinhole* cam1, Pinhole* cam2, const cv::KeyPoint& kp1, const cv::KeyPoint& kp2, const Mat3& R12, const Vec3& t12,
                                 const float sigmaLevel, const float unc)
{
    (void)sigmaLevel;
    //Compute Fundamental Matrix
    Mat3 t12x = SO3f::hat(t12);
    Mat3 K1 = cam1->toK_();
    Mat3 K2 = cam2->toK_();
    Mat3 F12 = K1.transpose().inverse() * t12x * R12 * K2.inverse();
    // Epipolar line in second image l = x1'F12 = [a b c]
    const float a = kp1.pt.x * F12(0, 0) + kp1.pt.y * F12(1, 0) + F12(2, 0);
    const float b = kp1.pt.x * F12(0, 1) + kp1.pt.y * F12(1, 1) + F12(2, 1);
    const float c = kp1.pt.x * F12(0, 2) + kp1.pt.y * F12(1, 2) + F12(2, 2);
    const float num = a * kp2.pt.x + b * kp2.pt.y + c;
    const float den = a * a + b * b;
    if (den == 0) return false;
    const float dsqr = num * num / den;
    return dsqr < 3.84 * unc;
}

static void RefThreeMaxima(std::vector<int>* histo, const int L, int& ind1, int& ind2, int& ind3)   // src/ORBmatcher3.cc:592-633
{
    int max1 = 0, max2 = 0, max3 = 0;
    for (int i = 0; i < L; i++) {
        const int s = (int)histo[i].size();
        if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
        else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
        else if (s > max3) { max3 = s; ind3 = i; }
    }
    if (max2 < 0.1f * (float)max1) { ind2 = -1; ind3 = -1; }
    else if (max3 < 0.1f * (float)max1) { ind3 = -1; }
}

static int RefSearchForTriangulation(KeyFrame* pKF1, KeyFrame* pKF2, Pairs& vMatchedPairs, const bool bOnlyStereo, const bool bCoarse,
                                     const bool mbCheckOrientation)
{
    const int TH_LOW = 50, HISTO_LENGTH = 30;
    const FeatureVector& vFeatVec1 = pKF1->mFeatVec;
    const FeatureVector& vFeatVec2 = pKF2->mFeatVec;
    //Compute epipole in second image
    SE3f T1w = pKF1->GetPose();
    SE3f T2w = pKF2->GetPose();
    SE3f Tw2 = pKF2->GetPoseInverse();
    Vec3 Cw = pKF1->GetCameraCenter();
    Vec3 C2 = T2w * Cw;
    Vec2 ep = pKF2->mpCamera->project(C2);
    SE3f T12 = T1w * Tw2;
    Mat3 R12 = T12.rotationMatrix();
    Vec3 t12 = T12.translation();
    Pinhole *pCamera1 = pKF1->mpCamera, *pCamera2 = pKF2->mpCamera;
    int nmatches = 0;
    std::vector<bool> vbMatched2(pKF2->N, false);
    std::vector<int> vMatches12(pKF1->N, -1);
    std::vector<int> rotHist[HISTO_LENGTH];
    const float factor = 1.0f / HISTO_LENGTH;
    auto f1it = vFeatVec1.begin(), f2it = vFeatVec2.begin();
    auto f1end = vFeatVec1.end(), f2end = vFeatVec2.end();
    while (f1it != f1end && f2it != f2end) {
        if (f1it->first == f2it->first) {
            for (size_t i1 = 0, iend1 = f1it->second.size(); i1 < iend1; i1++) {
                const size_t idx1 = f1it->second[i1];
                MapPoint* pMP1 = pKF1->GetMapPoint(idx1);
                // If there is already a MapPoint skip
                if (pMP1) continue;
                const bool bStereo1 = pKF1->mvuRight[idx1] >= 0;
                if (bOnlyStereo)
                    if (!bStereo1) continue;
                const cv::KeyPoint& kp1 = pKF1->mvKeysUn[idx1];
                const unsigned char* d1 = pKF1->mDescriptors.ptr((int)idx1);
                int bestDist = TH_LOW;
                int bestIdx2 = -1;
                for (size_t i2 = 0, iend2 = f2it->second.size(); i2 < iend2; i2++) {
                    size_t idx2 = f2it->second[i2];
                    MapPoint* pMP2 = pKF2->GetMapPoint(idx2);
                    // If we have already matched or there is a MapPoint skip
                    if (vbMatched2[idx2] || pMP2) continue;
                    const bool bStereo2 = pKF2->mvuRight[idx2] >= 0;
                    if (bOnlyStereo)
                        if (!bStereo2) continue;
                    const unsigned char* d2 = pKF2->mDescriptors.ptr((int)idx2);
                    const int dist = orbx_descriptor_distance(d1, d2);
                    if (dist > TH_LOW || dist > bestDist) continue;
                    const cv::KeyPoint& kp2 = pKF2->mvKeysUn[idx2];
                    if (!bStereo1 && !bStereo2) {
                        const float distex = ep(0) - kp2.pt.x;
                        const float distey = ep(1) - kp2.pt.y;
                        if (distex * distex + distey * distey < 100 * pKF2->mvScaleFactors[kp2.octave]) continue;
                    }
                    if (bCoarse || RefEpipolarConstrain(pCamera1, pCamera2, kp1, kp2, R12, t12, pKF1->mvLevelSigma2[kp1.octave],
                                                        pKF2->mvLevelSigma2[kp2.octave])) {
                        bestIdx2 = (int)idx2;
                        bestDist = dist;
                    }
                }
                if (bestIdx2 >= 0) {
                    const cv::KeyPoint& kp2 = pKF2->mvKeysUn[bestIdx2];
                    vMatches12[idx1] = bestIdx2;
                    nmatches++;
                    if (mbCheckOrientation) {
                        float rot = kp1.angle - kp2.angle;
                        if (rot < 0.0) rot += 360.0f;
                        int bin = (int)std::round(rot * factor);
                        if (bin == HISTO_LENGTH) bin = 0;
                        assert(bin >= 0 && bin < HISTO_LENGTH);
                        rotHist[bin].push_back((int)idx1);
                    }
                }
            }
            f1it++;
            f2it++;
        } else if (f1it->first < f2it->first) {
            f1it = vFeatVec1.lower_bound(f2it->first);
        } else {
            f2it = vFeatVec2.lower_bound(f1it->first);
        }
    }
    if (mbCheckOrientation) {
        int ind1 = -1, ind2 = -1, ind3 = -1;
        RefThreeMaxima(rotHist, HISTO_LENGTH, ind1, ind2, ind3);
        for (int i = 0; i < HISTO_LENGTH; i++) {
            if (i == ind1 || i == ind2 || i == ind3) continue;
            for (size_t j = 0, jend = rotHist[i].size(); j < jend; j++) {
                vMatches12[rotHist[i][j]] = -1;
                nmatches--;
            }
        }
    }
    vMatchedPairs.clear();
    vMatchedPairs.reserve(nmatches);
    for (size_t i = 0, iend = vMatches12.size(); i < iend; i++) {
        if (vMatches12[i] < 0) continue;
        vMatchedPairs.push_back(std::make_pair(i, (size_t)vMatches12[i]));
    }
    return nmatches;
}

// ---- scenes -------------------------------------------------------------------------------------------------------------------
struct Seen { int point; float angle_off; };                 // a neighbour sees 3-D point `point`, its key point rotated by angle_off
struct Scene {
    int n_points = 0;
    std::vector<int> kf1;                                    // the points KF1 sees, in feature order
    std::vector<int> kf1_occupied;                           // KF1 features holding a map point on entry
    std::vector<std::vector<Seen>> nbrs;
    std::vector<char> coarse;
    bool only_stereo = false, check_ori = false;
    int stop_after = -1;                                     // the body returns false after this neighbour
    int poke_kf = -1, poke_point = -1;                       // after neighbour 0, the body gives neighbour poke_kf's feature of poke_point a map point
    float stereo_frac = 0.f;
};
static std::vector<Seen> range(int a, int b, float off) { std::vector<Seen> v; for (int p = a; p < b; ++p) v.push_back({p, off}); return v; }
static std::vector<Seen> cat(std::vector<Seen> a, const std::vector<Seen>& b) { a.insert(a.end(), b.begin(), b.end()); return a; }
static std::vector<int> ids(int a, int b) { std::vector<int> v; for (int p = a; p < b; ++p) v.push_back(p); return v; }

static Scene make_scene(int s)
{
    Scene S;
    switch (s) {
    case 0:   // a KF1 feature matched by neighbour 0 is also the best candidate for neighbours 1 and 2: the batch drops it there
        S.n_points = 70; S.kf1 = ids(0, 70); S.kf1_occupied = {0, 1, 2, 3, 4};
        S.nbrs = {range(0, 60, 0.f), cat(range(0, 60, 0.f), range(60, 70, 0.f)), range(0, 60, 0.f)};
        S.coarse = {0, 1, 0};
        break;
    case 1:   // rotation filter: neighbour 1's raw result is dominated by bin 10 (points neighbour 0 takes first); after the drop
              // its 10 matches in bin 5 are the dominant bin and survive (a filter before the drop would remove them)
        S.n_points = 160; S.kf1 = ids(0, 160); S.check_ori = true;
        S.nbrs = {range(0, 150, 0.f), cat(range(0, 150, 300.f), range(150, 160, 150.f))};
        S.coarse = {0, 0};
        break;
    case 2:   // the body of neighbour 0 gives a feature of neighbour 2 a map point: exactly one re-search
        S.n_points = 60; S.kf1 = ids(0, 60);
        S.nbrs = {range(0, 20, 0.f), range(20, 40, 0.f), range(40, 60, 0.f)};
        S.coarse = {0, 0, 0}; S.poke_kf = 2; S.poke_point = 45;
        break;
    case 3:   // early stop after neighbour 1 (CheckNewKeyFrames)
        S.n_points = 60; S.kf1 = ids(0, 60);
        S.nbrs = {range(0, 30, 0.f), range(10, 40, 0.f), range(20, 60, 0.f)};
        S.coarse = {0, 0, 0}; S.stop_after = 1;
        break;
    case 4:   // two-camera key frame: both overloads throw
        S.n_points = 10; S.kf1 = ids(0, 10); S.nbrs = {range(0, 10, 0.f), range(0, 10, 0.f)}; S.coarse = {0, 0};
        break;
    default:  // overlapping neighbours, stereo features, bOnlyStereo, mixed bCoarse and the rotation filter
        S.n_points = 300; S.kf1 = ids(0, 300); S.kf1_occupied = {3, 50, 51, 52, 199};
        S.nbrs = {range(0, 120, 30.f), range(60, 200, 0.f), cat(range(100, 300, 60.f), range(0, 20, 0.f)), range(150, 300, 30.f)};
        S.coarse = {1, 0, 0, 1}; S.only_stereo = true; S.check_ori = true; S.stereo_frac = 0.7f;
        break;
    }
    return S;
}

struct World {
    std::vector<std::unique_ptr<KeyFrame>> kfs;              // kfs[0] = KF1, then the neighbours
    std::vector<std::unique_ptr<MapPoint>> mps;
    std::vector<std::vector<int>> feat_of;                   // [kf][point] feature index or -1
    MapPoint* new_point()
    {
        mps.emplace_back(new MapPoint);
        mps.back()->mnId = mps.size();
        return mps.back().get();
    }
};

static SE3f pose(float yaw, float tx, float ty, float tz)
{
    SE3f T;
    const float c = std::cos(yaw), s = std::sin(yaw);
    T.R = Mat3{{{c, 0, s}, {0, 1, 0}, {-s, 0, c}}};
    T.t = Vec3{{tx, ty, tz}};
    return T;
}

static void build(World& W, const Scene& S, int seed)
{
    std::mt19937 rng(1000 + seed);
    std::uniform_real_distribution<float> U(0.f, 1.f);
    std::vector<Vec3> X(S.n_points);
    std::vector<std::array<unsigned char, 32>> D(S.n_points);
    std::vector<float> ang(S.n_points);
    for (int p = 0; p < S.n_points; ++p) {
        X[p] = Vec3{{-2.5f + 5.f * U(rng), -1.5f + 3.f * U(rng), 5.f + 4.f * U(rng)}};
        for (auto& b : D[p]) b = (unsigned char)(rng() & 255);
        ang[p] = 40.f + 200.f * U(rng);
    }
    const int nK = 1 + (int)S.nbrs.size();
    W.feat_of.assign(nK, std::vector<int>(S.n_points, -1));
    for (int k = 0; k < nK; ++k) {
        W.kfs.emplace_back(new KeyFrame);
        KeyFrame* K = W.kfs.back().get();
        K->mnId = k;
        K->Tcw = k == 0 ? pose(0.f, 0.f, 0.f, 0.f) : pose(0.05f * k - 0.1f, -0.35f * k - 0.1f, 0.04f * k, 0.12f);
        std::vector<Seen> seen;
        if (k == 0) for (int p : S.kf1) seen.push_back({p, 0.f});
        else seen = S.nbrs[k - 1];
        if (k > 0) std::shuffle(seen.begin(), seen.end(), rng);
        const int N = (int)seen.size();
        K->N = N;
        K->mvKeysUn.resize(N);
        K->descBuf.resize((size_t)N * 32);
        K->mvuRight.assign(N, -1.f);
        K->mvpMapPoints.assign(N, nullptr);
        for (int i = 0; i < N; ++i) {
            const int p = seen[i].point;
            W.feat_of[k][p] = i;
            const Vec2 uv = K->cam.project(K->Tcw * X[p]);
            cv::KeyPoint& kp = K->mvKeysUn[i];
            kp.pt.x = uv(0); kp.pt.y = uv(1);
            kp.octave = (int)(rng() % 8); kp.size = 31.f; kp.response = 1.f; kp.class_id = -1;
            float a = ang[p] - seen[i].angle_off + (U(rng) - 0.5f) * 4.f;
            if (a < 0) a += 360.f;
            kp.angle = a;
            std::memcpy(&K->descBuf[(size_t)i * 32], D[p].data(), 32);
            const int flips = (int)(rng() % 4);
            for (int f = 0; f < flips; ++f) { const int bit = (int)(rng() % 256); K->descBuf[(size_t)i * 32 + bit / 8] ^= (unsigned char)(1u << (bit % 8)); }
            if (U(rng) < S.stereo_frac) K->mvuRight[i] = uv(0) - 20.f;
            K->mFeatVec[1 + (unsigned)p % 17].push_back((unsigned)i);      // a point's features share a vocabulary node
        }
        for (auto& node : K->mFeatVec) std::sort(node.second.begin(), node.second.end());
        K->mDescriptors = cv::Mat(N, 32, CV_8U, K->descBuf.data());
    }
    for (int i : S.kf1_occupied) W.kfs[0]->AddMapPoint(W.new_point(), i);
}

// The CreateNewMapPoints-shaped body: a new map point in KF1 and in the neighbour for every match (after triangulation, which
// the stand-ins skip), the scene's poke after neighbour 0, and the early stop.
struct Run { std::vector<Pairs> pairs; std::vector<int> ret; };
static bool body(World& W, const Scene& S, int k, const Pairs& vMatchedPairs, Run& R, int ret)
{
    R.pairs.push_back(vMatchedPairs);
    R.ret.push_back(ret);
    KeyFrame* pKF1 = W.kfs[0].get();
    KeyFrame* pKF2 = W.kfs[1 + k].get();
    for (const auto& pr : vMatchedPairs) {
        MapPoint* pMP = W.new_point();
        pKF1->AddMapPoint(pMP, pr.first);
        pKF2->AddMapPoint(pMP, pr.second);
    }
    if (k == 0 && S.poke_kf >= 0) W.kfs[1 + S.poke_kf]->AddMapPoint(W.new_point(), W.feat_of[1 + S.poke_kf][S.poke_point]);
    return k != S.stop_after;
}

static bool same(const World& A, const Run& a, const World& B, const Run& b, const char* what)
{
    bool ok = a.pairs == b.pairs && a.ret == b.ret;
    if (!ok) std::printf("%s: per-neighbour pairs or return values differ (%zu vs %zu neighbours)\n", what, a.pairs.size(), b.pairs.size());
    for (size_t k = 0; k < A.kfs.size(); ++k)
        for (int j = 0; j < A.kfs[k]->N; ++j) {
            const MapPoint* x = A.kfs[k]->mvpMapPoints[j];
            const MapPoint* y = B.kfs[k]->mvpMapPoints[j];
            if ((x ? (long)x->mnId : -1L) != (y ? (long)y->mnId : -1L)) { std::printf("%s: key frame %zu slot %d differs\n", what, k, j); ok = false; }
        }
    return ok;
}

int main(int argc, char** argv)
{
    if (argc < 2) { std::fprintf(stderr, "usage: %s SCENE [ref]\n", argv[0]); return 2; }
    const int scene = std::atoi(argv[1]);
    const Scene S = make_scene(scene);
    World R, G, T;
    build(R, S, scene); build(G, S, scene); build(T, S, scene);
    std::vector<KeyFrame*> nR, nG, nT;
    for (size_t k = 1; k < R.kfs.size(); ++k) { nR.push_back(R.kfs[k].get()); nG.push_back(G.kfs[k].get()); nT.push_back(T.kfs[k].get()); }
    Run rr, rg, rt;
    for (size_t k = 0; k < nR.size(); ++k) {
        Pairs v;
        const int n = RefSearchForTriangulation(R.kfs[0].get(), nR[k], v, S.only_stereo, S.coarse[k] != 0, S.check_ori);
        if (!body(R, S, (int)k, v, rr, n)) break;
    }
    std::printf("scene %d: ref n=", scene);
    for (int n : rr.ret) std::printf(" %d", n);
    std::printf("\n");
    if (argc > 2) return 0;                       // "ref": the reference run alone (no device needed)
    ORBmatcher matcher(0.6f, S.check_ori);
    if (scene == 4) {                             // two-camera key frames keep the reference code: both overloads throw
        int threw = 0;
        Pinhole second;
        nG[1]->mpCamera2 = &second;
        Pairs v;
        try { matcher.SearchForTriangulation(G.kfs[0].get(), nG[1], v, false); } catch (const std::invalid_argument&) { threw++; }
        try { matcher.SearchForTriangulation(G.kfs[0].get(), nG, S.coarse, false, [](int, Pairs&) { return true; }); } catch (const std::invalid_argument&) { threw++; }
        nG[1]->mpCamera2 = nullptr;
        G.kfs[0]->NLeft = 500;
        try { matcher.SearchForTriangulation(G.kfs[0].get(), nG[0], v, false); } catch (const std::invalid_argument&) { threw++; }
        std::printf("threw=%d\n", threw);
        std::printf(threw == 3 ? "OK\n" : "MISMATCH\n");
        return threw == 3 ? 0 : 1;
    }
    for (size_t k = 0; k < nT.size(); ++k) {      // the single overload in the loop
        Pairs v;
        const int n = matcher.SearchForTriangulation(T.kfs[0].get(), nT[k], v, S.only_stereo, S.coarse[k] != 0);
        if (!body(T, S, (int)k, v, rt, n)) break;
    }
    const int total = matcher.SearchForTriangulation(G.kfs[0].get(), nG, S.coarse, S.only_stereo,
                                                     [&](int k, Pairs& v) { return body(G, S, k, v, rg, (int)v.size()); });
    const orbx_adapter::TriangulationDiagnostics diag = orbx_adapter::triangulation_diagnostics;
    int sum = 0;
    for (int n : rr.ret) sum += n;
    std::printf("batched total=%d researched=%d dropped=%d\n", total, diag.researched_kfs, diag.dropped);
    bool ok = total == sum;
    ok = same(R, rr, T, rt, "single") && ok;
    ok = same(R, rr, G, rg, "batched") && ok;
    std::printf(ok ? "OK\n" : "MISMATCH\n");
    return ok ? 0 : 1;
}
