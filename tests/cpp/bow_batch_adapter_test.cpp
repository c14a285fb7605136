// Compiles csrc/adapter/ORBmatcher.h — `class ORB_SLAM3::ORBmatcher` — against stand-ins of ORB_SLAM3::Frame / KeyFrame / MapPoint
// (those of orbmatcher_class_test.cpp plus KeyFrame::isBad()) and drives the two place-recognition loops three ways:
//   Tracking::Relocalization          for each candidate: a NULL or bad one is discarded, else SearchByBoW(pKF, F, vvpMapPointMatches[i])
//   DetectCommonRegionsFromBoW        for each covisible: a NULL or bad one is skipped, else SearchByBoW(pKF1, vpCovKFi[j], vvpMatchedMPs[j])
// with the single overloads of the class in that loop, with the batched overloads (one call each), and with the CPU oracle's
// restatement of src/ORBmatcher1.cc:225-427 / src/ORBmatcher2.cc:36-171 (oracle/orb_oracle.cpp) in the same loop.  Every
// vnMatches entry, every MapPoint* and the returned sums must agree.  Scene in through a file written by
// tests/test_adapter_bow_batch_cpp.py; prints "reloc=<sum> loop=<sum>" and exits 0 when all three agree.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <vector>

#include <opencv2/core.hpp>

extern "C" {
int orbo_search_by_bow_kf_frame(const uint8_t* desc_kf, const float* angle_kf, const uint8_t* valid_kf, int n_kf, int fvk_n,
                                const uint32_t* fvk_nodes, const int32_t* fvk_off, const uint32_t* fvk_idx, const uint8_t* desc_f,
                                const float* angle_f, int n_f, int fvf_n, const uint32_t* fvf_nodes, const int32_t* fvf_off,
                                const uint32_t* fvf_idx, int Nleft, float mfNNratio, int mbCheckOrientation, int32_t* match_f);
int orbo_search_by_bow_kf_kf(const uint8_t* desc1, const float* angle1, const uint8_t* valid1, int n1, int fv1_n,
                             const uint32_t* fv1_nodes, const int32_t* fv1_off, const uint32_t* fv1_idx, const uint8_t* desc2,
                             const float* angle2, const uint8_t* valid2, int n2, int fv2_n, const uint32_t* fv2_nodes,
                             const int32_t* fv2_off, const uint32_t* fv2_idx, float mfNNratio, int mbCheckOrientation, int32_t* match12);
}

namespace ORB_SLAM3 {
struct Vec2 { float d[2]; float operator()(int i) const { return d[i]; } };
struct Vec3 { float d[3]; float operator()(int i) const { return d[i]; } };
struct SE3f {                                     // enough of Sophus::SE3f for the projection overloads the class also declares
    float R[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}, t[3] = {0, 0, 0};
    Vec3 operator*(const Vec3& p) const
    {
        Vec3 o;
        for (int r = 0; r < 3; ++r) o.d[r] = R[3 * r] * p.d[0] + R[3 * r + 1] * p.d[1] + R[3 * r + 2] * p.d[2] + t[r];
        return o;
    }
    SE3f inverse() const
    {
        SE3f o;
        for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) o.R[3 * r + c] = R[3 * c + r];
        for (int r = 0; r < 3; ++r) o.t[r] = -(o.R[3 * r] * t[0] + o.R[3 * r + 1] * t[1] + o.R[3 * r + 2] * t[2]);
        return o;
    }
    Vec3 translation() const { return Vec3{{t[0], t[1], t[2]}}; }
};
struct Pinhole {
    float fx, fy, cx, cy;
    Vec2 project(const Vec3& p) const { return Vec2{{fx * p(0) / p(2) + cx, fy * p(1) / p(2) + cy}}; }
};
class MapPoint {
public:
    bool mbTrackInView = false, mbBad = false;
    float mTrackProjX = 0, mTrackProjY = 0, mTrackProjXR = 0, mTrackViewCos = 0, mTrackDepth = 0;
    int mnTrackScaleLevel = 0, nObs = 1;
    unsigned char descriptor[32];
    Vec3 pos{{0, 0, 1}};
    bool isBad() { return mbBad; }
    int Observations() { return nObs; }
    cv::Mat GetDescriptor() { return cv::Mat(1, 32, CV_8U, descriptor); }
    Vec3 GetWorldPos() { return pos; }
};
typedef std::map<unsigned int, std::vector<unsigned int>> FeatureVector;      // DBoW2::FeatureVector
class Frame {
public:
    int N = 0, Nleft = -1;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn;
    std::vector<float> mvuRight, mvScaleFactors;
    std::vector<MapPoint*> mvpMapPoints;
    std::vector<bool> mvbOutlier;
    cv::Mat mDescriptors;
    FeatureVector mFeatVec;
    float mbf = 0, mb = 0;
    SE3f pose;
    Pinhole* mpCamera = nullptr;
    SE3f GetPose() const { return pose; }
    static float mnMinX, mnMaxX, mnMinY, mnMaxY, mfGridElementWidthInv, mfGridElementHeightInv;
};
float Frame::mnMinX, Frame::mnMaxX, Frame::mnMinY, Frame::mnMaxY, Frame::mfGridElementWidthInv, Frame::mfGridElementHeightInv;
class KeyFrame {
public:
    bool mbBad = false;
    std::vector<cv::KeyPoint> mvKeysUn;
    cv::Mat mDescriptors;
    FeatureVector mFeatVec;
    std::vector<MapPoint*> mvpMapPoints;
    bool isBad() { return mbBad; }
    std::vector<MapPoint*> GetMapPointMatches() { return mvpMapPoints; }
};
}  // namespace ORB_SLAM3

#include "ORBmatcher.h"

using namespace ORB_SLAM3;

template <class T> static std::vector<T> rd(FILE* f, size_t n) { std::vector<T> v(n); if (n && fread(v.data(), sizeof(T), n, f) != n) { std::perror("read"); exit(2); } return v; }

struct Csr {                                       // a FeatureVector as the oracle takes it
    std::vector<uint32_t> nodes, idx;
    std::vector<int32_t> off{0};
    explicit Csr(const FeatureVector& fv)
    {
        for (const auto& kv : fv) { nodes.push_back(kv.first); for (unsigned i : kv.second) idx.push_back(i); off.push_back((int32_t)idx.size()); }
    }
};

// One feature set of the scene: descriptors, angles, per-feature map-point bits (1: present, 2: isBad()) and its FeatureVector.
struct Set {
    int n = 0;
    std::vector<unsigned char> desc;
    std::vector<float> angle;
    std::vector<unsigned char> mp;
    FeatureVector fv;
    std::vector<MapPoint> points;
};

static Set read_set(FILE* f)
{
    Set s;
    s.n = rd<int32_t>(f, 1)[0];
    s.desc = rd<unsigned char>(f, (size_t)s.n * 32);
    s.angle = rd<float>(f, s.n);
    s.mp = rd<unsigned char>(f, s.n);
    const int nn = rd<int32_t>(f, 1)[0];
    const std::vector<uint32_t> nodes = rd<uint32_t>(f, nn);
    const std::vector<int32_t> off = rd<int32_t>(f, nn + 1);
    const std::vector<uint32_t> idx = rd<uint32_t>(f, off[nn]);
    for (int k = 0; k < nn; ++k) s.fv[nodes[k]] = std::vector<unsigned int>(idx.begin() + off[k], idx.begin() + off[k + 1]);
    s.points.resize(s.n);
    for (int i = 0; i < s.n; ++i) s.points[i].mbBad = (s.mp[i] & 2) != 0;
    return s;
}

static void make_kf(Set& s, KeyFrame& kf)
{
    kf.mvKeysUn.resize(s.n);
    kf.mDescriptors = cv::Mat(s.n, 32, CV_8U, s.desc.data());
    kf.mFeatVec = s.fv;
    kf.mvpMapPoints.assign(s.n, nullptr);
    for (int i = 0; i < s.n; ++i) { kf.mvKeysUn[i].angle = s.angle[i]; if (s.mp[i] & 1) kf.mvpMapPoints[i] = &s.points[i]; }
}

static std::vector<uint8_t> usable(const std::vector<MapPoint*>& v)
{
    std::vector<uint8_t> u(v.size());
    for (size_t i = 0; i < v.size(); ++i) u[i] = v[i] && !v[i]->isBad();
    return u;
}

static int fails = 0;
static void expect(bool ok, const char* what, int i)
{
    if (!ok) { std::printf("MISMATCH %s at %d\n", what, i); ++fails; }
}

static void compare(const char* loop, const std::vector<int>& n1, const std::vector<std::vector<MapPoint*>>& v1, const std::vector<int>& n2,
                    const std::vector<std::vector<MapPoint*>>& v2)
{
    expect(n1.size() == n2.size() && v1.size() == v2.size(), loop, -1);
    for (size_t i = 0; i < n1.size() && i < n2.size(); ++i) {
        expect(n1[i] == n2[i], loop, (int)i);
        expect(v1[i] == v2[i], loop, (int)i);
    }
}

int main(int argc, char** argv)
{
    if (argc < 2) { std::fprintf(stderr, "usage: %s scene.bin\n", argv[0]); return 2; }
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) { std::perror(argv[1]); return 2; }
    const int nK = rd<int32_t>(f, 1)[0];
    const std::vector<int32_t> state = rd<int32_t>(f, nK);                 // per slot: 0 = key frame, 1 = NULL, 2 = isBad()
    Set fixed = read_set(f);
    std::vector<Set> sets;
    for (int k = 0; k < nK; ++k) sets.push_back(read_set(f));
    std::fclose(f);

    std::vector<KeyFrame> kfs(nK);
    std::vector<KeyFrame*> vpKFs(nK, nullptr);
    for (int k = 0; k < nK; ++k) {
        make_kf(sets[k], kfs[k]);
        kfs[k].mbBad = state[k] == 2;
        if (state[k] != 1) vpKFs[k] = &kfs[k];
    }
    Frame F;
    F.N = fixed.n; F.mvKeys.resize(fixed.n); F.mvKeysUn.resize(fixed.n);
    F.mDescriptors = cv::Mat(fixed.n, 32, CV_8U, fixed.desc.data()); F.mFeatVec = fixed.fv;
    for (int j = 0; j < fixed.n; ++j) { F.mvKeys[j].angle = fixed.angle[j]; F.mvKeysUn[j].angle = fixed.angle[j]; }
    KeyFrame kf1;
    make_kf(fixed, kf1);
    const Csr cF(fixed.fv);

    // ---- Tracking::Relocalization: ORBmatcher matcher(0.75, true)
    {
        ORBmatcher matcher(0.75, true);
        std::vector<std::vector<MapPoint*>> vvS(nK), vvB, vvO(nK);
        std::vector<int> vnS(nK, 0), vnB, vnO(nK, 0);
        int sumS = 0, sumO = 0;
        for (int i = 0; i < nK; i++) {
            KeyFrame* pKF = vpKFs[i];
            if (!pKF || pKF->isBad()) continue;                             // vbDiscarded[i] = true
            vnS[i] = matcher.SearchByBoW(pKF, F, vvS[i]);
            sumS += vnS[i];
            const std::vector<MapPoint*> mps = pKF->GetMapPointMatches();
            const std::vector<uint8_t> ok = usable(mps);
            const Csr c(pKF->mFeatVec);
            std::vector<int32_t> m(F.N, -1);
            vnO[i] = orbo_search_by_bow_kf_frame(sets[i].desc.data(), sets[i].angle.data(), ok.data(), sets[i].n, (int)c.nodes.size(), c.nodes.data(),
                                                 c.off.data(), c.idx.data(), fixed.desc.data(), fixed.angle.data(), F.N, (int)cF.nodes.size(),
                                                 cF.nodes.data(), cF.off.data(), cF.idx.data(), -1, 0.75f, 1, m.data());
            sumO += vnO[i];
            vvO[i].assign(F.N, nullptr);
            for (int j = 0; j < F.N; ++j) if (m[j] >= 0) vvO[i][j] = mps[m[j]];
        }
        const int sumB = matcher.SearchByBoW(vpKFs, F, vvB, vnB);
        compare("reloc single/batch", vnS, vvS, vnB, vvB);
        compare("reloc oracle/batch", vnO, vvO, vnB, vvB);
        expect(sumS == sumB && sumO == sumB, "reloc sum", sumB);
        std::printf("reloc=%d ", sumB);
    }
    // ---- LoopClosing::DetectCommonRegionsFromBoW: ORBmatcher matcherBoW(0.9, true)
    {
        ORBmatcher matcherBoW(0.9, true);
        std::vector<std::vector<MapPoint*>> vvS(nK), vvB, vvO(nK);
        std::vector<int> vnS(nK, 0), vnB, vnO(nK, 0);
        int sumS = 0, sumO = 0;
        const std::vector<MapPoint*> mps1 = kf1.GetMapPointMatches();
        const std::vector<uint8_t> ok1 = usable(mps1);
        for (int j = 0; j < nK; ++j) {
            if (!vpKFs[j] || vpKFs[j]->isBad()) continue;
            vnS[j] = matcherBoW.SearchByBoW(&kf1, vpKFs[j], vvS[j]);
            sumS += vnS[j];
            const std::vector<MapPoint*> mps2 = vpKFs[j]->GetMapPointMatches();
            const std::vector<uint8_t> ok2 = usable(mps2);
            const Csr c(vpKFs[j]->mFeatVec);
            std::vector<int32_t> m(fixed.n, -1);
            vnO[j] = orbo_search_by_bow_kf_kf(fixed.desc.data(), fixed.angle.data(), ok1.data(), fixed.n, (int)cF.nodes.size(), cF.nodes.data(),
                                              cF.off.data(), cF.idx.data(), sets[j].desc.data(), sets[j].angle.data(), ok2.data(), sets[j].n,
                                              (int)c.nodes.size(), c.nodes.data(), c.off.data(), c.idx.data(), 0.9f, 1, m.data());
            sumO += vnO[j];
            vvO[j].assign(fixed.n, nullptr);
            for (int i = 0; i < fixed.n; ++i) if (m[i] >= 0) vvO[j][i] = mps2[m[i]];
        }
        const int sumB = matcherBoW.SearchByBoW(&kf1, vpKFs, vvB, vnB);
        compare("loop single/batch", vnS, vvS, vnB, vvB);
        compare("loop oracle/batch", vnO, vvO, vnB, vvB);
        expect(sumS == sumB && sumO == sumB, "loop sum", sumB);
        std::printf("loop=%d\n", sumB);
    }
    return fails ? 1 : 0;
}
