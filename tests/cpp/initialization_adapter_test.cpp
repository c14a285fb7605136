// Compiles csrc/adapter/ORBmatcher.h — `class ORB_SLAM3::ORBmatcher` with the reference's declaration of
//   int SearchForInitialization(Frame &F1, Frame &F2, std::vector<cv::Point2f> &vbPrevMatched, std::vector<int> &vnMatches12,
//                               int windowSize = 10)                                                 (include/ORBmatcher.h)
// — against stand-ins of ORB_SLAM3::Frame / KeyFrame / MapPoint (the same stand-ins as tests/cpp/orbmatcher_class_test.cpp) and
// calls it the way Tracking::MonocularInitialization does (src/Tracking3.cc:740-741): ORBmatcher(nnratio, checkOri) and the
// initial frame's key points as vbPrevMatched, then a second call on the updated vbPrevMatched.  Scene in, (return value,
// vnMatches12, vbPrevMatched) of both calls out, through files written / read by tests/test_adapter_init_cpp.py.
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <map>
#include <vector>

#include <opencv2/core.hpp>

namespace ORB_SLAM3 {
struct Vec2 { float d[2]; float operator()(int i) const { return d[i]; } };
struct Vec3 { float d[3]; float operator()(int i) const { return d[i]; } };
struct SE3f {                                     // rotation (row-major) + translation; enough of Sophus::SE3f for the call sites
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
    std::vector<cv::KeyPoint> mvKeysUn;
    cv::Mat mDescriptors;
    FeatureVector mFeatVec;
    std::vector<MapPoint*> mvpMapPoints;
    std::vector<MapPoint*> GetMapPointMatches() { return mvpMapPoints; }
};
}  // namespace ORB_SLAM3

#include "ORBmatcher.h"

using namespace ORB_SLAM3;

template <class T> static std::vector<T> rd(FILE* f, size_t n) { std::vector<T> v(n); if (n && fread(v.data(), sizeof(T), n, f) != n) { std::perror("read"); exit(2); } return v; }

static void read_frame(FILE* f, Frame& F, std::vector<unsigned char>& desc, int n, const std::vector<float>& scale)
{
    F.N = n;
    F.mvKeysUn = rd<cv::KeyPoint>(f, n); F.mvKeys = F.mvKeysUn;
    desc = rd<unsigned char>(f, (size_t)n * 32);
    F.mDescriptors = cv::Mat(n, 32, CV_8U, desc.data());
    F.mvScaleFactors = scale;
    F.mvuRight.assign(n, -1.0f);                                  // monocular
}

int main(int argc, char** argv)
{
    if (argc < 3) { std::fprintf(stderr, "usage: %s scene.bin result.bin\n", argv[0]); return 2; }
    FILE* f = std::fopen(argv[1], "rb");
    if (!f) { std::perror(argv[1]); return 2; }
    const std::vector<int32_t> hdr = rd<int32_t>(f, 6);          // n1, n2, n3, n levels, windowSize, checkOri
    const int n1 = hdr[0], n2 = hdr[1], n3 = hdr[2], nlev = hdr[3], window = hdr[4], check_ori = hdr[5];
    const std::vector<float> fl = rd<float>(f, 7);                // bounds(4), grid inv(2), nnratio
    const std::vector<float> scale = rd<float>(f, nlev);
    Frame::mnMinX = fl[0]; Frame::mnMinY = fl[1]; Frame::mnMaxX = fl[2]; Frame::mnMaxY = fl[3];
    Frame::mfGridElementWidthInv = fl[4]; Frame::mfGridElementHeightInv = fl[5];
    Frame F1, F2, F3;
    std::vector<unsigned char> d1, d2, d3;
    read_frame(f, F1, d1, n1, scale);
    read_frame(f, F2, d2, n2, scale);
    read_frame(f, F3, d3, n3, scale);
    std::fclose(f);
    // Tracking::MonocularInitialization: mvbPrevMatched[i] = mInitialFrame.mvKeysUn[i].pt
    std::vector<cv::Point2f> vbPrevMatched(n1);
    for (int i = 0; i < n1; ++i) vbPrevMatched[i] = F1.mvKeysUn[i].pt;
    std::vector<int> vnMatches12;
    ORBmatcher matcher(fl[6], check_ori != 0);
    FILE* g = std::fopen(argv[2], "wb");
    for (Frame* Fk : {&F2, &F3}) {
        const int nm = matcher.SearchForInitialization(F1, *Fk, vbPrevMatched, vnMatches12, window);
        std::fwrite(&nm, 4, 1, g);
        std::fwrite(vnMatches12.data(), 4, n1, g);
        std::fwrite(vbPrevMatched.data(), 8, n1, g);
        std::printf("nmatches=%d\n", nm);
    }
    std::fclose(g);
    return 0;
}
