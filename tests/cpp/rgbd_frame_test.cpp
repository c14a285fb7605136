// The RGB-D Frame constructor body of INTEGRATION.md, compiled against the cv stub and a Frame stand-in with the members the
// snippet touches, and run on a seeded frame: tests/test_rgbd_cpu.py builds it, tests/test_gpu_rgbd.py compares what it writes
// with orbx.extract_rgbd on the same inputs.
//   rgbd_frame_test <seed> <out.bin>   writes N, mvKeys, mvKeysUn, mDescriptors, mvuRight, mvDepth
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <vector>

#include "ORBextractor.h"

#ifndef CV_16U
#define CV_16U 2
#endif

// cv::Mat of a depth map, as far as the snippet reads it (the stub's cv::Mat is 8-bit only)
struct DepthMat {
    unsigned char* data;
    size_t step;
    int t;
    int type() const { return t; }
};

struct Frame {
    cv::Mat mK, mDistCoef;
    float mbf = 0;
    int N = 0;
    std::vector<cv::KeyPoint> mvKeys, mvKeysUn;
    std::vector<float> mvuRight, mvDepth;
    cv::Mat mDescriptors;
    ORB_SLAM3::ORBextractor* mpORBextractorLeft;

    Frame(const cv::Mat& imGray, const DepthMat& imDepth, ORB_SLAM3::ORBextractor* extractor, const cv::Mat& K, const cv::Mat& distCoef,
          float bf, float depthMapFactor)
        : mK(K), mDistCoef(distCoef), mbf(bf), mpORBextractorLeft(extractor)
    {
        // ---- INTEGRATION.md §1 step 4c: the body of Frame::Frame(imGray, imDepth, ...) from ExtractORB to ComputeStereoFromRGBD ----
        orbx_extractor* h = mpORBextractorLeft->nativeHandle();
        const int cap = orbx_max_keypoints_for(h, imGray.rows, imGray.cols);
        mvKeys.resize(cap); mvKeysUn.resize(cap); mvuRight.resize(cap); mvDepth.resize(cap);
        cv::Mat desc;
        desc.create(cap, 32, CV_8U);
        const float* k = (const float*)mK.data;                  // the 3x3 CV_32F camera matrix
        const orbx_rgbd_calib calib = {{k[0], k[4], k[2], k[5]}, (const float*)mDistCoef.data, mDistCoef.rows * mDistCoef.cols, mbf, depthMapFactor};
        int n = 0;
        if (orbx_extract_rgbd(h, imGray.data, imGray.rows, imGray.cols, imGray.step, 1, 0, imDepth.data, imDepth.type() == CV_16U ? 0 : 1,
                              imDepth.step, &calib, reinterpret_cast<orbx_keypoint*>(mvKeys.data()),
                              reinterpret_cast<orbx_keypoint*>(mvKeysUn.data()), desc.data, cap, &n, mvuRight.data(),
                              mvDepth.data()) != ORBX_OK)
            throw std::runtime_error(orbx_last_error());
        N = n;
        mvKeys.resize(N); mvKeysUn.resize(N); mvuRight.resize(N); mvDepth.resize(N);
        mDescriptors.create(N, 32, CV_8U);
        if (N) std::memcpy(mDescriptors.data, desc.data, (size_t)N * 32);
        // ---- end of the snippet ----
    }
};

int main(int argc, char** argv)
{
    if (argc < 3) { std::fprintf(stderr, "usage: rgbd_frame_test <seed> <out.bin>\n"); return 2; }
    const int cols = 640, rows = 480;
    std::vector<unsigned char> gray((size_t)cols * rows);
    orbx_synth_image_host((uint32_t)atoi(argv[1]), 0, cols, rows, 48, gray.data(), cols);
    // raw TUM-style depth (u16, 5000 per metre) that follows the pixel, with holes (the same map as test_snippet_on_the_gpu)
    std::vector<uint16_t> depth((size_t)cols * rows);
    for (int y = 0; y < rows; ++y)
        for (int x = 0; x < cols; ++x) depth[(size_t)y * cols + x] = (x + y) % 7 == 0 ? 0 : (uint16_t)(1000 + y * 97 + x);
    float km[9] = {517.306408f, 0, 318.643040f, 0, 516.469215f, 255.313989f, 0, 0, 1};
    float k[5] = {0.262383f, -0.953104f, -0.005358f, 0.002628f, 1.163314f};     // TUM1
    cv::Mat dist(1, 5, CV_8U, k);
    ORB_SLAM3::ORBextractor ex(1000, 1.2f, 8, 20, 7);
    Frame f(cv::Mat(rows, cols, CV_8UC1, gray.data()), DepthMat{(unsigned char*)depth.data(), (size_t)cols * 2, CV_16U}, &ex, cv::Mat(3, 3, CV_8U, km), dist, 40.0f,
            1.0f / 5000.0f);
    FILE* o = std::fopen(argv[2], "wb");
    if (!o) return 1;
    std::fwrite(&f.N, sizeof(int), 1, o);
    std::fwrite(f.mvKeys.data(), sizeof(cv::KeyPoint), f.N, o);
    std::fwrite(f.mvKeysUn.data(), sizeof(cv::KeyPoint), f.N, o);
    std::fwrite(f.mDescriptors.data, 32, f.N, o);
    std::fwrite(f.mvuRight.data(), sizeof(float), f.N, o);
    std::fwrite(f.mvDepth.data(), sizeof(float), f.N, o);
    std::fclose(o);
    std::printf("N=%d\n", f.N);
    return 0;
}
