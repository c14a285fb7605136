// rgbd_oracle.cpp — CPU ORACLE (TEST INFRASTRUCTURE ONLY, never shipped, never on the product path).
//
// The depth side of an RGB-D frame, restated from the reference:
//   Tracking::GrabImageRGBD (src/Tracking2.cc)      if ((fabs(mDepthMapFactor - 1.0f) > 1e-5) || imDepth.type() != CV_32F)
//                                                       imDepth.convertTo(imDepth, CV_32F, mDepthMapFactor);
//   Frame::ComputeStereoFromRGBD (src/Frame.cc:1014-1035)
//       const float d = imDepth.at<float>(v, u) with v = (int)kp.pt.y, u = (int)kp.pt.x of the DISTORTED keypoint mvKeys[i];
//       if (d > 0) { mvDepth[i] = d; mvuRight[i] = mvKeysUn[i].pt.x - mbf / d; }   (both -1 otherwise)
// convertTo(CV_32F, alpha) is OpenCV's cvt_32f: alpha and beta = 0 are cast to float and every element becomes (float)v * alpha + 0,
// one rounding (the + 0 only turns a -0 product into +0); tests/test_rgbd_cpu.py pins this restatement to cv2 bit for bit.  Built
// with -ffp-contract=off.
#include <cmath>
#include <cstddef>
#include <cstdint>
#include <vector>

namespace {
struct KeyPoint { float x, y, size, angle, response; int octave, class_id; };
}  // namespace

extern "C" {

// Tracking::GrabImageRGBD's predicate and conversion over the whole map.  depth_type 0 = CV_16U, 1 = CV_32F; dst is rows x cols
// floats.  Returns 1 when convertTo ran (on a CV_32F map that does not convert, dst is a copy).
int orbo_grab_depth(const void* depth, int depth_type, size_t depth_step, int rows, int cols, float depth_factor, float* dst)
{
    const bool convert = (std::fabs(depth_factor - 1.0f) > 1e-5) || depth_type != 1;
    const float alpha = depth_factor;
    for (int y = 0; y < rows; ++y) {
        const unsigned char* row = (const unsigned char*)depth + (size_t)y * depth_step;
        for (int x = 0; x < cols; ++x) {
            const float v = depth_type == 0 ? (float)((const uint16_t*)row)[x] : ((const float*)row)[x];
            dst[(size_t)y * cols + x] = convert ? v * alpha + 0.0f : v;
        }
    }
    return convert ? 1 : 0;
}

// Frame::ComputeStereoFromRGBD on a converted (CV_32F, rows x cols, dense) map.
void orbo_compute_stereo_from_rgbd(const float* depth, int rows, int cols, const KeyPoint* keys, const KeyPoint* keys_un, int n, float bf,
                                   float* uRight, float* depth_out)
{
    (void)rows;
    for (int i = 0; i < n; ++i) {
        uRight[i] = -1; depth_out[i] = -1;
        const int v = (int)keys[i].y, u = (int)keys[i].x;
        const float d = depth[(size_t)v * cols + u];
        if (d > 0) {
            depth_out[i] = d;
            uRight[i] = keys_un[i].x - bf / d;
        }
    }
}

// Both, as the RGB-D Frame reaches them: the raw map through GrabImageRGBD, then ComputeStereoFromRGBD.
void orbo_rgbd_depth(const void* depth, int depth_type, size_t depth_step, int rows, int cols, float depth_factor, const KeyPoint* keys,
                     const KeyPoint* keys_un, int n, float bf, float* uRight, float* depth_out)
{
    std::vector<float> map((size_t)rows * cols);
    orbo_grab_depth(depth, depth_type, depth_step, rows, cols, depth_factor, map.data());
    orbo_compute_stereo_from_rgbd(map.data(), rows, cols, keys, keys_un, n, bf, uRight, depth_out);
}

}  // extern "C"
