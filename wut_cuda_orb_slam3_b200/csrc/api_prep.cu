// api_prep.cu — host side of the preparation steps either side of the extractor (C ABI of include/orbx.h).
//
// Reference interfaces replaced (paths relative to the reference root):
//   Frame::UndistortKeyPoints                src/Frame.cc:777-810     (cv::undistortPoints)
//   System::TrackStereo's rectification      src/System.cc:253-260    (cv::remap with the maps of src/Settings.cc:488-491)
#include <cfloat>
#include <cmath>
#include <cstring>
#include <vector>

#include "orbx_internal.cuh"

struct orbx_rectifier {
    int device = 0, dw = 0, dh = 0;
    uint2* d_packed = nullptr;      // remap: quantised map; resize: x table (dw entries) then y table (dh entries)
    int resize = 0, src_w = 0, src_h = 0, area2x = 0;
    // single-image staging (grow-only)
    uint8_t *d_src = nullptr, *d_dst = nullptr;
    size_t src_bytes = 0, dst_bytes = 0;
    cudaStream_t st = nullptr;
};

using namespace orbx;

extern "C" {

int orbx_undistort_keypoints(int device, const orbx_keypoint* keypoints, int n, const float* K, const float* dist, int n_dist,
                             const float* new_K, orbx_keypoint* out)
{
    if (n < 0 || (n > 0 && (!keypoints || !out)) || !K || !new_K || n_dist < 0 || n_dist > 12 || (n_dist > 0 && !dist))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (n_dist == 0 || dist[0] == 0.0) {                                   // src/Frame.cc:779-783
        if (n && out != keypoints) memmove(out, keypoints, (size_t)n * sizeof(orbx_keypoint));
        return ORBX_OK;
    }
    int rc;
    if ((rc = set_device(device))) return rc;
    if (n == 0) return ORBX_OK;
    UndistortParams p{};
    p.fx = K[0]; p.fy = K[1]; p.cx = K[2]; p.cy = K[3];
    p.nfx = new_K[0]; p.nfy = new_K[1]; p.ncx = new_K[2]; p.ncy = new_K[3];
    for (int i = 0; i < n_dist; ++i) p.k[i] = dist[i];
    p.n_dist = n_dist;
    const size_t bytes = (size_t)n * sizeof(orbx_keypoint);
    Lease L(device);
    if ((rc = L.reserve(lease_pad(bytes)))) return rc;
    const size_t o_kp = L.take<orbx_keypoint>(n);
    L.upload_end = L.off;
    memcpy(L.host<orbx_keypoint>(o_kp), keypoints, bytes);
    orbx_keypoint* d_kp = L.dev<orbx_keypoint>(o_kp);
    cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, L.A.st);
    if (e == cudaSuccess) e = launch_undistort(d_kp, n, p, d_kp, L.A.st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(L.host<orbx_keypoint>(o_kp), d_kp, bytes, cudaMemcpyDeviceToHost, L.A.st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(L.A.st);
    if (e == cudaSuccess) memcpy(out, L.host<orbx_keypoint>(o_kp), bytes);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "undistort_keypoints: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

int orbx_rectifier_create(int device, const float* map_x, const float* map_y, size_t map_step_bytes, int dst_rows, int dst_cols,
                          orbx_rectifier** out)
{
    if (!out) return fail(ORBX_ERR_INVALID_ARG, "null output");
    *out = nullptr;
    if (!map_x || !map_y || dst_rows <= 0 || dst_cols <= 0 || map_step_bytes < (size_t)dst_cols * 4 || (map_step_bytes & 3))
        return fail(ORBX_ERR_INVALID_ARG, "bad rectification maps");
    int rc;
    if ((rc = set_device(device))) return rc;
    orbx_rectifier* r = new orbx_rectifier;
    r->device = device; r->dw = dst_cols; r->dh = dst_rows;
    const size_t n = (size_t)dst_rows * dst_cols;
    float *dx = nullptr, *dy = nullptr;
    cudaError_t e = cudaMalloc(&r->d_packed, n * sizeof(uint2));
    if (e == cudaSuccess) e = cudaMalloc(&dx, n * 4);
    if (e == cudaSuccess) e = cudaMalloc(&dy, n * 4);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r->st, cudaStreamNonBlocking);
    // stream-ordered copies: a synchronous copy from pageable memory may return before its DMA lands, and r->st is non-blocking
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(dx, (size_t)dst_cols * 4, map_x, map_step_bytes, (size_t)dst_cols * 4, dst_rows, cudaMemcpyHostToDevice, r->st);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(dy, (size_t)dst_cols * 4, map_y, map_step_bytes, (size_t)dst_cols * 4, dst_rows, cudaMemcpyHostToDevice, r->st);
    if (e == cudaSuccess) e = launch_remap_quantise(dx, dy, (size_t)dst_cols, dst_cols, dst_rows, r->d_packed, r->st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(r->st);
    cudaFree(dx); cudaFree(dy);
    if (e != cudaSuccess) { orbx_rectifier_destroy(r); return fail(ORBX_ERR_CUDA, "rectifier_create: %s", cudaGetErrorString(e)); }
    *out = r;
    return ORBX_OK;
}

int orbx_resizer_create(int device, int src_rows, int src_cols, int dst_rows, int dst_cols, orbx_rectifier** out)
{
    if (!out) return fail(ORBX_ERR_INVALID_ARG, "null output");
    *out = nullptr;
    if (src_rows <= 0 || src_cols <= 0 || dst_rows <= 0 || dst_cols <= 0 || src_rows > 65535 || src_cols > 65535)
        return fail(ORBX_ERR_INVALID_ARG, "bad sizes");
    int rc;
    if ((rc = set_device(device))) return rc;
    // cv::resize: inv_scale = dsize / ssize, scale = 1 / inv_scale; INTER_LINEAR turns into the INTER_AREA average for exact 2x
    const double scale_x = 1. / ((double)dst_cols / src_cols), scale_y = 1. / ((double)dst_rows / src_rows);
    const int iscale_x = (int)lrint(scale_x), iscale_y = (int)lrint(scale_y);
    const bool area_fast = std::abs(scale_x - iscale_x) < DBL_EPSILON && std::abs(scale_y - iscale_y) < DBL_EPSILON;
    const int area2x = (area_fast && iscale_x == 2 && iscale_y == 2) ? 1 : 0;
    // Columns clamp (sx, fx) at the image edges; rows keep (sy, fy) and clip the two row indices instead (cv::resize computes
    // yofs without clamping and resizeGeneric_Invoker clips the rows) — the two differ on up-scales only.
    auto entry = [&](int d, double sc, int n, bool clamp) -> uint2 {
        if (area2x) return make_uint2((uint32_t)(2 * d) | ((uint32_t)(2 * d + 1) << 16), 1u | (1u << 16));
        float f = (float)((d + 0.5) * sc - 0.5);
        int s = (int)floorf(f);
        f -= s;
        if (clamp && s < 0) { s = 0; f = 0.f; }
        if (clamp && s >= n - 1) { s = n - 1; f = 0.f; }
        const int c0 = (short)lrintf((1.f - f) * 2048.f), c1 = (short)lrintf(f * 2048.f);
        const int s0 = std::min(std::max(s, 0), n - 1), s1 = std::min(std::max(s + 1, 0), n - 1);
        return make_uint2((uint32_t)s0 | ((uint32_t)s1 << 16), ((uint32_t)c0 & 0xffffu) | ((uint32_t)c1 << 16));
    };
    std::vector<uint2> tab;
    for (int x = 0; x < dst_cols; ++x) tab.push_back(entry(x, scale_x, src_cols, true));
    for (int y = 0; y < dst_rows; ++y) tab.push_back(entry(y, scale_y, src_rows, false));
    orbx_rectifier* r = new orbx_rectifier;
    r->device = device; r->dw = dst_cols; r->dh = dst_rows; r->resize = 1; r->src_w = src_cols; r->src_h = src_rows; r->area2x = area2x;
    cudaError_t e = cudaMalloc(&r->d_packed, tab.size() * sizeof(uint2));
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&r->st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMemcpyAsync(r->d_packed, tab.data(), tab.size() * sizeof(uint2), cudaMemcpyHostToDevice, r->st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(r->st);
    if (e != cudaSuccess) { orbx_rectifier_destroy(r); return fail(ORBX_ERR_CUDA, "resizer_create: %s", cudaGetErrorString(e)); }
    *out = r;
    return ORBX_OK;
}

void orbx_rectifier_destroy(orbx_rectifier* r)
{
    if (!r) return;
    cudaSetDevice(r->device);
    cudaFree(r->d_packed); cudaFree(r->d_src); cudaFree(r->d_dst);
    if (r->st) cudaStreamDestroy(r->st);
    delete r;
}

int orbx_remap_device(orbx_rectifier* r, const uint8_t* d_src, int src_rows, int src_cols, size_t src_pitch, size_t src_frame_stride,
                      int n_frames, uint8_t* d_dst, size_t dst_pitch, size_t dst_frame_stride, void* stream)
{
    if (!r || !d_src || !d_dst || src_rows <= 0 || src_cols <= 0 || src_pitch < (size_t)src_cols || dst_pitch < (size_t)r->dw || n_frames < 0)
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc;
    if ((rc = set_device(r->device))) return rc;
    if (r->resize && (src_cols != r->src_w || src_rows != r->src_h))
        return fail(ORBX_ERR_INVALID_ARG, "resizer was created for %dx%d sources, got %dx%d", r->src_w, r->src_h, src_cols, src_rows);
    cudaError_t e = r->resize ? launch_resize(d_src, src_pitch, src_frame_stride, r->d_packed, r->d_packed + r->dw, r->area2x, d_dst, r->dw, r->dh,
                                              dst_pitch, dst_frame_stride, n_frames, (cudaStream_t)stream)
                              : launch_remap(d_src, src_cols, src_rows, src_pitch, src_frame_stride, r->d_packed, d_dst, r->dw, r->dh, dst_pitch,
                                             dst_frame_stride, n_frames, (cudaStream_t)stream);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "remap: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

int orbx_remap(orbx_rectifier* r, const uint8_t* src, int src_rows, int src_cols, size_t src_step, uint8_t* dst, size_t dst_step)
{
    if (!r || !src || !dst || src_rows <= 0 || src_cols <= 0 || src_step < (size_t)src_cols || dst_step < (size_t)r->dw)
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc;
    if ((rc = set_device(r->device))) return rc;
    const size_t spitch = ((size_t)src_cols + 15) & ~(size_t)15, dpitch = ((size_t)r->dw + 15) & ~(size_t)15;
    const size_t sb = spitch * src_rows, db = dpitch * r->dh;
    cudaError_t e = cudaSuccess;
    if (r->src_bytes < sb) { cudaFree(r->d_src); r->d_src = nullptr; r->src_bytes = 0; e = cudaMalloc(&r->d_src, sb); if (e == cudaSuccess) r->src_bytes = sb; }
    if (e == cudaSuccess && r->dst_bytes < db) { cudaFree(r->d_dst); r->d_dst = nullptr; r->dst_bytes = 0; e = cudaMalloc(&r->d_dst, db); if (e == cudaSuccess) r->dst_bytes = db; }
    if (e != cudaSuccess) return fail(ORBX_ERR_OOM, "remap staging: %s", cudaGetErrorString(e));
    e = cudaMemcpy2DAsync(r->d_src, spitch, src, src_step, (size_t)src_cols, src_rows, cudaMemcpyHostToDevice, r->st);
    if (e == cudaSuccess && r->resize && (src_cols != r->src_w || src_rows != r->src_h))
        return fail(ORBX_ERR_INVALID_ARG, "resizer was created for %dx%d sources, got %dx%d", r->src_w, r->src_h, src_cols, src_rows);
    if (e == cudaSuccess)
        e = r->resize ? launch_resize(r->d_src, spitch, 0, r->d_packed, r->d_packed + r->dw, r->area2x, r->d_dst, r->dw, r->dh, dpitch, 0, 1, r->st)
                      : launch_remap(r->d_src, src_cols, src_rows, spitch, 0, r->d_packed, r->d_dst, r->dw, r->dh, dpitch, 0, 1, r->st);
    if (e == cudaSuccess) e = cudaMemcpy2DAsync(dst, dst_step, r->d_dst, dpitch, (size_t)r->dw, r->dh, cudaMemcpyDeviceToHost, r->st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(r->st);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "remap: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

}  // extern "C"
