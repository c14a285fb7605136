// kernels_prep.cu — preparation steps either side of the extractor (SURVEY.md §8(f)3).
//
//   * Frame::UndistortKeyPoints (src/Frame.cc:777-810) = cv::undistortPoints(pts, K, mDistCoef, R = I, P = mK): normalise,
//     5 fixed-point iterations of the inverse radial-tangential distortion, re-project; double arithmetic, float results.
//     One thread per key point; --fmad=false keeps every multiply and add separately rounded like the x86-64 build of OpenCV.
//   * The RGB-D Frame constructor's tail (src/Frame.cc:202-260): the same undistortion plus ComputeStereoFromRGBD, one depth
//     sample per key point (rgbd_frame_kernel).
//   * System::TrackStereo rectification (src/System.cc:253-260) = cv::remap(im, out, M1, M2, INTER_LINEAR) with CV_32FC1 maps:
//     the map is quantised ONCE to OpenCV's 1/32-pixel fixed point (remap_quantise_kernel), every frame then costs four
//     gathers and one 15-bit fixed-point blend per pixel.  The packed map (8 bytes per pixel) stays L2-resident across a
//     batch, so HBM sees the source and destination bytes only; a thread produces 4 adjacent pixels and stores them as one word.
#include <climits>

#include "orbx_internal.cuh"

namespace orbx {

__device__ __forceinline__ orbx_keypoint undistort_point(orbx_keypoint kp, const UndistortParams& p)
{
    const double* k = p.k;
    const double ifx = 1. / p.fx, ify = 1. / p.fy;
    const double u = kp.x, v = kp.y;
    double x = (u - p.cx) * ifx, y = (v - p.cy) * ify;
    if (p.n_dist > 0) {
        const double x0 = x, y0 = y;
        for (int j = 0; j < 5; ++j) {
            const double r2 = x * x + y * y;
            const double icdist = (1 + ((k[7] * r2 + k[6]) * r2 + k[5]) * r2) / (1 + ((k[4] * r2 + k[1]) * r2 + k[0]) * r2);
            if (icdist < 0) { x = (u - p.cx) * ifx; y = (v - p.cy) * ify; break; }
            const double deltaX = 2 * k[2] * x * y + k[3] * (r2 + 2 * x * x) + k[8] * r2 + k[9] * r2 * r2;
            const double deltaY = k[2] * (r2 + 2 * y * y) + 2 * k[3] * x * y + k[10] * r2 + k[11] * r2 * r2;
            x = (x0 - deltaX) * icdist;
            y = (y0 - deltaY) * icdist;
        }
    }
    const double xx = p.nfx * x + 0.0 * y + p.ncx;
    const double yy = 0.0 * x + p.nfy * y + p.ncy;
    const double ww = 1. / (0.0 * x + 0.0 * y + 1.0);
    kp.x = (float)(xx * ww);
    kp.y = (float)(yy * ww);
    return kp;
}

__global__ void __launch_bounds__(128) undistort_kernel(const orbx_keypoint* __restrict__ in, int n, UndistortParams p,
                                                        orbx_keypoint* __restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    out[i] = undistort_point(in[i], p);
}

// The tail of the RGB-D Frame constructor (src/Frame.cc:202-260) per keypoint, grid (ceil(capacity / 128), frames): mvKeysUn
// (UndistortKeyPoints, :777-810), then ComputeStereoFromRGBD (:1014-1035) on ONE depth sample at the truncated coordinates of
// the DISTORTED keypoint.  Tracking::GrabImageRGBD's convertTo(CV_32F, mDepthMapFactor) is element-wise, so converting only the
// sampled pixel gives the same float as converting the whole map: fl32((float)v * factor), one rounding (OpenCV's + 0 only turns
// a -0 product into +0, which `d > 0` does not tell apart).  The index is in
// bounds by construction (keypoints keep EDGE_THRESHOLD - 3 pixels from every level's edge).  A frame whose count exceeds the
// capacity has no keypoint rows: nothing is read or written for it.
__global__ void __launch_bounds__(128) rgbd_frame_kernel(RgbdArgs a)
{
    const int f = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
    const int n = a.n[f];
    if (n > a.capacity || i >= n) return;
    const size_t r = (size_t)f * a.capacity + i;
    const orbx_keypoint kp = a.kp[r];
    const orbx_keypoint un = a.undistort ? undistort_point(kp, a.p) : kp;
    a.kp_un[r] = un;
    const uint8_t* row = a.depth + (size_t)f * a.depth_frame_stride + (size_t)(int)kp.y * a.depth_pitch;
    float d = a.depth_type == 0 ? (float)reinterpret_cast<const uint16_t*>(row)[(int)kp.x] : reinterpret_cast<const float*>(row)[(int)kp.x];
    if (a.convert) d = __fmul_rn(d, a.factor);
    float u = -1.f, z = -1.f;
    if (d > 0) { z = d; u = __fsub_rn(un.x, __fdiv_rn(a.bf, d)); }
    a.uRight[r] = u;
    a.depth_out[r] = z;
}

// cvRound(map * 32) -> (sx | sy << 16, fx | fy << 5); sx, sy saturate to int16 like OpenCV's XY buffer.
__global__ void __launch_bounds__(256) remap_quantise_kernel(const float* __restrict__ mapx, const float* __restrict__ mapy,
                                                             size_t map_step, int dw, int dh, uint2* __restrict__ packed)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y;
    if (x >= dw || y >= dh) return;
    const int sxq = __float2int_rn(__fmul_rn(mapx[(size_t)y * map_step + x], 32.0f));
    const int syq = __float2int_rn(__fmul_rn(mapy[(size_t)y * map_step + x], 32.0f));
    const int sx = max(-32768, min(32767, sxq >> 5)), sy = max(-32768, min(32767, syq >> 5));
    packed[(size_t)y * dw + x] = make_uint2(((uint32_t)sx & 0xffffu) | ((uint32_t)sy << 16), (uint32_t)(sxq & 31) | ((uint32_t)(syq & 31) << 5));
}

// grid (ceil(dw / 4 / 128), dh, ceil(frames / FPT)): a thread = 4 adjacent destination pixels of FPT consecutive frames.  The
// four map entries (32 bytes) and the 16 bilinear weights are loaded / computed once and reused for every frame of the group:
// the packed map is 8 bytes per pixel against 2 bytes of image traffic, so reading it per frame made L2 the bottleneck.
struct RemapTap { int off; int w0, w1, w2, w3; unsigned valid; };     // valid: bit0..3 = taps 00, 01, 10, 11 inside the image
__device__ __forceinline__ RemapTap remap_tap(uint2 m, int sw, int sh, size_t spitch)
{
    RemapTap t;
    const int sx = (int)(short)(m.x & 0xffffu), sy = (int)(short)(m.x >> 16);
    const int fx = (int)(m.y & 31u), fy = (int)(m.y >> 5);
    t.w0 = (32 - fy) * (32 - fx) * 32; t.w3 = fy * fx * 32;
    t.w1 = (32 - fy) * fx * 32; t.w2 = fy * (32 - fx) * 32;
    if (t.w0 == 32768) { t.w0 = 32767; t.w3 = 1; }          // saturate_cast<short>(32768) and OpenCV's sum fix-up
    const bool x0 = (unsigned)sx < (unsigned)sw, x1 = (unsigned)(sx + 1) < (unsigned)sw;
    const bool y0 = (unsigned)sy < (unsigned)sh, y1 = (unsigned)(sy + 1) < (unsigned)sh;
    t.valid = (x0 && y0 ? 1u : 0u) | (x1 && y0 ? 2u : 0u) | (x0 && y1 ? 4u : 0u) | (x1 && y1 ? 8u : 0u);
    t.off = t.valid ? sy * (int)spitch + sx : 0;            // BORDER_CONSTANT 0: taps outside the image read 0
    return t;
}
__device__ __forceinline__ uint32_t remap_apply(const uint8_t* __restrict__ s, const RemapTap& t, int spitch)
{
    int p00 = 0, p01 = 0, p10 = 0, p11 = 0;
    const uint8_t* q = s + t.off;
    if (t.valid == 15u) { p00 = __ldg(q); p01 = __ldg(q + 1); p10 = __ldg(q + spitch); p11 = __ldg(q + spitch + 1); }
    else {
        if (t.valid & 1u) p00 = __ldg(q);
        if (t.valid & 2u) p01 = __ldg(q + 1);
        if (t.valid & 4u) p10 = __ldg(q + spitch);
        if (t.valid & 8u) p11 = __ldg(q + spitch + 1);
    }
    return (uint32_t)((p00 * t.w0 + p01 * t.w1 + p10 * t.w2 + p11 * t.w3 + (1 << 14)) >> 15);
}

template <int FPT>
__global__ void __launch_bounds__(128, 8) remap_kernel(const uint8_t* __restrict__ src, int sw, int sh, size_t spitch, size_t sframe,
                                                       const uint2* __restrict__ packed, uint8_t* __restrict__ dst, int dw, int dh,
                                                       size_t dpitch, size_t dframe, int n_frames)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x4 >= dw) return;
    const int f0 = blockIdx.z * FPT, nf = min(FPT, n_frames - f0);
    const uint2* m = packed + (size_t)y * dw + x4;
    const int npx = min(4, dw - x4);
    RemapTap t[4];
    if (npx == 4 && ((dw & 1) == 0)) {                       // 16-byte aligned pair of entries
        const uint4 ma = __ldg(reinterpret_cast<const uint4*>(m)), mb = __ldg(reinterpret_cast<const uint4*>(m) + 1);
        t[0] = remap_tap(make_uint2(ma.x, ma.y), sw, sh, spitch); t[1] = remap_tap(make_uint2(ma.z, ma.w), sw, sh, spitch);
        t[2] = remap_tap(make_uint2(mb.x, mb.y), sw, sh, spitch); t[3] = remap_tap(make_uint2(mb.z, mb.w), sw, sh, spitch);
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) t[j] = remap_tap(j < npx ? __ldg(m + j) : make_uint2(0, 0), sw, sh, spitch);
    }
    const uint8_t* s = src + (size_t)f0 * sframe;
    uint8_t* d = dst + (size_t)f0 * dframe + (size_t)y * dpitch + x4;
    const int sp = (int)spitch;
    if (npx == 4 && (t[0].valid & t[1].valid & t[2].valid & t[3].valid) == 15u && ((reinterpret_cast<size_t>(d) | dframe) & 3) == 0) {
        // interior: all 16 taps inside the image, one word store per frame; every frame's loads are independent of the others
        const uint8_t *q0 = s + t[0].off, *q1 = s + t[1].off, *q2 = s + t[2].off, *q3 = s + t[3].off;
#pragma unroll
        for (int f = 0; f < FPT; ++f) {
            if (f < nf) {
                const int a = __ldg(q0) * t[0].w0 + __ldg(q0 + 1) * t[0].w1 + __ldg(q0 + sp) * t[0].w2 + __ldg(q0 + sp + 1) * t[0].w3;
                const int b = __ldg(q1) * t[1].w0 + __ldg(q1 + 1) * t[1].w1 + __ldg(q1 + sp) * t[1].w2 + __ldg(q1 + sp + 1) * t[1].w3;
                const int c = __ldg(q2) * t[2].w0 + __ldg(q2 + 1) * t[2].w1 + __ldg(q2 + sp) * t[2].w2 + __ldg(q2 + sp + 1) * t[2].w3;
                const int e = __ldg(q3) * t[3].w0 + __ldg(q3 + 1) * t[3].w1 + __ldg(q3 + sp) * t[3].w2 + __ldg(q3 + sp + 1) * t[3].w3;
                *reinterpret_cast<uint32_t*>(d) = (uint32_t)((a + 16384) >> 15) | ((uint32_t)((b + 16384) >> 15) << 8) |
                                                  ((uint32_t)((c + 16384) >> 15) << 16) | ((uint32_t)((e + 16384) >> 15) << 24);
                q0 += sframe; q1 += sframe; q2 += sframe; q3 += sframe; d += dframe;
            }
        }
        return;
    }
    for (int f = 0; f < nf; ++f, s += sframe, d += dframe) {
        const uint32_t v[4] = {remap_apply(s, t[0], sp), remap_apply(s, t[1], sp), remap_apply(s, t[2], sp), remap_apply(s, t[3], sp)};
        for (int j = 0; j < npx; ++j) d[j] = (uint8_t)v[j];
    }
}

// ---- tiled variant for batches: the source window of a 128 x 8 destination tile is staged in shared memory --------------------
// A rectification map is smooth, so the taps of a destination tile fall into a compact source window (a few KB).  Per CTA: map
// entries, weights and the window are worked out ONCE, then for every frame of the group the window is copied with coalesced
// 16-byte loads (double buffered: frame f + 1 is fetched while frame f is blended) and the four taps per pixel come from shared
// memory instead of four scattered byte loads through L1/L2.  Tiles whose window does not fit (wild maps) or whose source is
// not 16-byte aligned take the gather path of remap_kernel.
constexpr int RT_W = 128, RT_H = 8, RT_THREADS = 256, RT_SMEM = 4096, RT_STAGES = 4, RT_FPC = 32;

__device__ __forceinline__ int nitems_of(int SP, int nrow) { return (SP >> 4) * nrow; }

__global__ void __launch_bounds__(RT_THREADS, 4) remap_tiled_kernel(const uint8_t* __restrict__ src, int sw, int sh, size_t spitch, size_t sframe,
                                                                 const uint2* __restrict__ packed, uint8_t* __restrict__ dst, int dw, int dh,
                                                                 size_t dpitch, size_t dframe, int n_frames)
{
    __shared__ __align__(16) uint8_t win[RT_STAGES][RT_SMEM];
    __shared__ int s_box[4];                                  // min sx, max sx + 1, min sy, max sy + 1 over the taps inside the image
    const int tid = threadIdx.x, lane = tid & 31;
    const int x4 = blockIdx.x * RT_W + lane * 4, y = blockIdx.y * RT_H + (tid >> 5);
    const int f0 = blockIdx.z * RT_FPC, nf = min(RT_FPC, n_frames - f0);
    const bool row_ok = y < dh;
    const int npx = row_ok ? max(0, min(4, dw - x4)) : 0;
    if (tid == 0) { s_box[0] = INT_MAX; s_box[1] = -1; s_box[2] = INT_MAX; s_box[3] = -1; }
    __syncthreads();
    RemapTap t[4];
    int bx0 = INT_MAX, bx1 = -1, by0 = INT_MAX, by1 = -1;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint2 m = j < npx ? __ldg(packed + (size_t)y * dw + x4 + j) : make_uint2(0x80008000u, 0);   // sx = sy = -32768: no tap inside
        t[j] = remap_tap(m, sw, sh, spitch);
        if (t[j].valid) {
            const int sx = (int)(short)(m.x & 0xffffu), sy = (int)(short)(m.x >> 16);
            bx0 = min(bx0, max(sx, 0)); bx1 = max(bx1, min(sx + 1, sw - 1));
            by0 = min(by0, max(sy, 0)); by1 = max(by1, min(sy + 1, sh - 1));
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        bx0 = min(bx0, __shfl_xor_sync(0xffffffffu, bx0, d)); bx1 = max(bx1, __shfl_xor_sync(0xffffffffu, bx1, d));
        by0 = min(by0, __shfl_xor_sync(0xffffffffu, by0, d)); by1 = max(by1, __shfl_xor_sync(0xffffffffu, by1, d));
    }
    if (lane == 0 && bx1 >= 0) { atomicMin(&s_box[0], bx0); atomicMax(&s_box[1], bx1); atomicMin(&s_box[2], by0); atomicMax(&s_box[3], by1); }
    __syncthreads();
    const int X0 = s_box[0] & ~15, X1 = s_box[1], Y0 = s_box[2], Y1 = s_box[3];
    const bool any = X1 >= 0;
    const int nvec = any ? ((X1 - X0) >> 4) + 1 : 0, nrow = any ? Y1 - Y0 + 1 : 0, SP = nvec * 16;
    uint8_t* d = dst + (size_t)f0 * dframe + (size_t)y * dpitch + x4;
    const uint8_t* s = src + (size_t)f0 * sframe;
    const bool word_store = npx == 4 && ((reinterpret_cast<size_t>(d) | dframe) & 3) == 0;
    if (!any) {                                               // the whole tile maps outside the image: BORDER_CONSTANT 0
        for (int f = 0; f < nf; ++f, d += dframe)
            for (int j = 0; j < npx; ++j) d[j] = 0;
        return;
    }
    if (SP * nrow > RT_SMEM || nitems_of(SP, nrow) > RT_THREADS || (size_t)X0 + (size_t)SP > spitch) {   // window too large / would run over the row pitch: gather
        for (int f = 0; f < nf; ++f, s += sframe, d += dframe) {
            const uint32_t v[4] = {remap_apply(s, t[0], (int)spitch), remap_apply(s, t[1], (int)spitch), remap_apply(s, t[2], (int)spitch),
                                   remap_apply(s, t[3], (int)spitch)};
            for (int j = 0; j < npx; ++j) d[j] = (uint8_t)v[j];
        }
        return;
    }
    // tap offsets inside the staged window
    int off[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint2 m = j < npx ? __ldg(packed + (size_t)y * dw + x4 + j) : make_uint2(0x80008000u, 0);
        const int sx = (int)(short)(m.x & 0xffffu), sy = (int)(short)(m.x >> 16);
        off[j] = (sy - Y0) * SP + (sx - X0);                 // may be negative / past the window for taps whose valid bit is clear
    }
    const uint8_t* wsrc = s + (size_t)Y0 * spitch + X0;
    const int nitems = nrow * nvec;
    const bool interior = word_store && (t[0].valid & t[1].valid & t[2].valid & t[3].valid) == 15u;
    // RT_STAGES-deep cp.async ring: a thread moves at most RT_SMEM / 16 / RT_THREADS = 1 vector of the window per frame, straight
    // from global to shared memory; the copy of frame f + RT_STAGES - 1 is in flight while frame f is blended, which covers the
    // DRAM latency (a two-buffer version that waited for every frame's window ran at one DRAM round trip per frame: 0.41 ms).
    const int r0 = tid / nvec, v0 = tid - r0 * nvec;
    const bool h0 = tid < nitems;
    const size_t g0 = (size_t)r0 * spitch + (size_t)v0 * 16;
    const uint32_t q0 = (uint32_t)__cvta_generic_to_shared(&win[0][0]) + (uint32_t)(r0 * SP + v0 * 16);
    auto issue = [&](int f) {
        if (h0 && f < nf)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(q0 + (uint32_t)((f % RT_STAGES) * RT_SMEM)), "l"(wsrc + (size_t)f * sframe + g0) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
#pragma unroll
    for (int f = 0; f < RT_STAGES - 1; ++f) issue(f);
    for (int f = 0; f < nf; ++f, d += dframe) {
        asm volatile("cp.async.wait_group %0;" ::"n"(RT_STAGES - 2) : "memory");     // this thread's part of frame f has landed
        __syncthreads();                                      // ... everybody's has, and everybody is done with frame f - 1
        issue(f + RT_STAGES - 1);                             // into the buffer frame f - 1 used
        const uint8_t* W = win[f % RT_STAGES];
        uint32_t v[4];
        if (interior) {                                       // decided once per thread: no per-tap tests inside the frame loop
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint8_t* w = W + off[j];
                v[j] = (uint32_t)(((int)w[0] * t[j].w0 + (int)w[1] * t[j].w1 + (int)w[SP] * t[j].w2 + (int)w[SP + 1] * t[j].w3 + (1 << 14)) >> 15);
            }
            *reinterpret_cast<uint32_t*>(d) = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
            continue;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const RemapTap& q = t[j];
            int p00 = 0, p01 = 0, p10 = 0, p11 = 0;
            if (q.valid & 1u) p00 = W[off[j]];
            if (q.valid & 2u) p01 = W[off[j] + 1];
            if (q.valid & 4u) p10 = W[off[j] + SP];
            if (q.valid & 8u) p11 = W[off[j] + SP + 1];
            v[j] = (uint32_t)((p00 * q.w0 + p01 * q.w1 + p10 * q.w2 + p11 * q.w3 + (1 << 14)) >> 15);
        }
        if (word_store) *reinterpret_cast<uint32_t*>(d) = v[0] | (v[1] << 8) | (v[2] << 16) | (v[3] << 24);
        else for (int j = 0; j < npx; ++j) d[j] = (uint8_t)v[j];
    }
}

// cv::resize(src, dst, newImSize) (INTER_LINEAR, 8UC1) of System::TrackStereo / TrackMonocular (src/System.cc:261-263, 330, 407):
// OpenCV's 11-bit fixed-point bilinear (or the exact-2x INTER_AREA average) from per-column / per-row tables
// {s0 | s1 << 16, c0 | c1 << 16} evaluated once on the host with OpenCV's float formula — the same arithmetic as the pyramid.
__global__ void __launch_bounds__(128) resize_kernel(const uint8_t* __restrict__ src, size_t spitch, size_t sframe,
                                                     const uint2* __restrict__ xtab, const uint2* __restrict__ ytab, int area2x,
                                                     uint8_t* __restrict__ dst, int dw, int dh, size_t dpitch, size_t dframe)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4, y = blockIdx.y;
    if (x4 >= dw) return;
    const uint2 yt = __ldg(ytab + y);
    const uint8_t* S0 = src + (size_t)blockIdx.z * sframe + (size_t)(yt.x & 0xffff) * spitch;
    const uint8_t* S1 = src + (size_t)blockIdx.z * sframe + (size_t)(yt.x >> 16) * spitch;
    const int b0 = (int)(short)(yt.y & 0xffff), b1 = (int)(short)(yt.y >> 16);
    uint8_t* d = dst + (size_t)blockIdx.z * dframe + (size_t)y * dpitch + x4;
    uint32_t out = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        if (x4 + j >= dw) break;
        const uint2 xt = __ldg(xtab + x4 + j);
        const int sx0 = xt.x & 0xffff, sx1 = xt.x >> 16;
        const int a0 = (int)(short)(xt.y & 0xffff), a1 = (int)(short)(xt.y >> 16);
        const int p00 = __ldg(S0 + sx0), p01 = __ldg(S0 + sx1), p10 = __ldg(S1 + sx0), p11 = __ldg(S1 + sx1);
        uint32_t v;
        if (area2x) v = (uint32_t)((p00 + p01 + p10 + p11 + 2) >> 2);
        else {
            const int r0 = p00 * a0 + p01 * a1, r1 = p10 * a0 + p11 * a1;
            v = (uint32_t)((((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2) & 0xffu;
        }
        out |= v << (8 * j);
    }
    if (x4 + 4 <= dw && (reinterpret_cast<size_t>(d) & 3) == 0) *reinterpret_cast<uint32_t*>(d) = out;
    else for (int j = 0; j < 4 && x4 + j < dw; ++j) d[j] = (uint8_t)(out >> (8 * j));
}

// Tiled variant of resize_kernel for batches, same structure as remap_tiled_kernel: the source window of a 128 x 8 destination
// tile is a plain rectangle (rows sy0(first) .. sy1(last), columns sx0(first) .. sx1(last): the tables are monotone), staged
// per frame through a cp.async ring; every tap index in the tables is already clamped into the image, so there is no border case.
__global__ void __launch_bounds__(RT_THREADS, 4) resize_tiled_kernel(const uint8_t* __restrict__ src, size_t spitch, size_t sframe,
                                                                     const uint2* __restrict__ xtab, const uint2* __restrict__ ytab,
                                                                     int area2x, uint8_t* __restrict__ dst, int dw, int dh,
                                                                     size_t dpitch, size_t dframe, int n_frames)
{
    __shared__ __align__(16) uint8_t win[RT_STAGES][RT_SMEM];
    const int tid = threadIdx.x, lane = tid & 31;
    const int tx0 = blockIdx.x * RT_W, ty0 = blockIdx.y * RT_H;
    const int x4 = tx0 + lane * 4, y = ty0 + (tid >> 5);
    const int f0 = blockIdx.z * RT_FPC, nf = min(RT_FPC, n_frames - f0);
    const int npx = y < dh ? max(0, min(4, dw - x4)) : 0;
    const int txl = min(tx0 + RT_W, dw) - 1, tyl = min(ty0 + RT_H, dh) - 1;
    const int X0 = (int)(__ldg(xtab + tx0).x & 0xffff) & ~15, X1 = (int)(__ldg(xtab + txl).x >> 16);
    const int Y0 = (int)(__ldg(ytab + ty0).x & 0xffff), Y1 = (int)(__ldg(ytab + tyl).x >> 16);
    const int nvec = ((X1 - X0) >> 4) + 1, nrow = Y1 - Y0 + 1, SP = nvec * 16, nitems = nvec * nrow;
    const uint2 yt = __ldg(ytab + min(y, dh - 1));
    const int b0 = (int)(short)(yt.y & 0xffff), b1 = (int)(short)(yt.y >> 16);
    const int ro0 = ((int)(yt.x & 0xffff) - Y0) * SP, ro1 = ((int)(yt.x >> 16) - Y0) * SP;
    int c0[4], c1[4], a0[4], a1[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint2 xt = __ldg(xtab + min(x4 + j, dw - 1));
        c0[j] = (int)(xt.x & 0xffff) - X0; c1[j] = (int)(xt.x >> 16) - X0;
        a0[j] = (int)(short)(xt.y & 0xffff); a1[j] = (int)(short)(xt.y >> 16);
    }
    uint8_t* d = dst + (size_t)f0 * dframe + (size_t)y * dpitch + x4;
    const uint8_t* wsrc = src + (size_t)f0 * sframe + (size_t)Y0 * spitch + X0;
    const bool word_store = npx == 4 && ((reinterpret_cast<size_t>(d) | dframe) & 3) == 0;
    const bool staged = SP * nrow <= RT_SMEM && nitems <= RT_THREADS && (size_t)X0 + (size_t)SP <= spitch;
    const int r0 = tid / nvec, v0 = tid - r0 * nvec;
    const bool h0 = staged && tid < nitems;
    const size_t g0 = (size_t)r0 * spitch + (size_t)v0 * 16;
    const uint32_t q0 = (uint32_t)__cvta_generic_to_shared(&win[0][0]) + (uint32_t)(r0 * SP + v0 * 16);
    auto issue = [&](int f) {
        if (h0 && f < nf)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(q0 + (uint32_t)((f % RT_STAGES) * RT_SMEM)), "l"(wsrc + (size_t)f * sframe + g0) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    if (staged) {
#pragma unroll
        for (int f = 0; f < RT_STAGES - 1; ++f) issue(f);
    }
    for (int f = 0; f < nf; ++f, d += dframe) {
        const uint8_t* W;
        int sp;
        if (staged) {
            asm volatile("cp.async.wait_group %0;" ::"n"(RT_STAGES - 2) : "memory");
            __syncthreads();
            issue(f + RT_STAGES - 1);
            W = win[f % RT_STAGES]; sp = SP;
        } else {                                              // window too large for the ring (huge down-scales): read global
            W = wsrc + (size_t)f * sframe; sp = (int)spitch;
        }
        const uint8_t* S0 = W + (staged ? ro0 : (ro0 / SP) * sp);
        const uint8_t* S1 = W + (staged ? ro1 : (ro1 / SP) * sp);
        uint32_t out = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int p00 = S0[c0[j]], p01 = S0[c1[j]], p10 = S1[c0[j]], p11 = S1[c1[j]];
            uint32_t v;
            if (area2x) v = (uint32_t)((p00 + p01 + p10 + p11 + 2) >> 2);
            else {
                const int h0v = p00 * a0[j] + p01 * a1[j], h1v = p10 * a0[j] + p11 * a1[j];
                v = (uint32_t)((((b0 * (h0v >> 4)) >> 16) + ((b1 * (h1v >> 4)) >> 16) + 2) >> 2) & 0xffu;
            }
            out |= v << (8 * j);
        }
        if (word_store) *reinterpret_cast<uint32_t*>(d) = out;
        else for (int j = 0; j < npx; ++j) d[j] = (uint8_t)(out >> (8 * j));
    }
}

cudaError_t launch_undistort(const orbx_keypoint* d_in, int n, const UndistortParams& p, orbx_keypoint* d_out, cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    undistort_kernel<<<(n + 127) / 128, 128, 0, st>>>(d_in, n, p, d_out);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_rgbd_frame(const RgbdArgs& a, int n_frames, cudaStream_t st)
{
    if (n_frames <= 0) return cudaSuccess;
    rgbd_frame_kernel<<<dim3((a.capacity + 127) / 128, n_frames), 128, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_remap_quantise(const float* d_mapx, const float* d_mapy, size_t map_step, int dw, int dh, uint2* d_packed, cudaStream_t st)
{
    remap_quantise_kernel<<<dim3((dw + 255) / 256, dh), 256, 0, st>>>(d_mapx, d_mapy, map_step, dw, dh, d_packed);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_remap(const uint8_t* d_src, int sw, int sh, size_t spitch, size_t sframe, const uint2* d_packed, uint8_t* d_dst, int dw,
                         int dh, size_t dpitch, size_t dframe, int n_frames, cudaStream_t st)
{
    if (n_frames <= 0) return cudaSuccess;
    if ((size_t)sh * spitch >= (size_t)1 << 31) return cudaErrorInvalidValue;       // tap offsets are 32-bit
    if (n_frames >= 8 && ((reinterpret_cast<size_t>(d_src) | spitch | sframe) & 15) == 0) {
        remap_tiled_kernel<<<dim3((dw + RT_W - 1) / RT_W, (dh + RT_H - 1) / RT_H, (n_frames + RT_FPC - 1) / RT_FPC), RT_THREADS, 0, st>>>(
            d_src, sw, sh, spitch, sframe, d_packed, d_dst, dw, dh, dpitch, dframe, n_frames);
        count_launch();
        return cudaGetLastError();
    }
    if (n_frames >= 4)
        remap_kernel<4><<<dim3((dw + 511) / 512, dh, (n_frames + 3) / 4), 128, 0, st>>>(d_src, sw, sh, spitch, sframe, d_packed, d_dst, dw, dh,
                                                                                     dpitch, dframe, n_frames);
    else
        remap_kernel<1><<<dim3((dw + 511) / 512, dh, n_frames), 128, 0, st>>>(d_src, sw, sh, spitch, sframe, d_packed, d_dst, dw, dh, dpitch,
                                                                             dframe, n_frames);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_resize(const uint8_t* d_src, size_t spitch, size_t sframe, const uint2* d_xtab, const uint2* d_ytab, int area2x,
                          uint8_t* d_dst, int dw, int dh, size_t dpitch, size_t dframe, int n_frames, cudaStream_t st)
{
    if (n_frames <= 0) return cudaSuccess;
    if (n_frames >= 8 && ((reinterpret_cast<size_t>(d_src) | spitch | sframe) & 15) == 0) {
        resize_tiled_kernel<<<dim3((dw + RT_W - 1) / RT_W, (dh + RT_H - 1) / RT_H, (n_frames + RT_FPC - 1) / RT_FPC), RT_THREADS, 0, st>>>(
            d_src, spitch, sframe, d_xtab, d_ytab, area2x, d_dst, dw, dh, dpitch, dframe, n_frames);
        count_launch();
        return cudaGetLastError();
    }
    resize_kernel<<<dim3((dw + 511) / 512, dh, n_frames), 128, 0, st>>>(d_src, spitch, sframe, d_xtab, d_ytab, area2x, d_dst, dw, dh, dpitch, dframe);
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
