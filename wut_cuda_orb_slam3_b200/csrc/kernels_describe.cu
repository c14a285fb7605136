// kernels_describe.cu — blur, orientation, rBRIEF descriptors and output packing.
//
//  * blur_kernel:        cv::GaussianBlur(level, 7x7, sigma 2, BORDER_REFLECT_101)   (reference src/ORBextractor.cc:1270-1273)
//                        separable fixed point, kernel [18,34,48,56,48,34,18]/256 per axis, (v + 2^15) >> 16.
//                        Reads the *bordered* pyramid level: its 19-px border already holds the reflect-101 values, so
//                        the 3-px filter halo needs no index arithmetic at all.
//  * orient_describe_kernel: IC_Angle (summation pattern src/OpenCL/Kernel/Angle.cl:24-53, umax src/ORBextractor.cc:455-467,
//                        cv::fastAtan2) on the un-blurred level + computeOrbDescriptor (src/ORBextractor.cc:105-149) on the
//                        blurred level; one warp per keypoint, lane = descriptor byte.
//  * pack_kernel:        operator() output packing (src/ORBextractor.cc:1283-1306): scale, lapping-area split.
#include <float.h>

#include <algorithm>
#include <mutex>

#include "orbx_internal.cuh"

namespace orbx {

namespace {

__constant__ int c_umax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};

// Filled once per device by launch_orient_describe():
//   d_pattern_f[k][lane] = (x0, y0, x1, y1) of test 8*lane + k as floats (coalesced 16-byte loads, no int->float conversions)
//   d_mom_mask[|v|][j]   = byte mask of the patch-row words j = 0..7 (columns u = -15 + 4j .. -12 + 4j): 0xff where |u| <= umax[|v|]
__device__ float4 d_pattern_f[8][32];
__device__ uint4 d_mom_mask[16][2];

constexpr int BT_W = 128, BT_H = 32;          // blur tile
constexpr int BIN_P = kBlurBoxW;              // input tile pitch (bytes): image columns x0-16 .. x0+159 (16-byte aligned)
constexpr int BIN_R = BT_H + 6;

// cv::fastAtan2 (OpenCV mathfuncs_core atan_f32): float32, no FMA contraction.
__device__ __forceinline__ float fast_atan2_dev(float y, float x)
{
    const float scale = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale;
    const float p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
    const float ax = fabsf(x), ay = fabsf(y);
    float a, c, c2;
    if (ax >= ay) {
        c = __fdiv_rn(ay, __fadd_rn(ax, (float)DBL_EPSILON));
        c2 = __fmul_rn(c, c);
        a = __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c);
    } else {
        c = __fdiv_rn(ax, __fadd_rn(ay, (float)DBL_EPSILON));
        c2 = __fmul_rn(c, c);
        a = __fsub_rn(90.f, __fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fadd_rn(__fmul_rn(p7, c2), p5), c2), p3), c2), p1), c));
    }
    if (x < 0) a = __fsub_rn(180.f, a);
    if (y < 0) a = __fsub_rn(360.f, a);
    return a;
}

}  // namespace

// grid = (tiles over all levels, n_frames).  Separable fixed-point 7x7: the horizontal pass is two IDP.4A (dp4a) per
// pixel on byte windows realigned with funnel shifts (kernel bytes 18,34,48,56 | 48,34,18,0), the vertical pass a
// sliding 32-bit window using the kernel's symmetry; the tile leaves through shared memory as 16-byte stores.
__global__ void __launch_bounds__(256) blur_kernel(const __grid_constant__ FrameGeom fg, Workspace ws)
{
    __shared__ __align__(128) uint8_t in[kBlurBoxH * BIN_P];
    __shared__ __align__(16) uint32_t hb[BIN_R * BT_W];
    __shared__ __align__(16) uint8_t outt[BT_H * BT_W];
    const int tid = threadIdx.x;
    const int frame = blockIdx.y;
    // locate (level, tile)
    int t = blockIdx.x, level = 0, tx_n = 0;
#pragma unroll 1
    for (int l = 0; l < fg.nlevels; ++l) {
        tx_n = (fg.L[l].w + BT_W - 1) / BT_W;
        const int nt = tx_n * ((fg.L[l].h + BT_H - 1) / BT_H);
        if (t < nt) { level = l; break; }
        t -= nt;
    }
    const LevelGeom& g = fg.L[level];
    const int tyi = t / tx_n;
    const int ty0 = tyi * BT_H, tx0 = (t - tyi * tx_n) * BT_W;
    const uint8_t* base = ws.pyr + g.pyr_off + (size_t)frame * g.pyr_frame_stride;   // bordered buffer origin
    // input tile: buffer rows (ty0 - 3 + 19) .., buffer byte columns (tx0 - 16 + 32) .. : 16-byte aligned
    const int brow0 = ty0 - 3 + kEdge, bcol0 = tx0 - 16 + kXPad;
    if (ws.tmap_blur) {
        // TMA: kBlurBoxW x kBlurBoxH box of the bordered level (out-of-range rows/columns are zero-filled by the copy engine);
        // its last two rows are not used here
        __shared__ __align__(8) uint64_t bar;
        if (tid == 0) mbar_init(&bar, 1);
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&bar, kBlurBoxH * BIN_P);
            tma_load_3d(in, ws.tmap_blur + level, &bar, bcol0, brow0, frame);
        }
        mbar_wait(&bar, 0);
    } else {
        for (int i = tid; i < BIN_R * (BIN_P / 16); i += 256) {
            const int r = i / (BIN_P / 16), v = i - r * (BIN_P / 16);
            const int br = brow0 + r, bc = bcol0 + 16 * v;
            uint4 q = make_uint4(0, 0, 0, 0);
            if (br < g.rows_alloc && bc + 16 <= g.pitch) q = __ldg(reinterpret_cast<const uint4*>(base + (size_t)br * g.pitch + bc));
            reinterpret_cast<uint4*>(in)[i] = q;
        }
        __syncthreads();
    }
    // horizontal pass: task = (row, group of 4 columns); output x = 4q + j reads tile columns 4q+13+j .. 4q+19+j
    for (int i = tid; i < BIN_R * (BT_W / 4); i += 256) {
        const int r = i >> 5, q = i & 31;
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(in + r * BIN_P) + q + 3;
        const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2];
        const uint32_t KA = 0x38302212u, KB = 0x00122230u;
        uint4 h;
        h.x = __dp4a(__funnelshift_r(w0, w1, 8), KA, __dp4a(__funnelshift_r(w1, w2, 8), KB, 0u));
        h.y = __dp4a(__funnelshift_r(w0, w1, 16), KA, __dp4a(__funnelshift_r(w1, w2, 16), KB, 0u));
        h.z = __dp4a(__funnelshift_r(w0, w1, 24), KA, __dp4a(__funnelshift_r(w1, w2, 24), KB, 0u));
        h.w = __dp4a(w1, KA, __dp4a(w2, KB, 0u));
        *reinterpret_cast<uint4*>(hb + r * BT_W + 4 * q) = h;
    }
    __syncthreads();
    // vertical pass: thread = 2 adjacent columns x 8 rows, sliding window
    {
        const int cp = (tid & 63) * 2, r0 = (tid >> 6) * 8;
        uint2 w[14];
#pragma unroll
        for (int k = 0; k < 14; ++k) w[k] = *reinterpret_cast<const uint2*>(hb + (r0 + k) * BT_W + cp);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const uint32_t s0 = 18u * (w[i].x + w[i + 6].x) + 34u * (w[i + 1].x + w[i + 5].x) + 48u * (w[i + 2].x + w[i + 4].x) + 56u * w[i + 3].x;
            const uint32_t s1 = 18u * (w[i].y + w[i + 6].y) + 34u * (w[i + 1].y + w[i + 5].y) + 48u * (w[i + 2].y + w[i + 4].y) + 56u * w[i + 3].y;
            const uint32_t o = ((s0 + 32768u) >> 16) | (((s1 + 32768u) >> 16) << 8);
            *reinterpret_cast<uint16_t*>(outt + (r0 + i) * BT_W + cp) = (uint16_t)o;
        }
    }
    __syncthreads();
    // 16-byte stores (the blurred level's pitch is a multiple of 16, so the last vector of a row may spill into padding)
    {
        const int r = tid >> 3, v = tid & 7;
        const int y = ty0 + r, x = tx0 + 16 * v;
        if (y < g.h && x < g.w) {
            uint8_t* out = ws.blur + g.blur_off + (size_t)frame * g.blur_frame_stride + (size_t)y * g.bpitch + x;
            *reinterpret_cast<uint4*>(out) = *reinterpret_cast<const uint4*>(outt + r * BT_W + 16 * v);
        }
    }
}

// Register-streaming blur (default): one WARP per 128-column x 64-row band.  A lane owns 4 adjacent columns; for every input row
// it reads the three aligned words around them (L1 hits: neighbouring lanes read the same words), forms the horizontal 7-tap
// sums of its 4 pixels with 8 dp4a on funnel-shifted byte windows, and keeps the last 7 rows of sums in registers (the row loop
// is unrolled by 7 so the window rotates without moves); every new row completes one output row: symmetric vertical taps
// (3 adds + 4 multiply-adds), (v + 2^15) >> 16, four bytes packed into one coalesced 32-bit store.  No shared memory, no
// barriers, ~14 instructions per pixel instead of ~34 for the tiled kernel above (whose per-tile set-up and two shared-memory
// round trips dominate).  grid = (ceil(items / 4), n_frames), 4 warps per CTA.
constexpr int BS_ROWS = 64;

__device__ __forceinline__ void blur_load3(const uint8_t* __restrict__ rowp, uint32_t w[3])
{
    const uint32_t* wp = reinterpret_cast<const uint32_t*>(rowp);
    w[0] = __ldg(wp - 1); w[1] = __ldg(wp); w[2] = __ldg(wp + 1);
}
__device__ __forceinline__ void blur_hsum(const uint32_t w[3], uint32_t h[4])
{
    const uint32_t KA = 0x38302212u, KB = 0x00122230u;             // taps (18,34,48,56 | 48,34,18,0)
    // pixel j reads bytes j-3 .. j+3 relative to w[1]'s byte 0, i.e. the 8-byte window starting at byte (j + 1) of (w0, w1, w2)
    h[0] = __dp4a(__funnelshift_r(w[0], w[1], 8), KA, __dp4a(__funnelshift_r(w[1], w[2], 8), KB, 0u));
    h[1] = __dp4a(__funnelshift_r(w[0], w[1], 16), KA, __dp4a(__funnelshift_r(w[1], w[2], 16), KB, 0u));
    h[2] = __dp4a(__funnelshift_r(w[0], w[1], 24), KA, __dp4a(__funnelshift_r(w[1], w[2], 24), KB, 0u));
    h[3] = __dp4a(w[1], KA, __dp4a(w[2], KB, 0u));
}

__global__ void __launch_bounds__(128) blur_stream_kernel(const __grid_constant__ FrameGeom fg, Workspace ws)
{
    const int lane = threadIdx.x & 31;
    const int frame = blockIdx.y;
    int t = blockIdx.x * 4 + (threadIdx.x >> 5), level = -1, sx_n = 0;
#pragma unroll 1
    for (int l = 0; l < fg.nlevels; ++l) {
        sx_n = (fg.L[l].w + 127) / 128;
        const int nt = sx_n * ((fg.L[l].h + BS_ROWS - 1) / BS_ROWS);
        if (t < nt) { level = l; break; }
        t -= nt;
    }
    if (level < 0) return;
    const LevelGeom& g = fg.L[level];
    const int band = t / sx_n;
    const int x = (t - band * sx_n) * 128 + 4 * lane, y0 = band * BS_ROWS;
    if (x >= g.w) return;                                   // lanes right of the image neither load nor store
    const int rows = min(BS_ROWS, g.h - y0);
    const size_t pitch = g.pitch;
    // input row i (i = 0 .. rows + 5) is image row y0 - 3 + i of the bordered level (its 19-px border holds the reflect-101 halo)
    const uint8_t* in = ws.pyr + g.pyr_off + (size_t)frame * g.pyr_frame_stride + (size_t)(kEdge + y0 - 3) * pitch + kXPad + x;
    uint8_t* out = ws.blur + g.blur_off + (size_t)frame * g.blur_frame_stride + (size_t)y0 * g.bpitch + x;
    uint32_t W[7][4];
    {
        uint32_t w6[6][3];
#pragma unroll
        for (int i = 0; i < 6; ++i) blur_load3(in + (size_t)i * pitch, w6[i]);       // six independent row loads in flight
#pragma unroll
        for (int i = 0; i < 6; ++i) blur_hsum(w6[i], W[i]);
    }
    in += 6 * pitch;
    // two rows of loads stay in flight ahead of the arithmetic (rows past the band are clamped to its last input row)
    const uint8_t* in_last = in + (size_t)(rows - 1) * pitch;
    uint32_t na[3], nb[3];
    blur_load3(in, na);
    blur_load3(rows > 1 ? in + pitch : in_last, nb);
    in += 2 * pitch;
    for (int r = 0; r < rows; r += 7) {
#pragma unroll
        for (int k = 0; k < 7; ++k) {
            if (r + k < rows) {                             // warp-uniform
                blur_hsum(na, W[(k + 6) % 7]);              // input row (r + k) + 6 completes output row r + k
                na[0] = nb[0]; na[1] = nb[1]; na[2] = nb[2];
                blur_load3(in <= in_last ? in : in_last, nb);
                in += pitch;
                uint32_t o = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint32_t s = 18u * (W[k % 7][j] + W[(k + 6) % 7][j]) + 34u * (W[(k + 1) % 7][j] + W[(k + 5) % 7][j]) +
                                       48u * (W[(k + 2) % 7][j] + W[(k + 4) % 7][j]) + 56u * W[(k + 3) % 7][j];
                    o |= ((s + 32768u) >> 16) << (8 * j);
                }
                *reinterpret_cast<uint32_t*>(out) = o;      // bpitch is a multiple of 16: the last word of a row may spill into padding
                out += g.bpitch;
            }
        }
    }
}

// Tensor-core blur (default for batches when tensor maps are available).  The filter is an integer linear map, exact in int32
// up to the single final rounding, so int8 MMAs (imma_16832_u8) produce the same bytes as the scalar kernels in any summation
// order.  Every warp is persistent and owns one stage of one kBlurBoxW x kBlurBoxH TMA box (completion on an mbarrier); an item is a
// 128-column x 32-row band, worked as 8 column tiles of 16 outputs (g = lane / 4, t = lane % 4):
//  * Horizontal pass, transposed: H^T (16 columns x 8 rows) = Wh (16 x 32) . I^T (32 input columns x 8 rows).  The K window of a
//    tile starts one word left of it (input column c0 - 4), so Wh[m][k] = w[k - m - 1] is constant and a B register is 4
//    consecutive bytes of one staged row: one conflict-free 32-bit shared load.  Five such MMAs cover the 40 rows of the box.
//  * Vertical pass: S (16 rows x 8 columns) = Wv (16 x 32) . H (32 H rows x 8 columns).  The horizontal accumulators leave a
//    thread the H values of columns g and g + 8 in rows 2 t, 2 t + 1 of every 8-row block.  With K permuted (slot 16 u + 4 t + i
//    <-> H row 16 u + 8 (i / 2) + 2 t + i % 2) these are exactly its B slots, so Wv carries the permutation and no data moves
//    between lanes.  Row tile T uses the blocks 2T .. 2T+2; the fourth block of its K window has zero weight.
//  * H < 2^16 is split into bytes with PRMT: S = 256 acc_hi + acc_lo, acc_lo seeded with the rounding constant 2^15, and the output
//    byte is byte 2 of S (S < 2^24).  Per 16 x 16 outputs: 2.5 horizontal and 4 vertical MMAs.
//  * Two shuffles over the lane quad give each lane 8 consecutive output bytes of one row; they go to the columns of the stage the
//    tile has consumed (16 j .. 16 j + 15), and the finished band leaves as 16-byte stores, 128 contiguous bytes per row.
constexpr int kBmWarps = 4;
constexpr int kBmStageBytes = kBlurBoxW * kBlurBoxH;          // 7040, a multiple of 128 (TMA destination alignment)

__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

__global__ void __launch_bounds__(32 * kBmWarps) blur_mma_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int items_per_frame,
                                                                 int total_items)
{
    extern __shared__ __align__(128) uint8_t bm_smem[];
    __shared__ __align__(8) uint64_t bars[kBmWarps];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, t = lane & 3;
    uint8_t* stage = bm_smem + (size_t)warp * kBmStageBytes;
    uint64_t* bar = &bars[warp];
    if (lane == 0) mbar_init(bar, 1);
    __syncwarp();
    const int gw = blockIdx.x * kBmWarps + warp, nw = gridDim.x * kBmWarps;

    // constant A fragments: taps w[0..6] = bytes of kTaps (byte 7 = 0)
    uint32_t ah[4], av[4];
    {
        constexpr unsigned long long kTaps = 0x0012223038302212ull;
        auto tap = [](int d) -> uint32_t { return d >= 0 && d < 8 ? (uint32_t)(kTaps >> (8 * d)) & 0xffu : 0u; };
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int m = g + 8 * (q & 1);
            ah[q] = av[q] = 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                ah[q] |= tap(16 * (q >> 1) + 4 * t + i - m - 1) << (8 * i);
                av[q] |= tap(16 * (q >> 1) + 8 * (i >> 1) + 2 * t + (i & 1) - m) << (8 * i);
            }
        }
    }
    // the quad transpose of the output: round 1 (lanes t, t ^ 1) exchanges rows, round 2 (t, t ^ 2) exchanges column halves
    const int a = t & 1, hb = t >> 1;
    const uint32_t sel0 = a ? 0x1054u : 0x5410u, sel1 = a ? 0x3276u : 0x7632u;

    // item -> (frame, level, x0, y0)
    auto decode = [&](int item, int& frame, int& level, int& x0, int& y0) {
        frame = item / items_per_frame;
        int r = item - frame * items_per_frame;
        level = 0;
        int sx_n = 1;
#pragma unroll 1
        for (int l = 0; l < fg.nlevels; ++l) {
            sx_n = (fg.L[l].w + 127) / 128;
            const int nt = sx_n * ((fg.L[l].h + 31) / 32);
            level = l;
            if (r < nt) break;
            r -= nt;
        }
        const int band = r / sx_n;
        x0 = (r - band * sx_n) * 128;
        y0 = band * 32;
    };
    auto issue = [&](int item) {          // lane 0 only
        int frame, level, x0, y0;
        decode(item, frame, level, x0, y0);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        mbar_expect_tx(bar, kBmStageBytes);
        tma_load_3d(stage, ws.tmap_blur + level, bar, kXPad + x0 - 16, kEdge + y0 - 3, frame);
    };

    if (lane == 0 && gw < total_items) issue(gw);
    int k = 0;
    for (int item = gw; item < total_items; item += nw, ++k) {
        int frame, level, x0, y0;
        decode(item, frame, level, x0, y0);
        const LevelGeom& lg = fg.L[level];
        mbar_wait(bar, (uint32_t)(k & 1));
        const int ntiles = min(8, (lg.w - x0 + 15) >> 4);
#pragma unroll 1
        for (int j = 0; j < ntiles; ++j) {
            // horizontal pass: per 8-row block b and column half h, q = (H lo, H lo, H hi, H hi) of rows 2 t, 2 t + 1
            uint32_t hq[5][2];
            const uint8_t* bp = stage + g * kBlurBoxW + 16 * j + 12 + 4 * t;
#pragma unroll
            for (int b = 0; b < 5; ++b) {
                const uint32_t b0 = *reinterpret_cast<const uint32_t*>(bp + 8 * b * kBlurBoxW);
                const uint32_t b1 = *reinterpret_cast<const uint32_t*>(bp + 8 * b * kBlurBoxW + 16);
                int c[4] = {0, 0, 0, 0};
                imma_16832_u8(c, ah, b0, b1);
                hq[b][0] = prmt(c[0], c[1], 0x5140u);
                hq[b][1] = prmt(c[2], c[3], 0x5140u);
            }
#pragma unroll
            for (int T = 0; T < 2; ++T) {
                // vertical pass: s[h][c] = S + 2^15 of row g + 8 (c >> 1), column 8 h + 2 t + (c & 1)
                int s[2][4];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const uint32_t qa = hq[2 * T][h], qb = hq[2 * T + 1][h], qc = hq[2 * T + 2][h];
                    int lo[4] = {32768, 32768, 32768, 32768}, hi[4] = {0, 0, 0, 0};
                    imma_16832_u8(lo, av, prmt(qa, qb, 0x5410u), qc);          // qc's upper half sits in zero-weight slots
                    imma_16832_u8(hi, av, prmt(qa, qb, 0x7632u), qc >> 16);
#pragma unroll
                    for (int c = 0; c < 4; ++c) s[h][c] = lo[c] + (hi[c] << 8);
                }
                // w[r] = output bytes of row g + 8 r, columns 8 h + 2 t + {0, 1} for h = 0, 1
                uint32_t w[2];
#pragma unroll
                for (int r = 0; r < 2; ++r)
                    w[r] = prmt(prmt(s[0][2 * r], s[0][2 * r + 1], 0x62u), prmt(s[1][2 * r], s[1][2 * r + 1], 0x62u), 0x5410u);
                const uint32_t rx = __shfl_xor_sync(0xffffffffu, a ? w[0] : w[1], 1);
                const uint32_t keep = a ? w[1] : w[0];
                // row g + 8 a, columns 8 h + 4 hb .. + 3
                const uint32_t kh0 = prmt(keep, rx, sel0), kh1 = prmt(keep, rx, sel1);
                const uint32_t ry = __shfl_xor_sync(0xffffffffu, hb ? kh0 : kh1, 2);
                const uint32_t kk = hb ? kh1 : kh0;
                *reinterpret_cast<uint2*>(stage + (16 * T + g + 8 * a) * kBlurBoxW + 16 * j + 8 * hb) = hb ? make_uint2(ry, kk) : make_uint2(kk, ry);
            }
        }
        __syncwarp();
        {
            // the band leaves: lane = (row quarter, 16-byte column); the blurred level's pitch is a multiple of 16, so the last
            // vector of a row may spill into padding
            const int rows = min(32, lg.h - y0);
            const int cx = 16 * (lane & 7);
            uint8_t* out = ws.blur + lg.blur_off + (size_t)frame * lg.blur_frame_stride + (size_t)y0 * lg.bpitch + x0 + cx;
            if (x0 + cx < lg.w) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int r = 4 * i + (lane >> 3);
                    if (r < rows) *reinterpret_cast<uint4*>(out + (size_t)r * lg.bpitch) = *reinterpret_cast<const uint4*>(stage + r * kBlurBoxW + cx);
                }
            }
        }
        __syncwarp();                                               // every lane is done reading the stage
        if (lane == 0 && item + nw < total_items) issue(item + nw);
    }
}

// The packing of operator() (src/ORBextractor.cc:1283-1306) fused into the descriptor kernel for the two cases in which a
// keypoint's output row follows from its level-major index t alone: no keypoint lies in the lapping area (vLappingArea =
// {0, 0}: stereo / RGB-D, src/Frame.cc:124-125, 224) -> row t; every keypoint does ({0, 1000} on images up to 1000 px wide:
// monocular, src/Frame.cc:313) -> row nkp - 1 - t.  Anything else (a fisheye lapping area) takes pack_kernel.
struct FusedPack {
    int mode;                 // 0 = separate pack kernel, 1 = nothing lapping, 2 = everything lapping
    ChunkIO io;
};

// grid = (ceil(kp_slots / 8), n_frames), 8 warps per CTA, one warp per keypoint slot.
constexpr int kOdStage = kDescBoxW * kDescBoxH;   // bytes per warp
#ifndef ORBX_OD_MINB
#define ORBX_OD_MINB 5          // 47 registers, no spills; 6 and 8 CTAs per SM (40 / 32 registers, spills) measure the same, 1 (61 registers) 6 % slower
#endif

template <bool STAGED>
__global__ void __launch_bounds__(256, STAGED ? ORBX_OD_MINB : 1) orient_describe_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, FusedPack fp)
{
    extern __shared__ __align__(128) uint8_t od_smem[];      // [8 warps][64 x 40] when the blurred levels have tensor maps
    __shared__ __align__(8) uint64_t od_bar[8];
    const int lane = threadIdx.x & 31;
    const int slot = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int frame = blockIdx.y;
    if (slot >= fg.kp_slots) return;
    static_assert((kMaxLevels & (kMaxLevels - 1)) == 0, "binary search over a power of two");
    int level = 0;                                   // the level whose slot range holds `slot`: kp_base ascends, unused levels hold INT_MAX
#pragma unroll
    for (int step = kMaxLevels / 2; step >= 1; step >>= 1)
        if (slot >= fg.L[level + step].kp_base) level += step;
    const LevelGeom& g = fg.L[level];
    const int i = slot - g.kp_base;
    int n_level, t_out = 0, nkp = 0;
    if (fp.mode) {
        // per-level counts -> this level's offset and the frame total (one load per lane + a shuffle scan)
        const int c = lane < fg.nlevels ? ws.lvl_n[(size_t)frame * fg.nlevels + lane] : 0;
        int incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        n_level = __shfl_sync(0xffffffffu, c, level);
        t_out = __shfl_sync(0xffffffffu, incl - c, level) + i;
        nkp = __shfl_sync(0xffffffffu, incl, 31);
        if (slot == 0 && lane == 0) {                       // the frame's counters (src 1306: the return value is monoIndex)
            *fp.io.n_out(frame) = nkp;
            *fp.io.n_mono(frame) = nkp > fp.io.capacity ? -1 : (fp.mode == 1 ? nkp : 0);
        }
    } else {
        n_level = ws.lvl_n[(size_t)frame * fg.nlevels + level];
    }
    if (i >= n_level) return;
    const uint32_t key = ws.lvl_kp[(size_t)frame * fg.kp_slots + slot];
    const int x = (int)(key & 0xfff) + kWinBorder, y = (int)((key >> 12) & 0xfff) + kWinBorder;

    // The rBRIEF tests gather 512 bytes of the blurred level from a 39 x 39 window in an order set by the rotated pattern: as global
    // loads every warp instruction touches ~20 different lines.  With a tensor map the window is staged by ONE bulk copy issued
    // here, before the orientation is computed (the copy overlaps IC_Angle), and the gathers become shared-memory byte loads.
    constexpr bool staged = STAGED;
    const int warp = threadIdx.x >> 5;
    const int x0 = (x - 19) & ~15;                            // 16-byte aligned box start; x >= 19
    const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(od_smem) + (uint32_t)warp * kOdStage;
    if (staged) {
        if (lane == 0) {
            mbar_init(&od_bar[warp], 1);
            mbar_expect_tx(&od_bar[warp], kDescBoxW * kDescBoxH);
            tma_load_3d(od_smem + warp * kOdStage, ws.tmap_desc + level, &od_bar[warp], x0, y - 20, frame);
        }
        __syncwarp();
    }

    // ---- IC_Angle on the un-blurred level: lane <-> patch row v = lane - 15 ----
    // The row's 31 bytes arrive as 9 aligned 32-bit words, realigned with funnel shifts (the misalignment is the same for
    // every row: the pitch is a multiple of 16), masked to the disc |u| <= umax[|v|] and summed with dp4a:
    //   m10 = sum_u u * I(u, v) = dp4a(bytes, (u0, u0+1, u0+2, u0+3)),   m01 = v * sum_u I(u, v) = v * dp4a(bytes, (1,1,1,1)).
    int m10 = 0, m01 = 0;
    {
        const int v = lane - kHalfPatch;
        if (lane < 31) {
            // three 16-byte loads per row instead of nine 4-byte ones: a warp instruction touches 31 different lines either way,
            // and the L1 data pipe is this kernel's limiter (one wavefront per line per instruction)
            const uint8_t* rowp = level_interior((const uint8_t*)ws.pyr, g, frame) + (ptrdiff_t)(y + v) * g.pitch + (x - kHalfPatch);
            const int mis16 = (int)((uintptr_t)rowp & 15);                  // the same for every row: the pitch is a multiple of 16
            const int mis = mis16 & 3;
            const uint4* rq = reinterpret_cast<const uint4*>(rowp - mis16);
            const uint4 q0 = __ldg(rq), q1 = __ldg(rq + 1), q2 = __ldg(rq + 2);
            uint32_t w[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
            if (mis16 & 4) {                                                // warp-uniform: drop the leading words
#pragma unroll
                for (int j = 0; j < 11; ++j) w[j] = w[j + 1];
            }
            if (mis16 & 8) {
#pragma unroll
                for (int j = 0; j < 10; ++j) w[j] = w[j + 2];
            }
            const int av = v < 0 ? -v : v;
            const uint4 ma = d_mom_mask[av][0], mb = d_mom_mask[av][1];
            const uint32_t mk[8] = {ma.x, ma.y, ma.z, ma.w, mb.x, mb.y, mb.z, mb.w};
            const int sh = 8 * mis;
            int sum = 0;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const uint32_t px = __funnelshift_r(w[j], w[j + 1], sh) & mk[j];
                const int u0 = -kHalfPatch + 4 * j;
                const uint32_t wt = (uint32_t)(u0 & 0xff) | ((uint32_t)((u0 + 1) & 0xff) << 8) | ((uint32_t)((u0 + 2) & 0xff) << 16) |
                                    ((uint32_t)((u0 + 3) & 0xff) << 24);
                asm("dp4a.u32.s32 %0, %1, %2, %0;" : "+r"(m10) : "r"(px), "r"(wt));
                sum = (int)__dp4a(px, 0x01010101u, (uint32_t)sum);
            }
            m01 = v * sum;
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) {
            m10 += __shfl_xor_sync(0xffffffffu, m10, d);
            m01 += __shfl_xor_sync(0xffffffffu, m01, d);
        }
    }
    const float angle = fast_atan2_dev((float)m01, (float)m10);

    // ---- rBRIEF on the blurred level: lane <-> descriptor byte ----
    const float factorPI = (float)(3.14159265358979323846 / 180.f);
    const float arad = __fmul_rn(angle, factorPI);
    double sd, cd;
    sincos((double)arad, &sd, &cd);                 // same values as sin()/cos(), one argument reduction
    const float a = (float)cd, b = (float)sd;
    const uint8_t* center = ws.blur + g.blur_off + (size_t)frame * g.blur_frame_stride + (size_t)y * g.bpitch + x;
    const int step = g.bpitch;
    // cvRound (round half to even) without the conversion unit: adding 1.5 * 2^23 leaves the rounded integer in the low
    // mantissa bits (|value| <= 19 here), so int = bits - 0x4B400000
    const float kMagic = 12582912.0f;
    const int kMagicBits = 0x4B400000;
    uint32_t val = 0;
    if (staged) {
        mbar_wait(&od_bar[warp], 0);
        const uint32_t cb = stage_s + 20 * kDescBoxW + (uint32_t)(x - x0);      // the keypoint's byte in the staged window
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float4 q = d_pattern_f[k][lane];
            const int iy0 = __float_as_int(__fadd_rn(__fadd_rn(__fmul_rn(q.x, b), __fmul_rn(q.y, a)), kMagic)) - kMagicBits;
            const int ix0 = __float_as_int(__fadd_rn(__fsub_rn(__fmul_rn(q.x, a), __fmul_rn(q.y, b)), kMagic)) - kMagicBits;
            const int iy1 = __float_as_int(__fadd_rn(__fadd_rn(__fmul_rn(q.z, b), __fmul_rn(q.w, a)), kMagic)) - kMagicBits;
            const int ix1 = __float_as_int(__fadd_rn(__fsub_rn(__fmul_rn(q.z, a), __fmul_rn(q.w, b)), kMagic)) - kMagicBits;
            uint32_t t0, t1;
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t0) : "r"(cb + (uint32_t)(iy0 * kDescBoxW + ix0)));
            asm volatile("ld.shared.u8 %0, [%1];" : "=r"(t1) : "r"(cb + (uint32_t)(iy1 * kDescBoxW + ix1)));
            val |= (uint32_t)(t0 < t1) << k;
        }
    } else
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float4 q = d_pattern_f[k][lane];          // (x0, y0, x1, y1) of test 8 * lane + k
        const int iy0 = __float_as_int(__fadd_rn(__fadd_rn(__fmul_rn(q.x, b), __fmul_rn(q.y, a)), kMagic)) - kMagicBits;
        const int ix0 = __float_as_int(__fadd_rn(__fsub_rn(__fmul_rn(q.x, a), __fmul_rn(q.y, b)), kMagic)) - kMagicBits;
        const int iy1 = __float_as_int(__fadd_rn(__fadd_rn(__fmul_rn(q.z, b), __fmul_rn(q.w, a)), kMagic)) - kMagicBits;
        const int ix1 = __float_as_int(__fadd_rn(__fsub_rn(__fmul_rn(q.z, a), __fmul_rn(q.w, b)), kMagic)) - kMagicBits;
        const int t0 = __ldg(center + iy0 * step + ix0), t1 = __ldg(center + iy1 * step + ix1);
        val |= (uint32_t)(t0 < t1) << k;
    }
    ws.lvl_desc[((size_t)frame * fg.kp_slots + slot) * 32 + lane] = (uint8_t)val;
    if (lane == 0) ws.lvl_angle[(size_t)frame * fg.kp_slots + slot] = angle;
    if (fp.mode && nkp <= fp.io.capacity) {
        const int dst = fp.mode == 1 ? t_out : nkp - 1 - t_out;
        fp.io.desc(frame)[(size_t)dst * 32 + lane] = (uint8_t)val;
        if (lane < 7) {                                     // the 28-byte keypoint, one 32-bit field per lane
            float px = (float)x, py = (float)y;
            if (level != 0) { px = __fmul_rn(px, g.scale); py = __fmul_rn(py, g.scale); }       // src 1289-1291
            uint32_t w;
            switch (lane) {
                case 0: w = __float_as_uint(px); break;
                case 1: w = __float_as_uint(py); break;
                case 2: w = __float_as_uint(g.kp_size); break;
                case 3: w = __float_as_uint(angle); break;
                case 4: w = __float_as_uint((float)(key >> 24)); break;
                case 5: w = (uint32_t)level; break;
                default: w = 0xffffffffu; break;            // class_id = -1
            }
            reinterpret_cast<uint32_t*>(fp.io.kps(frame) + dst)[lane] = w;
        }
    }
}

// grid = n_frames, T threads: src/ORBextractor.cc:1283-1306.  T = 256 for batches (one CTA per frame, hundreds of frames in
// flight), 1024 for a few frames: the whole frame is then one pass with two barriers — the kernel sits on the critical path
// of the single-frame call.
template <int T>
__global__ void __launch_bounds__(T) pack_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int lap0, int lap1, const ChunkIO io)
{
    __shared__ int lvl_off[kMaxLevels + 1];
    __shared__ int warp_cnt[T / 32];
    __shared__ int carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.x;
    if (warp == 0) {                               // per-level counts -> offsets: independent loads + a shuffle scan
        static_assert(kMaxLevels <= 32, "one lane per level");
        const int c = lane < fg.nlevels ? ws.lvl_n[(size_t)frame * fg.nlevels + lane] : 0;
        int incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane < fg.nlevels) lvl_off[lane] = incl - c;
        if (lane == fg.nlevels - 1) lvl_off[fg.nlevels] = incl;
        if (lane == 0) carry = 0;
    }
    __syncthreads();
    const int nkp = lvl_off[fg.nlevels];
    const int capacity = io.capacity;
    int* n_out = io.n_out(frame);
    int* n_mono = io.n_mono(frame);
    if (nkp > capacity) {
        if (tid == 0) { *n_out = nkp; *n_mono = -1; }
        return;
    }
    orbx_keypoint* okp = io.kps(frame);
    uint8_t* odesc = io.desc(frame);
    const float flap0 = (float)lap0, flap1 = (float)lap1;
    for (int base = 0; base < nkp; base += T) {
        const int t = base + tid;
        bool valid = t < nkp, stereo = false;
        orbx_keypoint kp;
        int slot = 0;
        if (valid) {
            int level = 0;
            for (int l = 1; l < fg.nlevels; ++l)
                if (t >= lvl_off[l]) level = l;
            const LevelGeom& g = fg.L[level];
            slot = g.kp_base + (t - lvl_off[level]);
            const uint32_t key = ws.lvl_kp[(size_t)frame * fg.kp_slots + slot];
            float px = (float)((int)(key & 0xfff) + kWinBorder), py = (float)((int)((key >> 12) & 0xfff) + kWinBorder);
            if (level != 0) { px = __fmul_rn(px, g.scale); py = __fmul_rn(py, g.scale); }
            kp.x = px; kp.y = py; kp.size = g.kp_size;
            kp.angle = ws.lvl_angle[(size_t)frame * fg.kp_slots + slot];
            kp.response = (float)(key >> 24);
            kp.octave = level; kp.class_id = -1;
            stereo = px >= flap0 && px <= flap1;
        }
        const uint32_t mS = __ballot_sync(0xffffffffu, valid && stereo);
        if (lane == 0) warp_cnt[warp] = __popc(mS);
        __syncthreads();
        int before = carry;            // lapping-area keypoints before this chunk
        for (int w = 0; w < warp; ++w) before += warp_cnt[w];
        const int sBefore = before + __popc(mS & ((1u << lane) - 1));
        if (valid) {
            const int dst = stereo ? (nkp - 1 - sBefore) : (t - sBefore);
            okp[dst] = kp;
            const uint4* s = reinterpret_cast<const uint4*>(ws.lvl_desc + ((size_t)frame * fg.kp_slots + slot) * 32);
            uint4* d = reinterpret_cast<uint4*>(odesc + (size_t)dst * 32);
            d[0] = s[0]; d[1] = s[1];
        }
        __syncthreads();
        if (tid == 0) { int c = carry; for (int w = 0; w < T / 32; ++w) c += warp_cnt[w]; carry = c; }
        __syncthreads();
    }
    if (tid == 0) { *n_out = nkp; *n_mono = nkp - carry; }
}

cudaError_t launch_blur(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st)
{
    // the tensor-core kernel for batches, the tiled kernel (more parallel units) for a few frames, the register-streaming
    // kernel when no tensor maps are available or a batch has too many items for the persistent kernel
    if (ws.tmap_blur && n_frames >= 8) {
        int ipf = 0;
        for (int l = 0; l < fg.nlevels; ++l) ipf += ((fg.L[l].w + 127) / 128) * ((fg.L[l].h + 31) / 32);
        const long long total = (long long)ipf * n_frames;
        if (total > 0 && total < (1LL << 31)) {
            static int resident_ctas[64] = {0};          // per device (a process may drive several GPUs)
            const int smem = kBmWarps * kBmStageBytes;
            int dev = 0;
            cudaGetDevice(&dev);
            if (resident_ctas[dev & 63] == 0) {
                int n_sm = 0, per_sm = 0;
                cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
                cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, blur_mma_kernel, 32 * kBmWarps, smem);
                if (e != cudaSuccess) return e;
                resident_ctas[dev & 63] = std::max(n_sm, 1) * std::max(per_sm, 1);
            }
            const int ctas = (int)std::min<long long>((total + kBmWarps - 1) / kBmWarps, (long long)resident_ctas[dev & 63]);
            blur_mma_kernel<<<ctas, 32 * kBmWarps, smem, st>>>(fg, ws, ipf, (int)total);
            count_launch();
            return cudaGetLastError();
        }
    }
    if (!ws.tmap_blur || n_frames >= 8) {
        int items = 0;
        for (int l = 0; l < fg.nlevels; ++l) items += ((fg.L[l].w + 127) / 128) * ((fg.L[l].h + BS_ROWS - 1) / BS_ROWS);
        dim3 sgrid((items + 3) / 4, n_frames);
        blur_stream_kernel<<<sgrid, 128, 0, st>>>(fg, ws);
        count_launch();
        return cudaGetLastError();
    }
    int tiles = 0;
    for (int l = 0; l < fg.nlevels; ++l) tiles += ((fg.L[l].w + BT_W - 1) / BT_W) * ((fg.L[l].h + BT_H - 1) / BT_H);
    dim3 grid(tiles, n_frames);
    blur_kernel<<<grid, 256, 0, st>>>(fg, ws);
    count_launch();
    return cudaGetLastError();
}

static cudaError_t fill_describe_tables()
{
    static const int8_t pat[1024] = {
#include "brief_pattern.inc"
    };
    static const int umax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};
    float4 pf[8][32];
    for (int lane = 0; lane < 32; ++lane)
        for (int k = 0; k < 8; ++k) {
            const int8_t* t = pat + 4 * (8 * lane + k);
            pf[k][lane] = make_float4((float)t[0], (float)t[1], (float)t[2], (float)t[3]);
        }
    uint32_t mask[16][8];
    for (int av = 0; av < 16; ++av)
        for (int j = 0; j < 8; ++j) {
            uint32_t m = 0;
            for (int bb = 0; bb < 4; ++bb) {
                const int u = -15 + 4 * j + bb;
                if ((u < 0 ? -u : u) <= umax[av]) m |= 0xffu << (8 * bb);
            }
            mask[av][j] = m;
        }
    cudaError_t e = cudaMemcpyToSymbol(d_pattern_f, pf, sizeof pf);
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbol(d_mom_mask, mask, sizeof mask);
}

// The packing into io's slabs is fused when the lapping area allows it; *fused tells the caller whether pack_kernel is still
// needed.
cudaError_t launch_orient_describe(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st, int lap0, int lap1,
                                   const ChunkIO& io, bool* fused)
{
    FusedPack fp{};
    // a few frames only: the fused stores are scattered (7 lanes x 4 bytes per keypoint), which costs a 512-frame batch more than
    // the separate pack pass (measured 0.607 vs 0.557 + 0.024 ms), while a single frame saves a whole launch on its critical path
    if (fg.kp_slots > 0 && n_frames < 8) {
        // output x = level x * scale lies in [19, cols): the lapping test px >= lap0 && px <= lap1 is decided by the bounds
        if (lap1 < kEdge || lap0 >= fg.cols || lap0 > lap1) fp.mode = 1;
        else if (lap0 <= kEdge && lap1 >= fg.cols) fp.mode = 2;
        fp.io = io;
    }
    if (fused) *fused = fp.mode != 0;
    static bool filled[64] = {false};      // per device (the tables are __device__ symbols, one copy per context)
    static std::mutex mu;                  // the left / right extractors launch from two host threads
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    if (!filled[dev & 63]) {
        cudaError_t e = fill_describe_tables();          // synchronous copy: ordered before every later launch
        if (e != cudaSuccess) return e;
        filled[dev & 63] = true;
    }
    dim3 grid((fg.kp_slots + 7) / 8, n_frames);
    if (ws.tmap_desc) orient_describe_kernel<true><<<grid, 256, 8 * kOdStage, st>>>(fg, ws, fp);
    else orient_describe_kernel<false><<<grid, 256, 0, st>>>(fg, ws, fp);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_pack(const FrameGeom& fg, const Workspace& ws, int n_frames, int lap0, int lap1, const ChunkIO& io, cudaStream_t st)
{
    if (n_frames >= 8) pack_kernel<256><<<n_frames, 256, 0, st>>>(fg, ws, lap0, lap1, io);
    else pack_kernel<1024><<<n_frames, 1024, 0, st>>>(fg, ws, lap0, lap1, io);
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
