// kernels_pyramid.cu — ORBextractor::ComputePyramid (reference src/ORBextractor.cc:1309-1329) on sm_100a.
//
// Level 0 = copyMakeBorder(image, 19, BORDER_REFLECT_101); level l>0 = cv::resize(level l-1, INTER_LINEAR) followed
// by the same reflect-101 border.  The OpenCV 8U bilinear arithmetic is integer fixed point (11-bit coefficients,
// ((b0*(r0>>4))>>16)+((b1*(r1>>4))>>16)+2)>>2); the per-column / per-row source offsets and coefficients are computed
// once on the host with OpenCV's float/double formula (api.cu: build_resize_table) and read here from small tables,
// indexed by *bordered* coordinates so that the border needs no extra pass: a border pixel is simply the resized value
// at its reflected interior coordinate.
//
// Data layout: every level is a bordered buffer [rows+38][pitch] per frame, interior pixel (0,0) at byte
// 19*pitch + 32 (16-byte aligned), frames strided by pyr_frame_stride, levels by pyr_off.
//
// Kernels in this file (launch_pyramid picks per level):
//   pyr_level0_tiled_kernel   level 0: 128 x 32 tiles, 16-byte loads / stores (realigned word loads for unaligned rows), the
//                             tile that owns the mirrored pixels writes the reflect-101 border
//   pyr_resize_pipe_kernel    levels >= 1, the production path: one warp per 128 x 16 item of the BORDERED level, source window
//                             by TMA into the warp's stage, IDP.2A horizontal pass, row sums in registers (scale <= 1.5)
//   pyr_resize_tiled_kernel   levels >= 1 without tensor maps / scale in (1.5, 2]: 128 x 32 (128 x 16) tiles, u16 sum plane
//   pyr_level0_kernel, pyr_resize_kernel   generic per-word fallbacks (tiny levels, scale > 2): each thread produces one aligned
//                             32-bit word of a bordered row
//   cvt_gray_kernel           cv::cvtColor RGB/BGR(A) -> grey of Tracking::GrabImage*
#include <limits.h>
#include <stdlib.h>

#include <algorithm>

#include "orbx_internal.cuh"

namespace orbx {

__device__ __forceinline__ int reflect101_dev(int i, int n)
{
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
    return i;
}

// Level 0: copy + border.  grid = (ceil(words/128), rows_alloc, frames)
__global__ void __launch_bounds__(128) pyr_level0_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, const ChunkIO io)
{
    const LevelGeom& g = fg.L[0];
    const int word = blockIdx.x * blockDim.x + threadIdx.x;
    const int brow = blockIdx.y;              // bordered row 0..h+37
    const int frame = blockIdx.z;
    if (word * 4 >= g.pitch) return;
    const int sy = reflect101_dev(brow - kEdge, g.h);
    const uint8_t* src = io.image(frame) + (size_t)sy * io.pitch;
    uint32_t out = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = word * 4 + j;           // buffer column
        const int x = c - kXPad;              // interior x
        uint32_t v = 0;
        if (x >= -kEdge && x < g.w + kEdge) v = __ldg(src + reflect101_dev(x, g.w));
        out |= v << (8 * j);
    }
    uint8_t* dst = ws.pyr + g.pyr_off + (size_t)frame * g.pyr_frame_stride + (size_t)brow * g.pitch;
    reinterpret_cast<uint32_t*>(dst)[word] = out;
}

// Level l >= 1 from level l-1.  grid = (ceil(words/128), rows_alloc, frames)
__global__ void __launch_bounds__(128) pyr_resize_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int level)
{
    const LevelGeom& g = fg.L[level];
    const LevelGeom& p = fg.L[level - 1];
    const int word = blockIdx.x * blockDim.x + threadIdx.x;
    const int brow = blockIdx.y;
    const int frame = blockIdx.z;
    if (word * 4 >= g.pitch) return;
    const uint2 yt = __ldg(g.ytab + brow);
    const int sy0 = yt.x & 0xffff, sy1 = yt.x >> 16;
    const int b0 = (int)(yt.y & 0xffff), b1 = (int)(yt.y >> 16);
    const uint8_t* S = level_interior((const uint8_t*)ws.pyr, p, frame);
    const uint8_t* S0 = S + (size_t)sy0 * p.pitch;
    const uint8_t* S1 = S + (size_t)sy1 * p.pitch;
    uint32_t out = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int c = word * 4 + j;
        const int bc = c - (kXPad - kEdge);   // bordered column 0..w+37
        uint32_t v = 0;
        if (bc >= 0 && bc < g.w + 2 * kEdge) {
            const uint2 xt = __ldg(g.xtab + bc);
            const int sx0 = xt.x & 0xffff, sx1 = xt.x >> 16;
            const int a0 = (int)(xt.y & 0xffff), a1 = (int)(xt.y >> 16);
            const int p00 = S0[sx0], p01 = S0[sx1], p10 = S1[sx0], p11 = S1[sx1];
            if (g.area2x) {
                v = (uint32_t)((p00 + p01 + p10 + p11 + 2) >> 2);
            } else {
                const int r0 = p00 * a0 + p01 * a1;
                const int r1 = p10 * a0 + p11 * a1;
                v = (uint32_t)((((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2) & 0xffu;
            }
        }
        out |= v << (8 * j);
    }
    uint8_t* dst = ws.pyr + g.pyr_off + (size_t)frame * g.pyr_frame_stride + (size_t)brow * g.pitch;
    reinterpret_cast<uint32_t*>(dst)[word] = out;
}

// ---- tiled kernels (the production path; the per-word kernels above are the generic fallback) -----------------------
// Reflect-101 border written by the tile that owns the mirrored interior pixels (tile = x0..x0+tw, y0..y0+th of the
// interior, pixels in shared memory `t` with pitch TP): horizontal bands are copied as whole 16-byte row segments,
// vertical bands (<= 19 columns) with byte stores; corners ride along with the vertical bands.
template <int TP>
__device__ __forceinline__ void write_border_mirrors(uint8_t* D, int pitch, int w, int h, int x0, int y0, int tw, int th,
                                                     const uint8_t* t, int tid, int nthreads)
{
    const bool top = y0 <= kEdge, bottom = y0 + th >= h - 1 - kEdge;
    // horizontal bands: row y (1..19) -> row -y ; row y (h-20..h-2) -> row 2(h-1)-y ; 16-byte segments
    if (top || bottom) {
        const int nv = (tw + 15) >> 4;
        for (int i = tid; i < th * nv; i += nthreads) {
            const int ty = i / nv, v = i - ty * nv;
            const int y = y0 + ty;
            int ym = INT_MIN;
            if (y >= 1 && y <= kEdge) ym = -y;
            else if (y >= h - 1 - kEdge && y <= h - 2) ym = 2 * (h - 1) - y;
            if (ym == INT_MIN) continue;
            uint8_t* dst = D + (ptrdiff_t)ym * pitch + x0 + v * 16;
            if (v * 16 + 16 <= tw) *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(t + ty * TP + v * 16);
            else for (int b = v * 16; b < tw; ++b) dst[b - v * 16] = t[ty * TP + b];
            // a level lower than 40 rows can have a row in both bands
            if (y >= 1 && y <= kEdge && y >= h - 1 - kEdge && y <= h - 2) {
                uint8_t* d2 = D + (ptrdiff_t)(2 * (h - 1) - y) * pitch + x0 + v * 16;
                for (int b = v * 16; b < min(tw, v * 16 + 16); ++b) d2[b - v * 16] = t[ty * TP + b];
            }
        }
    }
    // vertical bands: columns 1..19 -> -x, columns w-20..w-2 -> 2(w-1)-x, for every row of the tile and its row mirrors
    const int lx0 = max(x0, 1), lx1 = min(x0 + tw - 1, kEdge);                 // left band columns inside this tile
    const int rx0 = max(x0, w - 1 - kEdge), rx1 = min(x0 + tw - 1, w - 2);     // right band columns inside this tile
    const int nl = max(lx1 - lx0 + 1, 0), nr = max(rx1 - rx0 + 1, 0);
    const int nb = nl + nr;
    if (nb == 0) return;
    for (int i = tid; i < th * nb; i += nthreads) {
        const int ty = i / nb, k = i - ty * nb;
        const int x = k < nl ? lx0 + k : rx0 + (k - nl);
        const int y = y0 + ty;
        const uint8_t val = t[ty * TP + (x - x0)];
        int ys[3], ny = 1;
        ys[0] = y;
        if (y >= 1 && y <= kEdge) ys[ny++] = -y;
        if (y >= h - 1 - kEdge && y <= h - 2) ys[ny++] = 2 * (h - 1) - y;
        for (int a = 0; a < ny; ++a) {
            if (x >= 1 && x <= kEdge) D[(ptrdiff_t)ys[a] * pitch - x] = val;
            if (x >= w - 1 - kEdge && x <= w - 2) D[(ptrdiff_t)ys[a] * pitch + 2 * (w - 1) - x] = val;
        }
    }
}

// Level 0, fast path (16-byte aligned input rows): copy 128x16 tiles with 16-byte loads/stores + border mirrors.
constexpr int PT_W = 128, PT_THREADS = 256;
constexpr int L0_H = 32;                     // level-0 copy tile height

// One 128 x 32 tile of level 0 (copy + the border mirrors it owns); t = L0_H * PT_W bytes of shared memory.  No trailing barrier.
// `aligned`: image base, frame stride and pitch are multiples of 16 (16-byte loads).  Otherwise (e.g. 1241-pixel KITTI rows at
// pitch = cols) a 16-byte segment is read as its 4 - 5 covering aligned words and realigned with funnel shifts; the misalignment
// differs from row to row.  `img_end` = one past the last image byte: the fifth word is only read when it lies inside the images.
__device__ __forceinline__ void level0_tile(const LevelGeom& g, const Workspace& ws, const uint8_t* __restrict__ S, size_t in_pitch,
                                            uint8_t* t, int tid, int x0, int y0, int frame, bool aligned, const uint8_t* img_end)
{
    const int tw = min(PT_W, g.w - x0), th = min(L0_H, g.h - y0);
    uint8_t* D = level_interior(ws.pyr, g, frame);
    if (tid < L0_H * (PT_W / 16)) {
        const int ty = tid >> 3, v = tid & 7;
        if (ty < th && v * 16 < tw) {
            const uint8_t* sp = S + (size_t)(y0 + ty) * in_pitch + x0 + v * 16;
            uint8_t* dp = D + (size_t)(y0 + ty) * g.pitch + x0 + v * 16;
            if (v * 16 + 16 <= tw) {
                uint4 q;
                if (aligned) {
                    q = __ldg(reinterpret_cast<const uint4*>(sp));
                } else {
                    const int mis = (int)((uintptr_t)sp & 3);
                    const uint32_t* wp = reinterpret_cast<const uint32_t*>(sp - mis);
                    const uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2), w3 = __ldg(wp + 3);
                    uint32_t w4 = 0;
                    if (mis) {
                        if (reinterpret_cast<const uint8_t*>(wp + 5) <= img_end) w4 = __ldg(wp + 4);
                        else for (int b = 0; b < mis; ++b) w4 |= (uint32_t)__ldg(sp + 16 - mis + b) << (8 * b);
                    }
                    const int sh = 8 * mis;
                    q = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh), __funnelshift_r(w3, w4, sh));
                }
                *reinterpret_cast<uint4*>(t + ty * PT_W + v * 16) = q;
                *reinterpret_cast<uint4*>(dp) = q;
            } else {
                for (int b = 0; b < tw - v * 16; ++b) { const uint8_t c = __ldg(sp + b); t[ty * PT_W + v * 16 + b] = c; dp[b] = c; }
            }
        }
    }
    const bool edge = x0 <= kEdge || x0 + tw >= g.w - kEdge - 1 || y0 <= kEdge || y0 + th >= g.h - kEdge - 1;
    if (!edge) return;
    __syncthreads();
    write_border_mirrors<PT_W>(D, g.pitch, g.w, g.h, x0, y0, tw, th, t, tid, PT_THREADS);
}

// img_end[k]: one past the last image byte of set k
__global__ void __launch_bounds__(PT_THREADS) pyr_level0_tiled_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, const ChunkIO io,
                                                                     int aligned, const uint8_t* img_end0, const uint8_t* img_end1)
{
    __shared__ __align__(16) uint8_t t[L0_H * PT_W];
    const int frame = blockIdx.z;
    level0_tile(fg.L[0], ws, io.image(frame), io.pitch, t, threadIdx.x, blockIdx.x * PT_W, blockIdx.y * L0_H, frame, aligned != 0,
                frame >= io.split ? img_end1 : img_end0);
}

// The two fixed-point passes, the interior stores and the border mirrors of one 128 x PT_H tile whose source window is already
// staged in `src` (row pitch `spitch`, first staged column `cbase`, first staged row `symin`).  Shared by the one-tile-per-CTA
// kernel (a persistent two-stage variant was measured and dropped, DESIGN.md §7).  Ends without a barrier.
template <int PT_H>
__device__ __forceinline__ void resize_tile_passes(const LevelGeom& g, const Workspace& ws, const uint8_t* src, uint16_t* hbuf, uint8_t* outt,
                                                   const uint2* ytl, uint2 xt, int tid, int tx, int x0, int y0, int frame, int tw, int th,
                                                   int cbase, int spitch, int symin, int nrows)
{
    // horizontal pass: thread = output column, every other source row.  The vertical rule only ever uses (r >> 4), so the
    // shift is applied once here (the exact-2x path adds the raw sums and keeps them unshifted); sums are non-negative
    // (coefficients in [0, 2048]).  Pointer-stepped and unrolled: 2 LDS + 2 IMAD + SHF + STS per row.
    {
        // second tap = first tap + 1, except where the table clamps it to the last source column — and there its
        // coefficient is 0 (f = 0), so reading the byte after it changes nothing: one pointer, two immediate offsets
        const int c0 = (int)(xt.x & 0xffff) - cbase;
        const bool same = (xt.x >> 16) == (xt.x & 0xffff);
        const uint32_t a0 = (xt.y & 0xffff) + (same ? (xt.y >> 16) : 0u), a1 = same ? 0u : (xt.y >> 16);
        const int rfirst = tid >> 7;
        const uint8_t* q0 = src + c0 + rfirst * spitch;
        uint16_t* hb = hbuf + tx + rfirst * PT_W;
        const int step = (PT_THREADS / PT_W) * spitch;
        const int n = (nrows - rfirst + (PT_THREADS / PT_W) - 1) / (PT_THREADS / PT_W);
        const int sh = g.area2x ? 0 : 4;
#pragma unroll 4
        for (int i = 0; i < n; ++i) {
            *hb = (uint16_t)(((uint32_t)q0[0] * a0 + (uint32_t)q0[1] * a1) >> sh);
            q0 += step; hb += (PT_THREADS / PT_W) * PT_W;
        }
    }
    __syncthreads();

    // vertical pass: thread = 4 consecutive columns x PT_H/8 rows -> one 32-bit word per row of the output tile.
    // ((b * (r >> 4)) >> 16) with b <= 2048 and (r >> 4) < 2^15 is the high word of (b << 16) * (r >> 4): one IMAD.HI.
    {
        const int xq = (tid & 31) * 4;
#pragma unroll
        for (int k = 0; k < PT_H / 8; ++k) {
            const int ty = (tid >> 5) + 8 * k;
            const uint2 yt = ytl[ty];
            const uint2 r0 = *reinterpret_cast<const uint2*>(hbuf + ((int)(yt.x & 0xffff) - symin) * PT_W + xq);     // 4 x u16
            const uint2 r1 = *reinterpret_cast<const uint2*>(hbuf + ((int)(yt.x >> 16) - symin) * PT_W + xq);
            uint32_t p0, p1, p2, p3;
            if (g.area2x) {
                const uint32_t s01 = r0.x + r1.x + 0x00020002u, s23 = r0.y + r1.y + 0x00020002u;   // halves <= 1022: no carry across
                p0 = (s01 & 0xffffu) >> 2; p1 = s01 >> 18; p2 = (s23 & 0xffffu) >> 2; p3 = s23 >> 18;
            } else {
                const uint32_t b0 = yt.y << 16, b1 = yt.y & 0xffff0000u;
                auto f = [&](uint32_t a, uint32_t b) { return (__umulhi(b0, a) + __umulhi(b1, b) + 2) >> 2; };
                p0 = f(r0.x & 0xffffu, r1.x & 0xffffu); p1 = f(r0.x >> 16, r1.x >> 16);
                p2 = f(r0.y & 0xffffu, r1.y & 0xffffu); p3 = f(r0.y >> 16, r1.y >> 16);
            }
            // low bytes of p0..p3 -> one word (same truncation as the & 0xff of the scalar rule)
            const uint32_t o = __byte_perm(__byte_perm(p0, p1, 0x0040), __byte_perm(p2, p3, 0x0040), 0x5410);
            *reinterpret_cast<uint32_t*>(outt + ty * PT_W + xq) = o;
        }
    }
    __syncthreads();

    // interior: 16-byte stores (interior rows are 16-byte aligned and x0 is a multiple of 128)
    uint8_t* D = level_interior(ws.pyr, g, frame);
    for (int i = tid; i < PT_H * (PT_W / 16); i += PT_THREADS) {
        const int ty = i >> 3, v = i & 7;
        if (ty < th && v * 16 < tw) {
            uint8_t* dst = D + (size_t)(y0 + ty) * g.pitch + x0 + v * 16;
            if (v * 16 + 16 <= tw) *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(outt + ty * PT_W + v * 16);
            else for (int b = v * 16; b < tw; ++b) dst[b - v * 16] = outt[ty * PT_W + b];
        }
    }
    const bool edge = x0 <= kEdge || x0 + tw >= g.w - kEdge - 1 || y0 <= kEdge || y0 + th >= g.h - kEdge - 1;
    if (!edge) return;
    write_border_mirrors<PT_W>(D, g.pitch, g.w, g.h, x0, y0, tw, th, outt, tid, PT_THREADS);
}

// Level l >= 1: one CTA produces a 128 x PT_H tile of the level interior (32 rows for scale <= 1.5, 16 rows up to 2).  The
// source footprint is staged in shared memory with 16-byte loads, the horizontal fixed-point pass runs once per source row
// into a u16 plane (pre-shifted sums), the vertical pass combines two rows per output row (4 pixels per thread, 64-bit shared loads),
// and the finished tile is written with 16-byte stores.
constexpr int PT_MINB = 6;                     // CTAs per SM the register budget must allow (the kernel is occupancy-bound)
template <int PT_H, int PT_SR, int PT_SP>      // tile rows, source rows, source pitch (bytes, multiple of 16)
__global__ void __launch_bounds__(PT_THREADS, PT_MINB) pyr_resize_tiled_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int level)
{
    __shared__ __align__(128) uint8_t src[PT_SR * PT_SP];
    __shared__ __align__(16) uint16_t hbuf[PT_SR * PT_W];      // horizontal sums, pre-shifted: <= 255 * 2048 >> 4 = 32640
    __shared__ __align__(16) uint8_t outt[PT_H * PT_W];
    __shared__ uint2 ytl[PT_H];

    const LevelGeom& g = fg.L[level];
    const LevelGeom& p = fg.L[level - 1];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int x0 = blockIdx.x * PT_W, y0 = blockIdx.y * PT_H, frame = blockIdx.z;
    const int tw = min(PT_W, g.w - x0), th = min(PT_H, g.h - y0);
    const int tx = tid & (PT_W - 1);

    // tables are indexed by bordered coordinates: interior x -> entry x + 19
    const uint2 xt = __ldg(g.xtab + kEdge + x0 + min(tx, tw - 1));
    if (tid < PT_H) ytl[tid] = __ldg(g.ytab + kEdge + y0 + min(tid, th - 1));
    const uint2 xfirst = __ldg(g.xtab + kEdge + x0), xlast = __ldg(g.xtab + kEdge + x0 + tw - 1);
    const uint2 yfirst = __ldg(g.ytab + kEdge + y0), ylast = __ldg(g.ytab + kEdge + y0 + th - 1);
    const int sxmin = (int)(xfirst.x & 0xffff), sxmax = (int)(xlast.x >> 16);
    const int symin = (int)(yfirst.x & 0xffff), symax = (int)(ylast.x >> 16);
    const int nrows = symax - symin + 1;
    int cbase, spitch;                                       // first staged source column, staged row pitch (bytes)
    if (PT_H == 32 && ws.tmap_resize) {
        // TMA: one elected thread issues a 3-D tiled bulk copy of the source window (box sized for this level's scale on
        // the host); completion is signalled on an mbarrier, nobody spends instructions on the copy.
        __shared__ __align__(8) uint64_t bar;
        cbase = sxmin & ~15;                                 // TMA needs a 16-byte aligned box start for 1-byte elements
        spitch = p.tma_box_w;
        if (tid == 0) mbar_init(&bar, 1);
        __syncthreads();
        if (tid == 0) {
            mbar_expect_tx(&bar, (uint32_t)(p.tma_box_w * p.tma_box_h));
            tma_load_3d(src, ws.tmap_resize + (level - 1), &bar, kXPad + cbase, kEdge + symin, frame);
        }
        mbar_wait(&bar, 0);
    } else {
        cbase = sxmin & ~15;
        spitch = PT_SP;
        const int nvec = ((sxmax - cbase) >> 4) + 1;        // 16-byte vectors per source row
        const uint8_t* P = level_interior((const uint8_t*)ws.pyr, p, frame) + (size_t)symin * p.pitch + cbase;
        if (lane < nvec)
            for (int r = warp; r < nrows; r += PT_THREADS / 32)
                *reinterpret_cast<uint4*>(src + r * PT_SP + lane * 16) = __ldg(reinterpret_cast<const uint4*>(P + (size_t)r * p.pitch) + lane);
        __syncthreads();
    }

    resize_tile_passes<PT_H>(g, ws, src, hbuf, outt, ytl, xt, tid, tx, x0, y0, frame, tw, th, cbase, spitch, symin, nrows);
}

// ---- warp-streaming resize (the batch path) ------------------------------------------------------------------------------------
// The tiled kernel above spends 44 lane-instructions per pixel: two byte gathers per horizontal sum, a u16 plane in shared memory
// between the passes, a staged output tile, and byte-wise border mirrors on most tiles.  Here a WARP owns an item of 128 buffer
// columns x 16 rows of the BORDERED level (the resize tables are indexed by bordered coordinates, so a border pixel is an ordinary
// output whose taps are those of its mirror image: no mirror pass), a lane owns 4 adjacent columns = one aligned 32-bit word per row:
//   * source window of the item: one TMA box (cp.async.bulk.tensor.3d -> mbarrier) into the warp's own shared-memory stage; warps
//     are persistent and never meet at a CTA barrier (the blur kernel's scheme: the round trip of a warp's copy hides behind the
//     other ~30 resident warps);
//   * horizontal pass of one source row: the lane's 8 taps lie in two aligned 8-byte windows (outputs 0-1, outputs 2-3; fixed for
//     the item): 4 LDS.32, one PRMT per pair with a per-lane selector puts (s0, s0+1, s1, s1+1) in one word, and one IDP.2A per
//     output forms a0*s[x] + a1*s[x+1] with the table's (a0 | a1 << 16) word as it is;
//   * vertical pass: the source rows of the box are walked once, top to bottom; the sums of the last two rows stay in registers
//     (two register sets that swap roles, the loop is unrolled by two) and the pair (r-1, r) produces the output row the host's
//     schedule names — or two rows at the rim, where a border row and its mirror image are the same bytes;
//     (b*(r>>4))>>16 is the upper half of a 32-bit IMAD (the product has 27 bits), PRMT gathers the upper halves of two pixels,
//     the sum, +2 and >>2 act on two pixels at a time, the four pixels leave as one coalesced 32-bit store.
// Everything that depends on the item's position only (coefficients, windows, selectors, row schedule) is tabulated on the host
// (api.cu: configure), so an item starts with three 16-byte loads.  Same integer arithmetic as the kernels above: bit-identical
// (tests/test_gpu_round2.py::test_batch_pyramid_streaming_kernel_is_bit_exact, bench.py's cfg4 checksum).
constexpr int kRpWarps = 4;
constexpr int kRpRows = 16;                         // bordered output rows per item
constexpr int kRpCol0 = kXPad - kEdge - 1;          // first buffer column of column tile 0 (12: word aligned; bordered column -1)

__global__ void __launch_bounds__(32 * kRpWarps) pyr_resize_pipe_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int level,
                                                                        int stage_bytes, int ntx, int nstrips, int total_items,
                                                                        uint32_t magic_frame, uint32_t magic_ntx)
{
    extern __shared__ __align__(128) uint8_t rp_smem[];
    __shared__ __align__(8) uint64_t bars[kRpWarps];
    __shared__ uint4 sched[kRpWarps][32];
    const LevelGeom& g = fg.L[level];
    const LevelGeom& p = fg.L[level - 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint8_t* stage = rp_smem + (size_t)warp * stage_bytes;
    const uint32_t stage_s = (uint32_t)__cvta_generic_to_shared(stage);
    const uint32_t sched_s = (uint32_t)__cvta_generic_to_shared(&sched[warp][0]);
    if (lane == 0) mbar_init(&bars[warp], 1);
    __syncwarp();
    const int gw = blockIdx.x * kRpWarps + warp, nw = gridDim.x * kRpWarps;
    const int bw = p.rp_box_w, bh = p.rp_box_h;
    const int per_frame = ntx * nstrips;
    const uint32_t pitch = (uint32_t)g.pitch;
    uint32_t phase = 0;
    for (int item = gw; item < total_items; item += nw) {
        // item -> (frame, strip, column tile): quotients by multiplication with floor(2^32 / d), one correction step
        int frame = (int)__umulhi((uint32_t)item, magic_frame);
        int t = item - frame * per_frame;
        if (t >= per_frame) { t -= per_frame; ++frame; }
        int strip = (int)__umulhi((uint32_t)t, magic_ntx);
        int ct = t - strip * ntx;
        if (ct >= ntx) { ct -= ntx; ++strip; }
        const uint4* xl = reinterpret_cast<const uint4*>(g.rp_xlane) + ((size_t)ct * 32 + lane) * 2;
        const uint4 A = __ldg(xl), Q = __ldg(xl + 1);          // a0..a3 | selectors, windows, keep mask, box start column
        const uint4* ys = reinterpret_cast<const uint4*>(g.rp_ysched) + (size_t)strip * (bh + 1);
        const uint4 hd = __ldg(ys);                            // {first source row of the box, rows used, -, -}
        const uint4 e = __ldg(ys + 1 + min(lane, bh - 1));
        asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(sched_s + 16 * lane), "r"(e.x), "r"(e.y), "r"(e.z), "r"(e.w) : "memory");
        if (lane == 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            mbar_expect_tx(&bars[warp], (uint32_t)(bw * bh));
            tma_load_3d(stage, ws.tmap_rpipe + (level - 1), &bars[warp], kXPad + (int)Q.w, kEdge + (int)hd.x, frame);
        }
        __syncwarp();
        const uint32_t selA = Q.x & 0xffffu, selB = Q.x >> 16, keep = Q.z;
        uint32_t ra = stage_s + (Q.y & 0xffffu), rb = stage_s + (Q.y >> 16);
        unsigned long long out = (unsigned long long)(ws.pyr + g.pyr_off + (size_t)frame * g.pyr_frame_stride + (size_t)(strip * kRpRows) * pitch +
                                                      (kRpCol0 + ct * 128 + 4 * lane));
        asm volatile("" : "+l"(out));                          // one finished base pointer: a row address is a single mad.wide
        const int nbox = (int)hd.y;
        auto hrow = [&](uint32_t h[4]) {                       // horizontal sums (>> 4) of the next source row
            uint32_t w0, w1, w2, w3;
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(ra));
            asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(w1) : "r"(ra));
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w2) : "r"(rb));
            asm volatile("ld.shared.u32 %0, [%1+4];" : "=r"(w3) : "r"(rb));
            ra += bw; rb += bw;
            const uint32_t pa = __byte_perm(w0, w1, selA), pb = __byte_perm(w2, w3, selB);
            h[0] = __dp2a_lo(A.x, pa, 0u) >> 4; h[1] = __dp2a_hi(A.y, pa, 0u) >> 4;
            h[2] = __dp2a_lo(A.z, pb, 0u) >> 4; h[3] = __dp2a_hi(A.w, pb, 0u) >> 4;
        };
        auto emit = [&](int k, const uint32_t h0[4], const uint32_t h1[4]) {     // the output row(s) of source rows (k - 1, k)
            uint32_t b0, b1, rows, unused;
            asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(b0), "=r"(b1), "=r"(rows), "=r"(unused) : "r"(sched_s + 16 * k));
            if ((rows & 0xffffu) == 0xffffu) return;           // warp-uniform
            // b <= 2048 and h < 2^15: the products fit 32 bits, so (b * h) >> 16 is the upper half of a plain IMAD (IMAD.HI runs at
            // a quarter of its rate); PRMT pulls the upper halves of two pixels into one word, +2 and >> 2 act on both halves
            const uint32_t p01 = __byte_perm(b0 * h0[0], b0 * h0[1], 0x7632), q01 = __byte_perm(b1 * h1[0], b1 * h1[1], 0x7632);
            const uint32_t p23 = __byte_perm(b0 * h0[2], b0 * h0[3], 0x7632), q23 = __byte_perm(b1 * h1[2], b1 * h1[3], 0x7632);
            const uint32_t x01 = (p01 + q01 + 0x00020002u) >> 2, x23 = (p23 + q23 + 0x00020002u) >> 2;       // halves <= 1022
            const uint32_t o = __byte_perm(x01, x23, 0x6420) & keep;
            unsigned long long addr;
            asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(addr) : "r"(rows & 0xffffu), "r"(pitch), "l"(out));
            asm volatile("st.global.u32 [%0], %1;" ::"l"(addr), "r"(o) : "memory");
            if (rows >= 0x10000u) {                            // the mirror image of a border row: same bytes
                asm("mad.wide.u32 %0, %1, %2, %3;" : "=l"(addr) : "r"((rows >> 16) - 1u), "r"(pitch), "l"(out));
                asm volatile("st.global.u32 [%0], %1;" ::"l"(addr), "r"(o) : "memory");
            }
        };
        mbar_wait(&bars[warp], phase);
        phase ^= 1u;
        if (keep != 0) {                                       // lanes right of the bordered level have nothing to do
            uint32_t ha[4], hb[4];
            hrow(ha);                                          // source row 0 of the box
#pragma unroll 1
            for (int k = 1; k < nbox; k += 2) {
                hrow(hb);
                emit(k, ha, hb);
                if (k + 1 < nbox) {
                    hrow(ha);
                    emit(k + 1, hb, ha);
                }
            }
        }
        __syncwarp();                                          // every lane is done with the stage and the schedule
    }
}

// One level with the warp-streaming kernel; false = not applicable (the caller falls back to the tiled kernel).
static bool launch_resize_pipe(const FrameGeom& fg, const Workspace& ws, int level, int n_frames, cudaStream_t st)
{
    const LevelGeom& g = fg.L[level];
    const LevelGeom& p = fg.L[level - 1];
    if (p.rp_box_w < 16 || p.rp_box_h < 2 || p.rp_box_h > 31 || !g.rp_xlane || !g.rp_ysched) return false;
    // + 8: a lane's second 4-byte word may start at the end of the last staged row (its bytes are then not selected)
    const int stage_bytes = (p.rp_box_w * p.rp_box_h + 8 + 127) & ~127;
    const int smem = kRpWarps * stage_bytes;
    if (smem > 64 * 1024) return false;
    const int ntx = (g.w + 2 * kEdge + 1 + 127) / 128, nstrips = (g.h + 2 * kEdge + kRpRows - 1) / kRpRows;
    const long long total = (long long)ntx * nstrips * n_frames;
    if (total <= 0 || total >= (1LL << 31)) return false;
    static int n_sm_dev[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    if (n_sm_dev[dev & 63] == 0) {
        int n = 0;
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
        if (cudaFuncSetAttribute(pyr_resize_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024) != cudaSuccess) {
            cudaGetLastError();
            n_sm_dev[dev & 63] = -1;
        } else {
            n_sm_dev[dev & 63] = n > 0 ? n : 148;
        }
    }
    if (n_sm_dev[dev & 63] < 0) return false;
    const int per_sm = std::min(9, std::max(1, (200 * 1024) / (smem + 1024)));
    const int ctas = (int)std::min<long long>((total + kRpWarps - 1) / kRpWarps, (long long)n_sm_dev[dev & 63] * per_sm);
    const uint32_t magic_frame = (uint32_t)((1ULL << 32) / (uint64_t)(ntx * nstrips)), magic_ntx = (uint32_t)((1ULL << 32) / (uint64_t)ntx);
    pyr_resize_pipe_kernel<<<ctas, 32 * kRpWarps, smem, st>>>(fg, ws, level, stage_bytes, ntx, nstrips, (int)total,
                                                              ntx * nstrips > 1 ? magic_frame : 0xffffffffu, ntx > 1 ? magic_ntx : 0xffffffffu);
    return true;
}

// Levels [level_lo, level_hi) (level_hi <= 0: all); level l >= 1 reads level l - 1, which must be complete on `st`.
cudaError_t launch_pyramid(const FrameGeom& fg, const Workspace& ws, const ChunkIO& io, int n_frames, cudaStream_t st, int level_lo,
                           int level_hi)
{
    if (level_hi <= 0) level_hi = fg.nlevels;
    // One launch per level.  A cooperative kernel for the whole pyramid was measured slower on 512-frame batches (1.19 ms vs
    // 0.81 ms for the eight dependent launches): a resident wave of persistent CTAs that walks its tiles in a fixed order and
    // stops at seven grid-wide barriers loses more to imbalance and to the exposed TMA round trip of every tile than the
    // launches lose at their boundaries (the hardware deals CTAs out as SMs free up).
    for (int l = level_lo; l < level_hi; ++l) {
        const LevelGeom& g = fg.L[l];
        const int words = g.pitch / 4;
        dim3 grid((words + 127) / 128, g.rows_alloc, n_frames);
        const bool big = g.w >= 2 * kEdge + 2 && g.h >= 2 * kEdge + 2;      // border band narrower than the level
        if (l == 0) {
            const int n0 = std::min(io.split, n_frames), n1 = n_frames - n0;
            const bool aligned = (((uintptr_t)io.img0 | (n1 > 0 ? (uintptr_t)io.img1 : 0)) & 15) == 0 && (io.frame_stride & 15) == 0 &&
                                 (io.pitch & 15) == 0;
            dim3 tgrid((g.w + PT_W - 1) / PT_W, (g.h + L0_H - 1) / L0_H, n_frames);
            // one past the last byte the caller's images of each set hold (the last row of the last frame ends at its last pixel)
            auto img_end = [&](const uint8_t* img, int n) {
                return n > 0 ? img + (size_t)(n - 1) * io.frame_stride + (size_t)(g.h - 1) * io.pitch + g.w : nullptr;
            };
            if (big) pyr_level0_tiled_kernel<<<tgrid, PT_THREADS, 0, st>>>(fg, ws, io, aligned ? 1 : 0, img_end(io.img0, n0), img_end(io.img1, n1));
            else pyr_level0_kernel<<<grid, 128, 0, st>>>(fg, ws, io);
        } else {
            const LevelGeom& p = fg.L[l - 1];
            // source footprint of a tile must fit the staged window: scale <= 1.5 -> 128x32 tiles, <= 2 -> 128x16 tiles
            const bool s15 = 2LL * p.w <= 3LL * g.w && 2LL * p.h <= 3LL * g.h;
            const bool s20 = (long long)p.w <= 2LL * g.w && (long long)p.h <= 2LL * g.h;
            // warp-streaming kernel whenever it applies (batches: 0.45 vs 0.81 ms per 512 frames; a single frame: 49 vs 52 us for
            // the eight levels, a stereo pair 236 vs 247 us).  ORBX_PYR_PIPE=0 forces the tiled kernel: a test hook, the only way
            // the suite reaches the kernel that levels the streaming resize does not apply to take
            static const char* rp_env = getenv("ORBX_PYR_PIPE");
            const bool want_pipe = rp_env ? atoi(rp_env) != 0 : true;
            if (big && s15 && !g.area2x && want_pipe && ws.tmap_rpipe && launch_resize_pipe(fg, ws, l, n_frames, st)) {
                // launched
            } else if (big && s15) {
                dim3 tgrid((g.w + PT_W - 1) / PT_W, (g.h + 31) / 32, n_frames);
                pyr_resize_tiled_kernel<32, 52, 224><<<tgrid, PT_THREADS, 0, st>>>(fg, ws, l);
            } else if (big && s20) {
                dim3 tgrid((g.w + PT_W - 1) / PT_W, (g.h + 15) / 16, n_frames);
                pyr_resize_tiled_kernel<16, 34, 304><<<tgrid, PT_THREADS, 0, st>>>(fg, ws, l);
            } else {
                pyr_resize_kernel<<<grid, 128, 0, st>>>(fg, ws, l);
            }
        }
        count_launch();
    }
    return cudaGetLastError();
}

// ---- image prep: cv::cvtColor(RGB/BGR/RGBA/BGRA -> GRAY) of Tracking::GrabImage* (reference src/Tracking2.cc:289-316) ---------
// OpenCV 8U: gray = (R*9798 + G*19235 + B*3735 + 2^14) >> 15 (checked bit-exact against cv2 4.13 in tests/test_oracle_cv2.py).
// One thread = 4 output pixels: 3 (or 4) aligned 32-bit loads, one 32-bit store.  grid = (ceil(cols/4/128), rows, frames).
template <int CH>
__global__ void __launch_bounds__(128) cvt_gray_kernel(const uint8_t* __restrict__ src, size_t src_pitch, size_t src_frame_stride, int swap_rb,
                                                       int rows, int cols, uint8_t* __restrict__ dst, size_t dst_pitch, size_t dst_frame_stride)
{
    const int x4 = blockIdx.x * 128 + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
    const int x = 4 * x4;
    if (x >= cols) return;
    const uint8_t* sp = src + (size_t)f * src_frame_stride + (size_t)y * src_pitch + (size_t)x * CH;
    uint8_t* dp = dst + (size_t)f * dst_frame_stride + (size_t)y * dst_pitch + x;
    const int c0 = swap_rb ? 3735 : 9798, c2 = swap_rb ? 9798 : 3735;          // weight of channel 0 / channel 2
    uint32_t px[4] = {0, 0, 0, 0};                                             // packed (ch0, ch1, ch2) per pixel
    const bool vec = x + 4 <= cols && (((uintptr_t)sp | src_pitch | src_frame_stride) & 3) == 0;
    if (vec) {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(sp);
        if (CH == 4) {
#pragma unroll
            for (int i = 0; i < 4; ++i) px[i] = __ldg(w + i);
        } else {
            const uint32_t a = __ldg(w), b = __ldg(w + 1), c = __ldg(w + 2);      // a = p0.012 p1.0 | b = p1.12 p2.01 | c = p2.2 p3.012
            px[0] = a; px[1] = __funnelshift_r(a, b, 24); px[2] = __funnelshift_r(b, c, 16); px[3] = c >> 8;
        }
    } else {
        for (int i = 0; i < 4 && x + i < cols; ++i)
            px[i] = (uint32_t)sp[i * CH] | ((uint32_t)sp[i * CH + 1] << 8) | ((uint32_t)sp[i * CH + 2] << 16);
    }
    uint32_t out = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const uint32_t v = (px[i] & 0xff) * c0 + ((px[i] >> 8) & 0xff) * 19235u + ((px[i] >> 16) & 0xff) * c2 + (1u << 14);
        out |= (v >> 15) << (8 * i);
    }
    if (x + 4 <= cols && (((uintptr_t)dp) & 3) == 0) *reinterpret_cast<uint32_t*>(dp) = out;
    else for (int i = 0; i < 4 && x + i < cols; ++i) dp[i] = (uint8_t)(out >> (8 * i));
}

cudaError_t launch_cvt_gray(const uint8_t* d_src, size_t src_pitch, size_t src_frame_stride, int channels, int rgb, int n_frames,
                            int rows, int cols, uint8_t* d_dst, size_t dst_pitch, size_t dst_frame_stride, cudaStream_t st)
{
    if (n_frames <= 0 || rows <= 0 || cols <= 0) return cudaSuccess;
    dim3 grid(((cols + 3) / 4 + 127) / 128, rows, n_frames);
    // channel 0 is R for RGB / RGBA input (mbRGB, src/Tracking2.cc:292-296) and B for BGR / BGRA
    if (channels == 3) cvt_gray_kernel<3><<<grid, 128, 0, st>>>(d_src, src_pitch, src_frame_stride, rgb ? 0 : 1, rows, cols, d_dst, dst_pitch, dst_frame_stride);
    else cvt_gray_kernel<4><<<grid, 128, 0, st>>>(d_src, src_pitch, src_frame_stride, rgb ? 0 : 1, rows, cols, d_dst, dst_pitch, dst_frame_stride);
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
