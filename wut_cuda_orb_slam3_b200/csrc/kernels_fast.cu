// kernels_fast.cu — grid FAST-9/16 with the iniThFAST/minThFAST two-threshold retry per 35-px cell.
//
// Semantics reproduced: the CPU cell loop `tileCalcKeypoints` (reference src/ORBextractor.cc:867-950, window at
// 958-966): every cell is an independent cv::FAST(roi, iniThFAST, nms=true) call on the (wCell+6)x(hCell+6) ROI and,
// only if that returns nothing, cv::FAST(roi, minThFAST, true).  cv::FAST evaluates ROI pixels >= 3 px from the ROI
// edge, its 3x3 strict-'>' NMS sees un-evaluated neighbours as 0, and keypoints come out in (y,x) order.
//
// One score pass is enough: the FAST score (max threshold for which the pixel is still a corner) does not depend on
// the detection threshold, so FAST(roi, ini) == {k in FAST(roi, min): score >= ini} (SURVEY.md Appendix A.2).
//
// Mapping: one 128-thread CTA per cell (exactly the reference's unit of independence, so NMS is naturally
// cell-masked).  ROI -> shared memory with aligned 32-bit loads, 8-point pre-test + shared-memory compaction so that
// the expensive arc test runs on dense warps, packed s16x2 min/max (VIMNMX.S16x2) computes the bright and dark arc
// scores at once, NMS only visits pre-test survivors, and position-indexed bitmaps + a warp scan write the survivors
// in (y,x) order into the cell's staging slot (no atomics on the output order).
#include "orbx_internal.cuh"

#include <algorithm>

namespace orbx {

namespace {

constexpr int kRoiPitch = 80;                   // >= 3 (misalignment) + 70 + 6, multiple of 16
constexpr int kRoiRows = 76;                    // >= 70 + 6
constexpr int kPlane = kRoiRows * kRoiPitch;    // ROI plane and score plane share one geometry
constexpr int kMaxEval = kMaxCellDim * kMaxCellDim;
constexpr int kListCap = kMaxEval + 4 * 32;     // four warp-private regions, each rounded up to 32
constexpr int kBitWords = (kPlane + 31) / 32;   // survivor bitmaps are indexed by plane position

// Shared-memory accessors on explicit 32-bit shared addresses.  (nvcc re-derives the shared-window base — S2UR
// SR_CgaCtaId + ULEA — at every use inside divergent regions when it goes through C++ pointers; the first version of this
// kernel spent ~15 % of its issue slots on that.)  Offsets are compile-time immediates folded into the instruction.
#define ORBX_LDS_U8(dst, addr, off) asm volatile("ld.shared.u8 %0, [%1+" #off "];" : "=r"(dst) : "r"(addr))
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts_u8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_u32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_zero16(uint32_t a) { asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(a), "r"(0u) : "memory"); }
__device__ __forceinline__ void atom_or(uint32_t a, uint32_t v) { asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }

// FAST score of the pixel whose plane address is `c`: max over the 16 arcs of 9 contiguous circle pixels of
// min(v - ring) / min(ring - v), minus 1.  Both signs are carried in one register as s16x2 (low = v - ring "centre
// brighter", high = ring - v) so one VIMNMX.S16x2 serves both.
//   packing:  A = (v+1, 1-v),  ~(r, -r) = r*0xFFFF - 1  ->  P = A + ~(r,-r) per half = (v - r, r - v)
//   windows:  prefix/suffix minima inside the two half-circles, window k = min(suffix(k), prefix(k+8))
__device__ __forceinline__ int fast_score(uint32_t c)
{
    // base moved to the top-left of the 7x7 neighbourhood so that every offset is a non-negative immediate
    const uint32_t b = c - 3 * kRoiPitch - 3;
    uint32_t v, r[16];
    ORBX_LDS_U8(v, b, 243);       // (3,3)
    ORBX_LDS_U8(r[0], b, 483);    // ( 0, 3): row 6, col 3
    ORBX_LDS_U8(r[1], b, 484);    // ( 1, 3)
    ORBX_LDS_U8(r[2], b, 405);    // ( 2, 2): row 5, col 5
    ORBX_LDS_U8(r[3], b, 326);    // ( 3, 1): row 4, col 6
    ORBX_LDS_U8(r[4], b, 246);    // ( 3, 0)
    ORBX_LDS_U8(r[5], b, 166);    // ( 3,-1): row 2, col 6
    ORBX_LDS_U8(r[6], b, 85);     // ( 2,-2): row 1, col 5
    ORBX_LDS_U8(r[7], b, 4);      // ( 1,-3): row 0, col 4
    ORBX_LDS_U8(r[8], b, 3);      // ( 0,-3)
    ORBX_LDS_U8(r[9], b, 2);      // (-1,-3)
    ORBX_LDS_U8(r[10], b, 81);    // (-2,-2): row 1, col 1
    ORBX_LDS_U8(r[11], b, 160);   // (-3,-1): row 2, col 0
    ORBX_LDS_U8(r[12], b, 240);   // (-3, 0)
    ORBX_LDS_U8(r[13], b, 320);   // (-3, 1)
    ORBX_LDS_U8(r[14], b, 401);   // (-2, 2): row 5, col 1
    ORBX_LDS_U8(r[15], b, 482);   // (-1, 3): row 6, col 2
    const uint32_t A = v * 0xFFFF0001u + 0x00010001u;
    uint32_t P[16], pf[16], sf[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) P[k] = __vadd2(A, r[k] * 0xFFFFu + 0xFFFFFFFFu);
    pf[0] = P[0]; pf[8] = P[8]; sf[7] = P[7]; sf[15] = P[15];
#pragma unroll
    for (int k = 1; k < 8; ++k) {
        pf[k] = __vmins2(pf[k - 1], P[k]);
        pf[8 + k] = __vmins2(pf[8 + k - 1], P[8 + k]);
        sf[7 - k] = __vmins2(sf[8 - k], P[7 - k]);
        sf[15 - k] = __vmins2(sf[16 - k], P[15 - k]);
    }
    uint32_t w[16];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        w[k] = __vmins2(sf[k], pf[k + 8]);        // window k..k+8
        w[k + 8] = __vmins2(sf[k + 8], pf[k]);    // window k+8..k+16
    }
#pragma unroll
    for (int s = 8; s >= 1; s >>= 1)
#pragma unroll
        for (int k = 0; k < s; ++k) w[k] = __vmaxs2(w[k], w[k + s]);
    const int a = (int)(short)(w[0] & 0xffff), bb = (int)(short)(w[0] >> 16);
    return max(a, bb) - 1;
}
static_assert(kRoiPitch == 80, "fast_score() hard-codes the 7x7 offsets for an 80-byte pitch");

}  // namespace

__global__ void __launch_bounds__(128) fast_cells_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int cell_lo)
{
    __shared__ __align__(16) uint8_t roi[kPlane];
    __shared__ __align__(16) uint8_t sc[kPlane];
    __shared__ __align__(4) uint16_t list[kListCap];
    __shared__ uint32_t selA[kBitWords], selH[kBitWords];
    __shared__ int off[kBitWords];
    __shared__ int wcnt[4], total;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y;
    // cell -> (level, cell row, cell column) from a small table (built by the host with the geometry)
    const int gcell = cell_lo + (int)blockIdx.x;
    const uint32_t ct = __ldg(fg.cell_tab + gcell);
    const int level = ct & 15, ci = (ct >> 4) & 0xfff, cj = ct >> 16;
    const LevelGeom& g = fg.L[level];
    const int cell = gcell - g.cell_base;
    int* count_out = ws.cell_count + (size_t)frame * fg.total_cells + gcell;

    const int maxBX = g.w - kWinBorder, maxBY = g.h - kWinBorder;
    const int iniX = kWinBorder + cj * g.wCell, iniY = kWinBorder + ci * g.hCell;
    const int maxX = min(iniX + g.wCell + 6, maxBX), maxY = min(iniY + g.hCell + 6, maxBY);
    const int rw = maxX - iniX, rh = maxY - iniY;
    const int ew = rw - 6, eh = rh - 6;
    if (iniY >= maxBY - 3 || iniX >= maxBX - 6 || ew <= 0 || eh <= 0) {   // src/ORBextractor.cc:892,899
        if (tid == 0) *count_out = 0;
        return;
    }
    const int minTh = max(fg.minTh, 1), iniTh = fg.iniTh;
    const uint32_t roi_s = (uint32_t)__cvta_generic_to_shared(roi), sc_s = (uint32_t)__cvta_generic_to_shared(sc);
    const uint32_t list_s = (uint32_t)__cvta_generic_to_shared(list);
    const uint32_t selA_s = (uint32_t)__cvta_generic_to_shared(selA), selH_s = (uint32_t)__cvta_generic_to_shared(selH);

    // 1. ROI -> shared memory with aligned 32-bit loads (the row misalignment m is the same for every row because the
    //    pitch is a multiple of 16); zero the score plane and the survivor bitmaps
    const uint8_t* src = level_interior((const uint8_t*)ws.pyr, g, frame) + (size_t)iniY * g.pitch + iniX;
    const int m = (int)((uintptr_t)src & 3);
    {
        const int nwords = (m + rw + 3) >> 2;                   // <= 20
        const uint32_t* src4 = reinterpret_cast<const uint32_t*>(src - m) + lane;
        const int wpitch = g.pitch >> 2;
        // all global loads of this lane are issued before the first shared store (the stores are volatile asm, which would
        // otherwise serialise ~10 dependent L2 round trips at the start of every CTA)
        constexpr int kRowsPerWarp = (kRoiRows + 3) / 4;
        uint32_t tmp[kRowsPerWarp];
        const bool ld = lane < nwords;
#pragma unroll
        for (int k = 0; k < kRowsPerWarp; ++k) {
            const int y = warp + 4 * k;
            tmp[k] = (ld && y < rh) ? __ldg(src4 + (size_t)y * wpitch) : 0u;
        }
        const int nz = (rh * kRoiPitch + 15) >> 4;
        for (int i = tid; i < nz; i += 128) sts_zero16(sc_s + i * 16);
        for (int i = tid; i < kBitWords; i += 128) { sts_u32(selA_s + i * 4, 0); sts_u32(selH_s + i * 4, 0); }
#pragma unroll
        for (int k = 0; k < kRowsPerWarp; ++k) {
            const int y = warp + 4 * k;
            if (ld && y < rh) sts_u32(roi_s + y * kRoiPitch + lane * 4, tmp[k]);
        }
    }
    __syncthreads();

    // 2. pre-test on the 8 even circle points: every 9-arc contains one point of each opposite pair, so a corner needs
    //    max_p min(r_a, r_b) < v - t  (bright) or  min_p max(r_a, r_b) > v + t  (dark).  Each warp owns a contiguous
    //    quarter of the pixels and compacts its survivors (plane positions) into its own region of `list`: no atomics.
    const int npix = ew * eh;
    const int Q = (((npix + 3) >> 2) + 31) & ~31;               // pixels per warp, multiple of 32
    {
        const int e0 = warp * Q + lane;
        const int eend = min(warp * Q + Q, npix);               // warp-uniform end of this warp's range
        const float inv_ew = 1.0f / (float)ew;
        int ey = (int)(((float)e0 + 0.5f) * inv_ew);
        int ex = e0 - ey * ew;
        int pos = (ey + 3) * kRoiPitch + m + ex + 3;
        const int wrapfix = kRoiPitch - ew;
        const int safe = 3 * kRoiPitch + m + 3;                  // first evaluated pixel: a valid address for idle lanes
        uint32_t wl = list_s + (uint32_t)(warp * Q) * 2;        // write cursor of this warp (bytes)
        const int vlo = minTh, vhi = minTh;
        for (int base = warp * Q; base < eend; base += 32) {
            const bool valid = base + lane < eend;
            const uint32_t b = roi_s + (valid ? pos : safe) - 3 * kRoiPitch - 3;
            uint32_t v, r0, r2, r4, r6, r8, r10, r12, r14;
            ORBX_LDS_U8(v, b, 243);
            ORBX_LDS_U8(r0, b, 483);  ORBX_LDS_U8(r8, b, 3);
            ORBX_LDS_U8(r4, b, 246);  ORBX_LDS_U8(r12, b, 240);
            ORBX_LDS_U8(r2, b, 405);  ORBX_LDS_U8(r10, b, 81);
            ORBX_LDS_U8(r6, b, 85);   ORBX_LDS_U8(r14, b, 401);
            const int M1 = max(max(min(r0, r8), min(r4, r12)), max(min(r2, r10), min(r6, r14)));
            const int M2 = min(min(max(r0, r8), max(r4, r12)), min(max(r2, r10), max(r6, r14)));
            const bool pass = valid & ((M1 < (int)v - vlo) | (M2 > (int)v + vhi));
            const uint32_t mk = __ballot_sync(0xffffffffu, pass);
            if (pass) sts_u16(wl + 2 * __popc(mk & ((1u << lane) - 1)), (uint32_t)pos);
            wl += 2 * __popc(mk);
            ex += 32; pos += 32;
            while (ex >= ew) { ex -= ew; pos += wrapfix; }
        }
        if (lane == 0) wcnt[warp] = (int)((wl - list_s) >> 1) - warp * Q;
    }
    __syncthreads();

    // flat index over the four warp regions -> list slot
    const int c0 = wcnt[0], c1 = c0 + wcnt[1], c2 = c1 + wcnt[2], nl = c2 + wcnt[3];
    auto slot = [&](int i) { return i < c0 ? i : (i < c1 ? Q + i - c0 : (i < c2 ? 2 * Q + i - c1 : 3 * Q + i - c2)); };

    // 3. full arc score on the compacted list (order inside the list is irrelevant)
    for (int i = tid; i < nl; i += 128) {
        const uint32_t pos = lds_u16(list_s + 2 * slot(i));
        const int s = fast_score(roi_s + pos);
        if (s >= minTh) sts_u8(sc_s + pos, (uint32_t)s);
    }
    __syncthreads();

    // 4. 3x3 strict NMS inside the cell (pixels outside the evaluated region hold score 0 = cv::FAST's zeroed buffer);
    //    survivors set their bit in position-indexed bitmaps
    for (int i = tid; i < nl; i += 128) {
        const uint32_t pos = lds_u16(list_s + 2 * slot(i));
        const uint32_t b = sc_s + pos - kRoiPitch - 1;
        uint32_t s;
        ORBX_LDS_U8(s, b, 81);
        if (s > 0) {
            uint32_t n0, n1, n2, n3, n4, n5, n6, n7;
            ORBX_LDS_U8(n0, b, 0);   ORBX_LDS_U8(n1, b, 1);   ORBX_LDS_U8(n2, b, 2);
            ORBX_LDS_U8(n3, b, 80);  ORBX_LDS_U8(n4, b, 82);
            ORBX_LDS_U8(n5, b, 160); ORBX_LDS_U8(n6, b, 161); ORBX_LDS_U8(n7, b, 162);
            const uint32_t mx = max(max(max(n0, n1), max(n2, n3)), max(max(n4, n5), max(n6, n7)));
            if (s > mx) {
                atom_or(selA_s + (pos >> 5) * 4, 1u << (pos & 31));
                if ((int)s >= iniTh) atom_or(selH_s + (pos >> 5) * 4, 1u << (pos & 31));
            }
        }
    }
    __syncthreads();

    // 5. per-cell threshold selection (ini if it yields anything, else min) + exclusive offsets (warp 0)
    const int nwordsB = ((rh * kRoiPitch) + 31) >> 5;
    if (warp == 0) {
        uint32_t anyH = 0;
        for (int w = lane; w < nwordsB; w += 32) anyH |= selH[w];
        anyH = __ballot_sync(0xffffffffu, anyH != 0);
        int running = 0;
        for (int base = 0; base < nwordsB; base += 32) {
            const int w = base + lane;
            uint32_t mk = 0;
            if (w < nwordsB) { mk = anyH ? selH[w] : selA[w]; selA[w] = mk; }
            const int cnt = __popc(mk);
            int incl = cnt;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, incl, d);
                if (lane >= d) incl += t;
            }
            if (w < nwordsB) off[w] = running + incl - cnt;
            running += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) { total = running; *count_out = running; }
    }
    __syncthreads();

    // 6. ordered scatter: plane position order == (y, x) order
    if (total == 0) return;
    uint32_t* out = ws.cand + (size_t)frame * fg.cand_frame_stride + g.cand_off + (size_t)cell * g.cell_cap;
    const int xbase = cj * g.wCell - m, ybase = ci * g.hCell;          // x_rel = cj*wCell + 3 + ex, ex = col - m - 3
    for (int w = tid; w < nwordsB; w += 128) {
        uint32_t mk = selA[w];
        int o = off[w];
        while (mk) {
            const int b = __ffs(mk) - 1;
            mk &= mk - 1;
            const int pos = (w << 5) + b;
            const int y = pos / kRoiPitch, x = pos - y * kRoiPitch;
            out[o++] = (uint32_t)(xbase + x) | ((uint32_t)(ybase + y) << 12) | ((uint32_t)sc[pos] << 24);
        }
    }
}

// =====================================================================================================================
// Throughput kernel: ONE WARP PER CELL (4 independent warps per CTA, no CTA-wide barrier).
//
// The CTA-per-cell kernel above spends a fifth of its issue slots on per-CTA set-up (each of the 128 threads repeats it
// for only ~11 pixels) and evaluates the 8-point pre-test one pixel per lane.  Here a lane owns ~43 pixels, and:
//   * the ROI is staged as u16 per pixel (plane A: low byte = pixel, high byte = 0, later the pixel's FAST score), so one
//     aligned LDS.64 yields four horizontally adjacent pixels as two ready-made u16x2 operands: the pre-test handles FOUR
//     pixels per lane with VIMNMX.U16x2 / VIMNMX3.U16x2 and no unpacking (the odd-offset ring points (+-3, 0) take one
//     PRMT each); the threshold compare is two plain 32-bit IADD3 (biased so that the halves cannot borrow) + one max;
//   * the arc score packs (r, 255 - r) per ring pixel with one IMAD, takes all 16 nine-pixel arc maxima with two layers
//     of three-input max (m3[k] = max3(X[k..k+2]), m9[k] = max3(m3[k], m3[k+3], m3[k+6])) and min-reduces them with
//     three-input min: 40 VIMNMX3 instead of 59 two-input min/max;
//       low  half: min_k max_arc(r)       -> bright score = v - lo - 1
//       high half: min_k max_arc(255 - r) -> dark   score = (255 - hi) - v - 1
//   * scores live in the high bytes of plane A (the score/NMS phases use byte loads, the pre-test is over by then), the
//     ordered-scatter offsets stay in registers: ~7.6 KB of shared memory per cell;
//   * phases are separated by __syncwarp() only.
// PA = plane pitch in pixels (48 / 64 / 80).  The host launches one grid per group of consecutive pyramid levels with
// similar cell size (deep levels have few, taller cells), so that the shared-memory carve-up fits the group.
template <int PA>
__device__ __forceinline__ int fast_score16(uint32_t c /* byte address of the centre pixel in plane A */)
{
    const uint32_t b = c - (3 * PA + 3) * 2;
    uint32_t v, r[16];
#define ORBX_LDS_PX(dst, addr, off) asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(dst) : "r"(addr), "n"(off))
    ORBX_LDS_PX(v, b, (3 * PA + 3) * 2);
    ORBX_LDS_PX(r[0], b, (6 * PA + 3) * 2);    // ( 0, 3)
    ORBX_LDS_PX(r[1], b, (6 * PA + 4) * 2);    // ( 1, 3)
    ORBX_LDS_PX(r[2], b, (5 * PA + 5) * 2);    // ( 2, 2)
    ORBX_LDS_PX(r[3], b, (4 * PA + 6) * 2);    // ( 3, 1)
    ORBX_LDS_PX(r[4], b, (3 * PA + 6) * 2);    // ( 3, 0)
    ORBX_LDS_PX(r[5], b, (2 * PA + 6) * 2);    // ( 3,-1)
    ORBX_LDS_PX(r[6], b, (1 * PA + 5) * 2);    // ( 2,-2)
    ORBX_LDS_PX(r[7], b, (0 * PA + 4) * 2);    // ( 1,-3)
    ORBX_LDS_PX(r[8], b, (0 * PA + 3) * 2);    // ( 0,-3)
    ORBX_LDS_PX(r[9], b, (0 * PA + 2) * 2);    // (-1,-3)
    ORBX_LDS_PX(r[10], b, (1 * PA + 1) * 2);   // (-2,-2)
    ORBX_LDS_PX(r[11], b, (2 * PA + 0) * 2);   // (-3,-1)
    ORBX_LDS_PX(r[12], b, (3 * PA + 0) * 2);   // (-3, 0)
    ORBX_LDS_PX(r[13], b, (4 * PA + 0) * 2);   // (-3, 1)
    ORBX_LDS_PX(r[14], b, (5 * PA + 1) * 2);   // (-2, 2)
    ORBX_LDS_PX(r[15], b, (6 * PA + 2) * 2);   // (-1, 3)
#undef ORBX_LDS_PX
    uint32_t X[16], m3[16], m9[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) X[k] = r[k] * 0xFFFF0001u + 0x00FF0000u;     // (r, 255 - r)
#pragma unroll
    for (int k = 0; k < 16; ++k) m3[k] = __vmaxu2(__vmaxu2(X[k], X[(k + 1) & 15]), X[(k + 2) & 15]);
#pragma unroll
    for (int k = 0; k < 16; ++k) m9[k] = __vmaxu2(__vmaxu2(m3[k], m3[(k + 3) & 15]), m3[(k + 6) & 15]);
    uint32_t a0 = __vminu2(__vminu2(m9[0], m9[1]), m9[2]);
    uint32_t a1 = __vminu2(__vminu2(m9[3], m9[4]), m9[5]);
    uint32_t a2 = __vminu2(__vminu2(m9[6], m9[7]), m9[8]);
    uint32_t a3 = __vminu2(__vminu2(m9[9], m9[10]), m9[11]);
    uint32_t a4 = __vminu2(__vminu2(m9[12], m9[13]), m9[14]);
    a0 = __vminu2(__vminu2(a0, a1), a2);
    a3 = __vminu2(__vminu2(a3, a4), m9[15]);
    a0 = __vminu2(a0, a3);
    const int bright = (int)v - (int)(a0 & 0xffffu);
    const int dark = 255 - (int)(a0 >> 16) - (int)v;
    return max(bright, dark) - 1;
}

#ifndef ORBX_FAST_WPC
#define ORBX_FAST_WPC 1
#endif
constexpr int kWarpsPerCta = ORBX_FAST_WPC;

// per-warp shared-memory carve-up for a plane of `rows` x PA pixels and `list_cap` pre-test survivors
struct WarpSmem {
    int a_bytes;      // u16 plane (+ slack: the pre-test reads up to 4 pixels past the end of a row)
    int list_bytes;   // u16 positions of pre-test survivors
    int total;
};
__host__ __device__ inline WarpSmem warp_smem(int rows, int pa, int list_cap)
{
    WarpSmem s;
    s.a_bytes = (rows * pa * 2 + 16 + 15) & ~15;
    s.list_bytes = (list_cap * 2 + 15) & ~15;
    s.total = s.a_bytes + s.list_bytes;
    return s;
}

struct WarpLaunch {
    int cell_lo, cell_hi;   // global cell ids [lo, hi) handled by this launch
    int rows_alloc;         // plane rows (>= hCell + 6 of every level in the group)
    int list_cap;           // >= evaluated pixels of any cell in the group
};

template <int PA>
__global__ void __launch_bounds__(32 * kWarpsPerCta) fast_cells_warp_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, WarpLaunch wlc)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gcell = wlc.cell_lo + blockIdx.x * kWarpsPerCta + warp;
    if (gcell >= wlc.cell_hi) return;
    const int frame = blockIdx.y;
    const WarpSmem sm = warp_smem(wlc.rows_alloc, PA, wlc.list_cap);
    const uint32_t A_s = (uint32_t)__cvta_generic_to_shared(smem_raw) + (uint32_t)(warp * sm.total);
    const uint32_t list_s = A_s + sm.a_bytes;

    const uint32_t ct = __ldg(fg.cell_tab + gcell);
    const int level = ct & 15, ci = (ct >> 4) & 0xfff, cj = ct >> 16;
    const LevelGeom& g = fg.L[level];
    const int cell = gcell - g.cell_base;
    int* count_out = ws.cell_count + (size_t)frame * fg.total_cells + gcell;

    const int maxBX = g.w - kWinBorder, maxBY = g.h - kWinBorder;
    const int iniX = kWinBorder + cj * g.wCell, iniY = kWinBorder + ci * g.hCell;
    const int maxX = min(iniX + g.wCell + 6, maxBX), maxY = min(iniY + g.hCell + 6, maxBY);
    const int rw = maxX - iniX, rh = maxY - iniY;
    const int ew = rw - 6, eh = rh - 6;
    if (iniY >= maxBY - 3 || iniX >= maxBX - 6 || ew <= 0 || eh <= 0) {   // src/ORBextractor.cc:892,899
        if (lane == 0) *count_out = 0;
        return;
    }
    const int minTh = max(fg.minTh, 1), iniTh = fg.iniTh;

    // 1. ROI -> plane A (u16 per pixel, high byte 0 = "no score") with aligned 32-bit global loads; zero the bitmaps
    const uint8_t* src = level_interior((const uint8_t*)ws.pyr, g, frame) + (size_t)iniY * g.pitch + iniX;
    const int m = (int)((uintptr_t)src & 3);
    {
        constexpr int LPR = PA <= 64 ? 16 : 32;         // lanes per ROI row
        constexpr int RPI = 32 / LPR;                   // rows per warp iteration
        constexpr int U = 4;
        const int nwords = (m + rw + 3) >> 2;           // <= PA / 4
        const int wl = lane % LPR, rsub = lane / LPR;
        const uint32_t* src4 = reinterpret_cast<const uint32_t*>(src - m) + wl;
        const int wpitch = g.pitch >> 2;
        const bool ld = wl < nwords;
        for (int y0 = 0; y0 < rh; y0 += RPI * U) {
            uint32_t tmp[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int y = y0 + u * RPI + rsub;
                tmp[u] = (ld && y < rh) ? __ldg(src4 + (size_t)y * wpitch) : 0u;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int y = y0 + u * RPI + rsub;
                if (ld && y < rh) {
                    const uint32_t lo = __byte_perm(tmp[u], 0, 0x4140), hi = __byte_perm(tmp[u], 0, 0x4342);
                    asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(A_s + (uint32_t)(y * PA + wl * 4) * 2), "r"(lo), "r"(hi) : "memory");
                }
            }
        }
    }
    __syncwarp();

    // The two thresholds are two passes over the staged cell, exactly as the reference runs them (src/ORBextractor.cc:908-925):
    // FAST at iniThFAST and, only if that yields no keypoint, FAST at minThFAST.  Three quarters of the cells of a textured
    // frame stop after the first pass, whose pre-test lets a quarter as many pixels through as the minThFAST one (11 % against
    // 42 % over the levels of the synthetic frames) — the score, the NMS and the list handling shrink with it.  (Round 1
    // scored everything once at minThFAST and selected afterwards: the score does not depend on the threshold.)  A second pass
    // starts from a clean plane (the first pass's score bytes are cleared) and recomputes the same values for a superset.
    int ns = 0;
#pragma unroll 1
    for (int th = iniTh;; th = minTh) {
    // 2. pre-test on the 8 even circle points, FOUR pixels (two u16x2 pairs at x, x+2; x a multiple of 4) per lane: every
    //    9-arc contains one point of each opposite pair, so a corner needs max_p min(r_a, r_b) < v - t (bright) or
    //    min_p max(r_a, r_b) > v + t (dark).  Survivors are ballot-compacted into `list` (plane positions; order irrelevant).
    int nl;
    {
        const int xlo = m + 3, xhi = m + rw - 4;                // evaluated plane columns, inclusive
        const int ql = xlo >> 2, nQ = (xhi >> 2) - ql + 1;      // quads per row
        const int nItems = eh * nQ;
        const uint32_t magic = 0xFFFFFFFFu / (uint32_t)nQ + 1u; // exact floor(i / nQ) for i < 2^16 (nQ >= 2)
        // per half: 0x200 + v - M1 - t (bright) and 0x200 + M2 - v - t (dark) never borrow across halves: plain 32-bit adds
        const uint32_t K = 0x02000200u - (uint32_t)th * 0x00010001u;
        uint32_t wl = list_s;
        const uint32_t ltmask = (1u << lane) - 1u;
        for (int i0 = 0; i0 < nItems; i0 += 32) {
            const int i = min(i0 + lane, nItems - 1);
            const int row = nQ == 1 ? i : (int)__umulhi((uint32_t)i, magic);
            const int x = 4 * (ql + i - row * nQ);
            const int pos = (row + 3) * PA + x;
            const uint32_t b = A_s + (uint32_t)(pos - 3 * PA - 4) * 2;      // 3 rows up, 4 pixels left: all offsets >= 0
            uint32_t wm2, wm1, c0, c1, w2, w3, t0, t1, b0, b1, u10, ua, ub, d14, da, db, u2, d2;
#define ORBX_LDS_W(dst, off) asm volatile("ld.shared.u32 %0, [%1+%2];" : "=r"(dst) : "r"(b), "n"(off))
#define ORBX_LDS_W2(d0, d1, off) asm volatile("ld.shared.v2.u32 {%0, %1}, [%2+%3];" : "=r"(d0), "=r"(d1) : "r"(b), "n"(off))
            ORBX_LDS_W2(wm2, wm1, (3 * PA + 0) * 2);    // row y: pixels x-4 .. x-1
            ORBX_LDS_W2(c0, c1, (3 * PA + 4) * 2);      //        pixels x .. x+3
            ORBX_LDS_W2(w2, w3, (3 * PA + 8) * 2);      //        pixels x+4 .. x+7
            ORBX_LDS_W2(b0, b1, (6 * PA + 4) * 2);      // row y+3: ( 0, 3) of both pairs
            ORBX_LDS_W2(t0, t1, (0 * PA + 4) * 2);      // row y-3: ( 0,-3)
            ORBX_LDS_W(d14, (5 * PA + 2) * 2);          // row y+2: pixels x-2, x-1 -> (-2, 2) of pair 0
            ORBX_LDS_W2(da, db, (5 * PA + 4) * 2);      //          pixels x .. x+3 -> (-2, 2) of pair 1 | ( 2, 2) of pair 0
            ORBX_LDS_W(d2, (5 * PA + 8) * 2);           //          pixels x+4, x+5 -> ( 2, 2) of pair 1
            ORBX_LDS_W(u10, (1 * PA + 2) * 2);          // row y-2 likewise: (-2,-2) of pair 0
            ORBX_LDS_W2(ua, ub, (1 * PA + 4) * 2);      //          (-2,-2) of pair 1 | ( 2,-2) of pair 0
            ORBX_LDS_W(u2, (1 * PA + 8) * 2);           //          ( 2,-2) of pair 1
#undef ORBX_LDS_W
#undef ORBX_LDS_W2
            uint32_t p01, p23;
            {   // pair 0: pixels x, x+1.  Opposite pairs: (0,3)/(0,-3), (3,0)/(-3,0), (2,2)/(-2,-2), (2,-2)/(-2,2)
                const uint32_t r4 = __byte_perm(c1, w2, 0x5432), r12 = __byte_perm(wm2, wm1, 0x5432);
                const uint32_t M1 = __vmaxu2(__vmaxu2(__vminu2(b0, t0), __vminu2(r4, r12)), __vmaxu2(__vminu2(db, u10), __vminu2(ub, d14)));
                const uint32_t M2 = __vminu2(__vminu2(__vmaxu2(b0, t0), __vmaxu2(r4, r12)), __vminu2(__vmaxu2(db, u10), __vmaxu2(ub, d14)));
                p01 = __vmaxu2(c0 + K - M1, M2 + K - c0);
            }
            {   // pair 1: pixels x+2, x+3
                const uint32_t r4 = __byte_perm(w2, w3, 0x5432), r12 = __byte_perm(wm1, c0, 0x5432);
                const uint32_t M1 = __vmaxu2(__vmaxu2(__vminu2(b1, t1), __vminu2(r4, r12)), __vmaxu2(__vminu2(d2, ua), __vminu2(u2, da)));
                const uint32_t M2 = __vminu2(__vminu2(__vmaxu2(b1, t1), __vmaxu2(r4, r12)), __vminu2(__vmaxu2(d2, ua), __vmaxu2(u2, da)));
                p23 = __vmaxu2(c1 + K - M1, M2 + K - c1);
            }
            const bool valid = i0 + lane < nItems;
            const bool pass0 = valid && x >= xlo && (p01 & 0xffffu) > 0x200u;
            const bool pass1 = valid && x + 1 >= xlo && x + 1 <= xhi && p01 > 0x0200ffffu;
            const bool pass2 = valid && x + 2 >= xlo && x + 2 <= xhi && (p23 & 0xffffu) > 0x200u;
            const bool pass3 = valid && x + 3 <= xhi && p23 > 0x0200ffffu;
            const uint32_t mk0 = __ballot_sync(0xffffffffu, pass0), mk1 = __ballot_sync(0xffffffffu, pass1);
            const uint32_t mk2 = __ballot_sync(0xffffffffu, pass2), mk3 = __ballot_sync(0xffffffffu, pass3);
            if ((mk0 | mk1 | mk2 | mk3) == 0) continue;
            // lane-major order inside the iteration: lanes below me first, then my own earlier pixels
            uint32_t o = wl + 2 * (__popc(mk0 & ltmask) + __popc(mk1 & ltmask) + __popc(mk2 & ltmask) + __popc(mk3 & ltmask));
            if (pass0) { sts_u16(o, (uint32_t)pos); o += 2; }
            if (pass1) { sts_u16(o, (uint32_t)pos + 1); o += 2; }
            if (pass2) { sts_u16(o, (uint32_t)pos + 2); o += 2; }
            if (pass3) { sts_u16(o, (uint32_t)pos + 3); }
            wl += 2 * (__popc(mk0) + __popc(mk1) + __popc(mk2) + __popc(mk3));
        }
        nl = (int)((wl - list_s) >> 1);
    }
    __syncwarp();

    // 3. full arc score on the compacted list, two candidates per lane in flight; the score goes to the pixel's high byte
    for (int i = lane; i < nl; i += 64) {
        const bool two = i + 32 < nl;
        const uint32_t pos0 = lds_u16(list_s + 2 * i);
        const uint32_t pos1 = two ? lds_u16(list_s + 2 * (i + 32)) : pos0;
        const int s0 = fast_score16<PA>(A_s + pos0 * 2);
        const int s1 = fast_score16<PA>(A_s + pos1 * 2);
        if (s0 >= th) sts_u8(A_s + pos0 * 2 + 1, (uint32_t)s0);
        if (two && s1 >= th) sts_u8(A_s + pos1 * 2 + 1, (uint32_t)s1);
    }
    __syncwarp();

    // 4. 3x3 strict NMS inside the cell (pixels outside the evaluated region keep score 0 = cv::FAST's zeroed buffer).  The
    //    list is sorted by plane position (the pre-test compacts lane-major, lanes walk the cell row-major), so a ballot
    //    compaction of the survivors IN PLACE keeps (y, x) order: no bitmaps, no atomics.  Only scores >= th count: a pixel
    //    scored in the first pass that this pass's pre-test does not reach is not in the list, and every listed pixel's byte
    //    holds either 0 or a score >= the threshold of the pass that wrote it (>= th in both passes for listed pixels).
    ns = 0;
    {
        const uint32_t ltmask = (1u << lane) - 1u;
        for (int base = 0; base < nl; base += 32) {
            const int i = base + lane;
            uint32_t pos = 0, s = 0;
            if (i < nl) {
                pos = lds_u16(list_s + 2 * i);
                s = lds_u8(A_s + pos * 2 + 1);
            }
            bool keep = false;
            if (s > 0) {
                const uint32_t b = A_s + (pos - PA - 1) * 2 + 1;
                uint32_t n0, n1, n2, n3, n4, n5, n6, n7;
#define ORBX_LDS_B(dst, off) asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(dst) : "r"(b), "n"((off) * 2))
                ORBX_LDS_B(n0, 0);          ORBX_LDS_B(n1, 1);          ORBX_LDS_B(n2, 2);
                ORBX_LDS_B(n3, PA);         ORBX_LDS_B(n4, PA + 2);
                ORBX_LDS_B(n5, 2 * PA);     ORBX_LDS_B(n6, 2 * PA + 1); ORBX_LDS_B(n7, 2 * PA + 2);
#undef ORBX_LDS_B
                keep = s > max(max(max(n0, n1), max(n2, n3)), max(max(n4, n5), max(n6, n7)));
            }
            const uint32_t mk = __ballot_sync(0xffffffffu, keep);
            // every entry of this iteration is in registers and ns <= base: the in-place write cannot hit an unread entry
            if (keep) sts_u16(list_s + 2 * (ns + __popc(mk & ltmask)), pos);
            ns += __popc(mk);
        }
    }
    __syncwarp();
    if (ns > 0 || th == minTh) break;          // src/ORBextractor.cc:918: retry with minThFAST only if the cell stayed empty
    // The cell stayed empty although the pass may have stored scores (equal maxima next to each other suppress one another):
    // the pre-test of the next pass reads the plane as u16 pixels, so the score bytes go back to 0 first.  ns == 0: the in-place
    // compaction wrote nothing, the list still holds all nl entries of this pass.
    for (int i = lane; i < nl; i += 32) sts_u8(A_s + lds_u16(list_s + 2 * i) * 2 + 1, 0u);
    __syncwarp();
    }

    // 5. ordered output of the pass that produced keypoints
    const int total = ns;
    if (lane == 0) *count_out = total;
    if (total == 0) return;
    uint32_t* out = ws.cand + (size_t)frame * fg.cand_frame_stride + g.cand_off + (size_t)cell * g.cell_cap;
    const int xbase = cj * g.wCell - m, ybase = ci * g.hCell;
    {
        const uint32_t ltmask = (1u << lane) - 1u;
        int o = 0;
        for (int base = 0; base < ns; base += 32) {
            const int i = base + lane;
            uint32_t pos = 0, sc8 = 0;
            bool sel = false;
            if (i < ns) {
                pos = lds_u16(list_s + 2 * i);
                sc8 = lds_u8(A_s + pos * 2 + 1);
                sel = true;
            }
            const uint32_t mk = __ballot_sync(0xffffffffu, sel);
            if (sel) {
                const int y = (int)pos / PA, x = (int)pos - y * PA;
                out[o + __popc(mk & ltmask)] = (uint32_t)(xbase + x) | ((uint32_t)(ybase + y) << 12) | (sc8 << 24);
            }
            o += __popc(mk);
        }
    }
}

template <int PA>
static cudaError_t launch_fast_warp(const FrameGeom& fg, const Workspace& ws, int n_frames, const WarpLaunch& wlc, cudaStream_t st)
{
    const size_t smem = (size_t)warp_smem(wlc.rows_alloc, PA, wlc.list_cap).total * kWarpsPerCta;
    static size_t configured[64] = {0};  // per instantiation and device; grows monotonically (benign race: the attribute is idempotent)
    int dev = 0;
    cudaGetDevice(&dev);
    if (smem > configured[dev & 63]) {
        cudaError_t e = cudaFuncSetAttribute(fast_cells_warp_kernel<PA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        configured[dev & 63] = smem;
    }
    dim3 grid((wlc.cell_hi - wlc.cell_lo + kWarpsPerCta - 1) / kWarpsPerCta, n_frames);
    fast_cells_warp_kernel<PA><<<grid, 32 * kWarpsPerCta, smem, st>>>(fg, ws, wlc);
    count_launch();
    return cudaGetLastError();
}

static int plane_pitch_for(int wCell) { const int need = (3 + wCell + 6 + 3) & ~3; return need <= 48 ? 48 : (need <= 64 ? 64 : 80); }

// Levels [level_lo, level_hi) (level_hi <= 0: all).
cudaError_t launch_fast(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st, int level_lo, int level_hi)
{
    if (level_hi <= 0) level_hi = fg.nlevels;
    if (fg.total_cells == 0 || level_lo >= level_hi) return cudaSuccess;
    // Small jobs (single frames: the SLAM tracking case) keep one CTA per cell for latency; batches use one warp per cell.
    if ((long long)fg.total_cells * n_frames < 8192) {
        const int cell_lo = fg.L[level_lo].cell_base;
        const int cell_hi = fg.L[level_hi - 1].cell_base + fg.L[level_hi - 1].nCols * fg.L[level_hi - 1].nRows;
        if (cell_hi <= cell_lo) return cudaSuccess;
        dim3 grid(cell_hi - cell_lo, n_frames);
        fast_cells_kernel<<<grid, 128, 0, st>>>(fg, ws, cell_lo);
        count_launch();
        return cudaGetLastError();
    }
    // group consecutive levels whose cells have the same plane pitch and (within 10 %) the same height
    int l = level_lo;
    while (l < level_hi) {
        const LevelGeom& g0 = fg.L[l];
        if (g0.nCols <= 0 || g0.nRows <= 0) { ++l; continue; }
        const int pa = plane_pitch_for(g0.wCell);
        int min_h = g0.hCell, max_h = g0.hCell, max_w = g0.wCell, e = l + 1;
        int cell_hi = g0.cell_base + g0.nCols * g0.nRows;
        for (; e < level_hi; ++e) {
            const LevelGeom& g = fg.L[e];
            if (g.nCols <= 0 || g.nRows <= 0) continue;
            const int nmin = std::min(min_h, g.hCell), nmax = std::max(max_h, g.hCell);
            if (plane_pitch_for(g.wCell) != pa || nmax * 10 > nmin * 11 || g.cell_base != cell_hi) break;
            min_h = nmin; max_h = nmax; max_w = std::max(max_w, g.wCell);
            cell_hi = g.cell_base + g.nCols * g.nRows;
        }
        WarpLaunch wlc{g0.cell_base, cell_hi, max_h + 6, max_h * max_w + 8};
        cudaError_t err = pa == 48 ? launch_fast_warp<48>(fg, ws, n_frames, wlc, st)
                        : pa == 64 ? launch_fast_warp<64>(fg, ws, n_frames, wlc, st)
                                   : launch_fast_warp<80>(fg, ws, n_frames, wlc, st);
        if (err != cudaSuccess) return err;
        l = e;
    }
    return cudaSuccess;
}

}  // namespace orbx
