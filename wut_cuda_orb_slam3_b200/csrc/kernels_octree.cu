// kernels_octree.cu — ORBextractor::DistributeOctTree (reference src/ORBextractor.cc:584-774, DivideNode 515-567,
// compareNodes 569-582) as a deterministic array algorithm: one CTA per (frame, level).
//
// Reformulation (bit-exact, see DESIGN.md "Octree"):
//  * A key's path through the quadtree depends only on geometry: root = (int)(x / hX), then at every depth the
//    quadrant given by x < UL.x + ceil(w/2), y < UL.y + ceil(h/2).  Every key gets a path code (root, 2 bits per depth,
//    n1=0,n2=1,n3=2,n4=3).  ONE counting sort on the leading root + 2*Dsort bits of the code (shared-memory atomics; Dsort = 5
//    for the usual two roots) makes every node down to depth Dsort a contiguous segment whose child boundaries are plain
//    look-ups in the scanned bin table — the tree of N ~ 200 nodes rarely goes deeper.  A node below depth Dsort covers a
//    few pixels and holds a handful of keys: the lane that splits it partitions its segment in place by the next two code
//    bits.  DivideNode's stable partition keeps a node's keys in original (cell-major, y, x) order; that order only matters
//    for the "first key with maximal response" rule, which is evaluated on the carried original position (the key's slot in
//    the FAST staging area is monotone in it), so the order inside a segment is free.
//  * The std::list is an array in list order.  A sweep that splits a set of nodes processed in the order p=0..nS-1
//    turns the list into [children(p=nS-1) n4..n1, ..., children(p=0) n4..n1, untouched nodes in old order]
//    (every split push_front()s its non-empty children n1..n4 and erases the parent).  Positions come from prefix sums.
//  * Phase 1 (src 635-693) splits every node with >1 key in list order.  Phase 2 (699-752) sorts the expandable
//    nodes with std::sort(compareNodes) — replayed exactly (introsort_replay.h) because ties are broken by the
//    algorithm's internal permutation — and splits from the back until size >= N.
//  * Retain (756-771): first key with maximal response per node, in list order.
#include <mutex>

#include "introsort_replay.h"
#include "orbx_internal.cuh"

namespace orbx {

namespace {

constexpr int kSortBitsMax = 12;            // counting-sort bins: root bits + 2 * Dsort <= 12 (16 KB of bin starts)

struct Smem {
    // carved from dynamic shared memory; M = node capacity
    int* bstart;           // [nb + 1] first sorted position of every bin (exclusive scan of the bin counts)
    int* cursor;           // [nb] scatter cursors; aliases the node arrays below (dead before the roots are built)
    int* warp_tmp;         // [64]
    int* sort_stk;         // [3*72]
    uint32_t* nbeg[2];     // node segment begin           [M] x2 (ping-pong)
    uint32_t* ncnt[2];     // node key count
    uint32_t* nx[2];       // ULx | URx << 16
    uint32_t* ndep[2];     // depth
    uint32_t* npre[2];     // path-code prefix of the node (root, 2 bits per depth)
    uint32_t* cc;          // [4*M] child counts of processed node p: cc[4*p+k]
    int* sa;               // [M] scan scratch a
    int* sb;               // [M] scan scratch b
    int* sc;               // [M] scan scratch c
    int* sd;               // [M] scratch d
    int* procpos;          // [M] list position of the p-th processed node
    unsigned long long* vec;   // [M] expandable nodes, creation order: (cnt<<13 | ULx) << 32 | list position
    unsigned long long* vec2;  // [M]
};

// Exclusive prefix sum of a[0..n) in place (int), returns the total.  All T threads must call.
template <int T>
__device__ int block_exclusive_scan(int* a, int n, int* warp_tmp)
{
    __shared__ int carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < n; base += T) {
        const int i = base + tid;
        const int v = i < n ? a[i] : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (lane == 31) warp_tmp[warp] = incl;
        __syncthreads();
        int woff = 0;
        for (int w = 0; w < warp; ++w) woff += warp_tmp[w];
        const int c = carry;
        if (i < n) a[i] = c + woff + incl - v;
        __syncthreads();
        if (tid == T - 1) carry = c + woff + incl;
        __syncthreads();
    }
    const int total = carry;
    __syncthreads();            // nobody may re-enter (and reset carry) before everyone has read the total
    return total;
}

// Exclusive prefix sum of a[0..n) in place, raking: thread t owns ceil(n / T) consecutive elements (one pass, three barriers
// whatever n is).  Returns the total.  All T threads must call.
template <int T>
__device__ int block_exclusive_scan_raking(int* a, int n, int* warp_tmp)
{
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int per = (n + T - 1) / T;
    const int i0 = min(tid * per, n), i1 = min(i0 + per, n);
    int sum = 0;
    for (int i = i0; i < i1; ++i) sum += a[i];
    int incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += t;
    }
    if (lane == 31) warp_tmp[warp] = incl;
    __syncthreads();
    int woff = 0, total = 0;
    for (int w = 0; w < T / 32; ++w) { const int v = warp_tmp[w]; if (w < warp) woff += v; total += v; }
    int run = woff + incl - sum;
    for (int i = i0; i < i1; ++i) { const int v = a[i]; a[i] = run; run += v; }
    __syncthreads();
    return total;
}

// One Hoare partition (libstdc++ __unguarded_partition) by ONE WARP, as rank arithmetic (introsort_replay.h,
// unguarded_partition_ranked_, checked against std::sort on the host): ballots give every scan-stop position its rank from
// the left / from the right, swap k pairs the k-th stops while they have not crossed.  posL / posR: scratch indexed by
// absolute position (a range only touches its own span, so concurrent ranges never collide).
__device__ __forceinline__ int warp_partition_ranked(uint32_t* base, int first, int last, int pivot, uint32_t* posL, uint32_t* posR, int lane)
{
    const uint32_t pv = base[pivot];
    const uint32_t below = (1u << lane) - 1u;
    int nl = 0, nr = 0;
    for (int c = first; c < last; c += 32) {
        const int i = c + lane;
        const bool stop = i < last && !orbx_sort::lt(base[i], pv);
        const uint32_t mk = __ballot_sync(0xffffffffu, stop);
        if (stop) posL[first + nl + __popc(mk & below)] = (uint32_t)i;
        nl += __popc(mk);
    }
    for (int c = last - 1; c >= first; c -= 32) {
        const int i = c - lane;
        const bool stop = i >= first && !orbx_sort::lt(pv, base[i]);
        const uint32_t mk = __ballot_sync(0xffffffffu, stop);
        if (stop) posR[first + nr + __popc(mk & below)] = (uint32_t)i;
        nr += __popc(mk);
    }
    __syncwarp();
    const int nm = min(nl, nr);
    int K = 0;                                         // L_k < R_k is monotone in k: the pairs to swap form a prefix
    for (int c = 0; c < nm; c += 32) {
        const int k = c + lane;
        const bool ok = k < nm && posL[first + k] < posR[first + k];
        const uint32_t mk = __ballot_sync(0xffffffffu, ok);
        K += __popc(mk);
        if (mk != 0xffffffffu) break;                  // warp-uniform
    }
    for (int k = lane; k < K; k += 32) {
        const uint32_t l = posL[first + k], r = posR[first + k];
        const uint32_t x = base[l], y = base[r];
        base[l] = y; base[r] = x;
    }
    int ret = last;
    if (K < nl) ret = (int)posL[first + K];
    if (K > 0) ret = min(ret, (int)posR[first + K - 1]);
    __syncwarp();
    return ret;
}

// std::sort replay, range-parallel (introsort_replay.h): all T threads call.  base[m] = 32-bit items in shared memory,
// blk[m] / tmp[m] / aux[m] = shared scratch, q = 224 ints of shared scratch (three round counters + two queues of <= 32
// ranges: a range in a queue is longer than 16 elements and m <= 512).  Every range of a round is partitioned by its own
// warp (warp_partition_ranked).  One barrier per round: the counters rotate (the one read in round k is cleared in round
// k + 1 and refilled in round k + 2).
template <int T>
__device__ void sort_replay_parallel(uint32_t* base, int m, uint32_t* blk, uint32_t* tmp, uint32_t* aux, int* q)
{
    constexpr int NW = T / 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int* cnt = q;
    int* Q[2] = {q + 8, q + 8 + 96};
    if (m <= 16) {
        for (int i = tid; i < m; i += T) blk[i] = (uint32_t)m << 16;
    } else if (tid == 0) {
        Q[0][0] = 0; Q[0][1] = m; Q[0][2] = orbx_sort::initial_depth(m);
    }
    if (tid == 0) { cnt[0] = m > 16 ? 1 : 0; cnt[1] = 0; cnt[2] = 0; }
    __syncthreads();
    for (int round = 0;; ++round) {
        const int c = cnt[round % 3];
        if (c == 0) break;                                   // uniform
        if (tid == 0) cnt[(round + 2) % 3] = 0;
        int* nxt_cnt = cnt + (round + 1) % 3;
        const int* qi = Q[round & 1];
        int* qo = Q[(round + 1) & 1];
        for (int r = warp; r < c; r += NW) {
            const int first = qi[3 * r], last = qi[3 * r + 1], depth = qi[3 * r + 2];
            if (depth == 0) {                                // depth budget exhausted: heap sort (one lane), final
                if (lane == 0) orbx_sort::heap_sort_(base + first, last - first);
                for (int i = first + lane; i < last; i += 32) blk[i] = (uint32_t)i | ((uint32_t)(i + 1) << 16);
                __syncwarp();
                continue;
            }
            if (lane == 0)
                orbx_sort::move_median_to_first_(base + first, base + first + 1, base + first + (last - first) / 2, base + last - 1);
            __syncwarp();
            const int cut = warp_partition_ranked(base, first + 1, last, first, tmp, aux, lane);
            const int cf[2] = {first, cut}, cl[2] = {cut, last};
#pragma unroll
            for (int ch = 0; ch < 2; ++ch) {
                if (cl[ch] - cf[ch] > 16) {
                    if (lane == 0) {
                        const int slot = atomicAdd(nxt_cnt, 1);
                        qo[3 * slot] = cf[ch]; qo[3 * slot + 1] = cl[ch]; qo[3 * slot + 2] = depth - 1;
                    }
                } else {
                    const uint32_t bb = (uint32_t)cf[ch] | ((uint32_t)cl[ch] << 16);
                    for (int i = cf[ch] + lane; i < cl[ch]; i += 32) blk[i] = bb;
                }
            }
        }
        __syncthreads();
    }
    // __final_insertion_sort == stable sort of every leftover block: rank counting, one lane per element
    for (int i = tid; i < m; i += T) {
        const uint32_t b = blk[i];
        tmp[orbx_sort::block_stable_pos(base, (int)(b & 0xffffu), (int)(b >> 16), i)] = base[i];
    }
    __syncthreads();
    for (int i = tid; i < m; i += T) base[i] = tmp[i];
    __syncthreads();
}

// Leading part of a key's path code (window-relative x, y): root index, then 2 bits per depth for `levels` depths.
__device__ __forceinline__ uint32_t path_code_top(int x, int y, const LevelGeom& g, int winH, int levels)
{
    const int r = (int)__fdiv_rn((float)x, g.hX);                      // vpIniNodes[kp.pt.x / hX]   (src 613)
    int ulx = (int)__fmul_rn(g.hX, (float)r), urx = (int)__fmul_rn(g.hX, (float)(r + 1));   // src 602-603
    int uly = 0, bry = winH;
    uint32_t code = (uint32_t)r;
#pragma unroll 1
    for (int d = 0; d < levels; ++d) {
        const int mx = ulx + ((urx - ulx + 1) >> 1);                   // UL.x + ceil((UR.x-UL.x)/2)   (src 517)
        const int my = uly + ((bry - uly + 1) >> 1);
        const uint32_t qx = x >= mx, qy = y >= my;                     // src 546-557
        code = (code << 2) | qx | (qy << 1);
        if (qx) ulx = mx; else urx = mx;
        if (qy) uly = my; else bry = my;
    }
    return code;
}

// Exclusive prefix sum of a[0..n) in place by ONE warp (lane-strided chunks, running carry).  Returns the total.
__device__ __forceinline__ int warp_exclusive_scan(int* a, int n, int lane)
{
    int carry = 0;
    for (int base = 0; base < n; base += 32) {
        const int i = base + lane;
        const int v = i < n ? a[i] : 0;
        int incl = v;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += t;
        }
        if (i < n) a[i] = carry + incl - v;
        carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    return carry;
}

}  // namespace

// counting-sort depth of a level: as many leading code bits as fit kSortBitsMax
__host__ __device__ inline int octree_sort_depth(int depth, int root_bits)
{
    const int d = (kSortBitsMax - root_bits) / 2;
    return d < depth ? (d > 0 ? d : 0) : depth;
}

int octree_bins(const LevelGeom& g) { return 1 << (g.root_bits + 2 * octree_sort_depth(g.depth, g.root_bits)); }

size_t octree_smem_bytes(int M, int NB)
{
    size_t b = 0;
    b += sizeof(uint32_t) * (size_t)M * 10;     // node arrays x2
    b += sizeof(uint32_t) * (size_t)M * 4;      // cc
    b += sizeof(int) * (size_t)M * 5;           // sa, sb, sc, sd, procpos
    b += 8;                                     // alignment slack
    b += sizeof(unsigned long long) * (size_t)M * 2;
    const size_t cur = sizeof(int) * (size_t)NB;
    return sizeof(int) * (64 + 224) + sizeof(int) * ((size_t)NB + 2) + (b > cur ? b : cur);
}

// grid = (n_frames, levels of this launch); dynamic smem sized for the largest level's node capacity M and bin count NB.
#ifndef ORBX_OCT_THREADS_PER_SM
#define ORBX_OCT_THREADS_PER_SM 1024      // resident threads per SM the register budget is set for (64 registers)
#endif
template <int T>
__global__ void __launch_bounds__(T, ORBX_OCT_THREADS_PER_SM / T) octree_kernel(const __grid_constant__ FrameGeom fg, Workspace ws, int M, int NB,
                                                   int level_base, int* __restrict__ err_flag)
{
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_nL, s_nS, s_total;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    // level-major dispatch: the CTAs of level 0 (most candidates, longest) start first, the short deep levels pack the tail
    const int frame = blockIdx.x, level = level_base + blockIdx.y;
    const LevelGeom& g = fg.L[level];
    const int N = g.nfeat;
    // optional phase timing of one CTA (orbx_debug_octree_timing): dbg[0..6] cycles, dbg[7..] counters
    long long* dbg = (ws.dbg && frame == 0 && level == ws.dbg_level && tid == 0) ? ws.dbg : nullptr;
    long long t_prev = dbg ? clock64() : 0;
#define OCT_MARK(slot) do { if (dbg) { const long long t_now = clock64(); dbg[slot] += t_now - t_prev; t_prev = t_now; } } while (0)
    long long t_fine = t_prev;          // finer split of the first phase (slots 11..15), independent of the slots above
#define OCT_FINE(slot) do { if (dbg) { const long long t_now = clock64(); dbg[slot] += t_now - t_fine; t_fine = t_now; } } while (0)
    const int winW = g.w - 2 * kWinBorder, winH = g.h - 2 * kWinBorder;

    Smem S;
    {
        unsigned char* p = smem_raw;
        S.warp_tmp = (int*)p; p += sizeof(int) * 64;
        S.sort_stk = (int*)p; p += sizeof(int) * 224;
        S.bstart = (int*)p; p += sizeof(int) * ((size_t)NB + 2);
        S.cursor = (int*)p;             // aliases the arrays below: used by the counting sort only, which ends with a barrier
        for (int b = 0; b < 2; ++b) {
            S.nbeg[b] = (uint32_t*)p; p += 4 * (size_t)M;
            S.ncnt[b] = (uint32_t*)p; p += 4 * (size_t)M;
            S.nx[b] = (uint32_t*)p; p += 4 * (size_t)M;
            S.ndep[b] = (uint32_t*)p; p += 4 * (size_t)M;
            S.npre[b] = (uint32_t*)p; p += 4 * (size_t)M;
        }
        S.cc = (uint32_t*)p; p += 16 * (size_t)M;
        S.sa = (int*)p; p += 4 * (size_t)M;
        S.sb = (int*)p; p += 4 * (size_t)M;
        S.sc = (int*)p; p += 4 * (size_t)M;
        S.sd = (int*)p; p += 4 * (size_t)M;
        S.procpos = (int*)p; p += 4 * (size_t)M;
        p = (unsigned char*)(((uintptr_t)p + 7) & ~(uintptr_t)7);
        S.vec = (unsigned long long*)p; p += 8 * (size_t)M;
        S.vec2 = (unsigned long long*)p;
    }

    int* out_n = ws.lvl_n + (size_t)frame * fg.nlevels + level;
    int* out_ncand = ws.lvl_ncand + (size_t)frame * fg.nlevels + level;
    uint32_t* out_kp = ws.lvl_kp + (size_t)frame * fg.kp_slots + g.kp_base;

    const int ncells = g.nCols * g.nRows;
    if (ncells <= 0 || g.nIni <= 0 || winW <= 0 || winH <= 0) {
        if (tid == 0) { *out_n = 0; *out_ncand = 0; }
        return;
    }

    // ---- 0./1. counting sort of the level's candidates by the leading bits of their path codes -----------------------
    // A candidate's identity is its rank k in the reference's vToDistributeKeys order (cells row-major, (y, x) inside a cell):
    // k = (candidates in earlier cells) + slot, which is all the retain rule needs.  The passes are arranged so that a warp
    // waits for as few dependent global round trips as possible (the kernel is latency-bound): cell counts first (one trip),
    // then the candidates of eight cells per warp iteration (one trip each), then dense key-parallel passes.
    const int Dsort = octree_sort_depth(g.depth, g.root_bits);
    const int nb = 1 << (g.root_bits + 2 * Dsort);
    uint32_t* scratch = ws.oct + (size_t)frame * fg.oct_frame_stride + g.oct_off;
    const int nmax = g.cand_max;
    uint32_t* K = scratch;                                       // rank k | score << 24, bin-sorted
    uint32_t* K2 = scratch + nmax;                               // the packed candidate (x | y << 12 | score << 24), same order
    uint32_t* stash = scratch + 2 * (size_t)nmax;                // packed candidates in rank order
    uint32_t* binst = scratch + 3 * (size_t)nmax;                // their bins
    int* coff = (int*)(scratch + 5 * (size_t)nmax);              // [ncells] candidates in earlier cells
    const int* __restrict__ cell_count = ws.cell_count + (size_t)frame * fg.total_cells + g.cell_base;
    const uint32_t* __restrict__ cand = ws.cand + (size_t)frame * fg.cand_frame_stride + g.cand_off;
    for (int i = tid; i <= nb; i += T) S.bstart[i] = 0;
    for (int c = tid; c < ncells; c += T) coff[c] = __ldg(cell_count + c);
    __syncthreads();
    OCT_FINE(11);
    const int n = block_exclusive_scan_raking<T>(coff, ncells, S.warp_tmp);
    OCT_FINE(12);
    if (tid == 0) *out_ncand = n;
    if (n == 0) {
        if (tid == 0) *out_n = 0;
        return;
    }
    // gather: the candidates of eight cells per warp iteration, all loads of an iteration in flight together
    constexpr int GU = T >= 512 ? 2 : 8;          // cells per warp iteration (a big CTA has the warps instead of the unrolling)
    for (int c0 = warp * GU; c0 < ncells; c0 += (T / 32) * GU) {
        int cnt[GU], o[GU];
        uint32_t k[GU];
#pragma unroll
        for (int u = 0; u < GU; ++u) {
            const bool in = c0 + u < ncells;
            cnt[u] = in ? __ldg(cell_count + c0 + u) : 0;
            o[u] = in ? coff[c0 + u] : 0;
        }
#pragma unroll
        for (int u = 0; u < GU; ++u) k[u] = lane < cnt[u] ? cand[(size_t)(c0 + u) * g.cell_cap + lane] : 0u;
#pragma unroll
        for (int u = 0; u < GU; ++u) {
            if (lane < cnt[u]) stash[o[u] + lane] = k[u];
            for (int i = lane + 32; i < cnt[u]; i += 32) stash[o[u] + i] = cand[(size_t)(c0 + u) * g.cell_cap + i];   // > 32 candidates (rare)
        }
    }
    __syncthreads();
    OCT_FINE(13);
    // bins, dense over the keys (every lane busy).  Only the Dsort leading depths of the path are evaluated (the deeper bits
    // are needed by the rare splits below depth Dsort, which work them out on demand), once: binst carries the bin on.
    constexpr int KU = T >= 512 ? 1 : 4;          // keys per thread in flight
    for (int k0 = tid; k0 < n; k0 += KU * T) {
        uint32_t kk[KU];
#pragma unroll
        for (int u = 0; u < KU; ++u) kk[u] = k0 + u * T < n ? stash[k0 + u * T] : 0u;
#pragma unroll
        for (int u = 0; u < KU; ++u) {
            const int k = k0 + u * T;
            if (k < n) {
                const uint32_t bin = path_code_top((int)(kk[u] & 0xfff), (int)((kk[u] >> 12) & 0xfff), g, winH, Dsort);
                atomicAdd(&S.bstart[bin], 1);
                binst[k] = bin;
            }
        }
    }
    __syncthreads();
    OCT_FINE(14);
    block_exclusive_scan_raking<T>(S.bstart, nb, S.warp_tmp);
    OCT_FINE(15);
    if (tid == 0) S.bstart[nb] = n;
    for (int i = tid; i < nb; i += T) S.cursor[i] = S.bstart[i];
    __syncthreads();
    OCT_MARK(0);
    for (int k0 = tid; k0 < n; k0 += KU * T) {                   // dense: independent keys per thread in flight
        uint32_t kk[KU], bb[KU];
#pragma unroll
        for (int u = 0; u < KU; ++u) {
            const int k = k0 + u * T;
            kk[u] = k < n ? stash[k] : 0u;
            bb[u] = k < n ? binst[k] : 0u;
        }
#pragma unroll
        for (int u = 0; u < KU; ++u) {
            const int k = k0 + u * T;
            if (k < n) {
                const int pos = atomicAdd(&S.cursor[bb[u]], 1);
                K[pos] = (uint32_t)k | (kk[u] & 0xff000000u);
                K2[pos] = kk[u];
            }
        }
    }
    __syncthreads();            // the cursors are dead from here on: their bytes become the node arrays

    OCT_MARK(1);
    // ---- 2./3. the tree phases run in WARP 0 (a few hundred nodes: warp-wide scans and __syncwarp instead of CTA-wide
    // barriers); the other warps join for the std::sort replay and the final retain step. -------------------------------
    int a = 0;   // active node buffer (every thread tracks it)
    if (warp == 0) {
        if (lane == 0) {        // root nodes (src 589-626)
            int m = 0;
            for (int r = 0; r < g.nIni; ++r) {
                const int lo = S.bstart[r << (2 * Dsort)], hi = S.bstart[(r + 1) << (2 * Dsort)];
                if (hi > lo) {
                    S.nbeg[a][m] = (uint32_t)lo; S.ncnt[a][m] = (uint32_t)(hi - lo);
                    const int ulx = (int)__fmul_rn(g.hX, (float)r), urx = (int)__fmul_rn(g.hX, (float)(r + 1));
                    S.nx[a][m] = (uint32_t)ulx | ((uint32_t)urx << 16);
                    S.ndep[a][m] = 0;
                    S.npre[a][m] = (uint32_t)r;
                    ++m;
                }
            }
            s_nL = m;
        }
        __syncwarp();
    }

    // 2-bit quadrant of the key with payload `pl` at depth `dep` of its path (dep >= Dsort: not part of the sorted prefix)
    auto quadrant_at = [&](uint32_t kk, int dep) -> uint32_t {
        return path_code_top((int)(kk & 0xfff), (int)((kk >> 12) & 0xfff), g, winH, dep + 1) & 3u;
    };

    // Computes the children of the node at list position `pos` into cc[4*p..]; returns (#non-empty) | (#expandable << 8).
    auto split_counts = [&](int p, int pos) -> int {
        const uint32_t beg = S.nbeg[a][pos], cnt = S.ncnt[a][pos];
        const int dep = (int)S.ndep[a][pos];
        int ne = 0, nx = 0;
        if (dep >= g.depth) {           // cannot happen for distinct pixels (depth is sized for it); flag, keep the node whole
            atomicExch(err_flag, 1);
            S.cc[4 * p] = cnt; S.cc[4 * p + 1] = S.cc[4 * p + 2] = S.cc[4 * p + 3] = 0;
            return 1 | ((cnt > 1 ? 1 : 0) << 8);
        }
        const uint32_t e = beg + cnt;
        uint32_t b1, b2, b3;
        if (dep < Dsort) {
            // the children are runs of whole bins: their boundaries are entries of the scanned bin table
            const int sh = 2 * (Dsort - 1 - dep);
            const uint32_t base = S.npre[a][pos] << 2;
            b1 = (uint32_t)S.bstart[(base | 1u) << sh]; b2 = (uint32_t)S.bstart[(base | 2u) << sh]; b3 = (uint32_t)S.bstart[(base | 3u) << sh];
        } else {
            // below the sorted prefix: partition the (small) segment in place by the key's quadrant at this depth.  Order
            // inside a child is free, so an unstable American-flag pass does; re-partitioning an already partitioned segment
            // (a phase-2 split that was computed but cut off) is a no-op.
            uint32_t c4[4] = {0, 0, 0, 0};
            for (uint32_t i = beg; i < e; ++i) {
                const uint32_t d = quadrant_at(K2[i], dep);
                c4[0] += d == 0; c4[1] += d == 1; c4[2] += d == 2; c4[3] += d == 3;
            }
            b1 = beg + c4[0]; b2 = b1 + c4[1]; b3 = b2 + c4[2];
            uint32_t nx0 = beg, nx1 = b1, nx2 = b2, nx3 = b3;
            const uint32_t end0 = b1, end1 = b2, end2 = b3;
            auto place = [&](uint32_t i, uint32_t d) {     // swap element i with the head of bucket d, advance that head
                uint32_t& h = d == 0 ? nx0 : (d == 1 ? nx1 : (d == 2 ? nx2 : nx3));
                const uint32_t tk = K[i], tk2 = K2[i];
                K[i] = K[h]; K[h] = tk; K2[i] = K2[h]; K2[h] = tk2;
                ++h;
            };
            while (nx0 < end0) { const uint32_t d = quadrant_at(K2[nx0], dep); if (d == 0) ++nx0; else place(nx0, d); }
            while (nx1 < end1) { const uint32_t d = quadrant_at(K2[nx1], dep); if (d == 1) ++nx1; else place(nx1, d); }
            while (nx2 < end2) { const uint32_t d = quadrant_at(K2[nx2], dep); if (d == 2) ++nx2; else place(nx2, d); }
        }
        const uint32_t c0 = b1 - beg, c1 = b2 - b1, c2 = b3 - b2, c3 = e - b3;
        S.cc[4 * p] = c0; S.cc[4 * p + 1] = c1; S.cc[4 * p + 2] = c2; S.cc[4 * p + 3] = c3;
        ne = (c0 > 0) + (c1 > 0) + (c2 > 0) + (c3 > 0);
        nx = (c0 > 1) + (c1 > 1) + (c2 > 1) + (c3 > 1);
        return ne | (nx << 8);
    };

    // WARP 0.  Applies the splits of processed nodes p = 0..nS-1 (list positions procpos[p], child counts in cc, sa[p] =
    // #non-empty, sb[p] = #expandable), builds the new list in buffer a^1 and the new expandable vector in `vout`.
    // Publishes the new list size in s_nL and the new vector length in s_total.
    auto apply_splits = [&](int nL, int nS, unsigned long long* vout) {
        const int b = a ^ 1;
        for (int i = lane; i < nL; i += 32) S.sc[i] = 1;                       // keep flags: sc[pos] = 1 for untouched nodes
        __syncwarp();
        for (int p = lane; p < nS; p += 32) S.sc[S.procpos[p]] = 0;
        __syncwarp();
        const int nKeep = warp_exclusive_scan(S.sc, nL, lane);                 // sc[pos] = rank among kept (valid where kept)
        for (int p = lane; p < nS; p += 32) S.sc[S.procpos[p]] = -1;           // processed nodes are marked, not kept
        int* packed = S.sd;                                                    // ne/nx survive the scans of sa/sb here
        for (int p = lane; p < nS; p += 32) packed[p] = S.sa[p] | (S.sb[p] << 8);
        __syncwarp();
        const int Stot = warp_exclusive_scan(S.sa, nS, lane);                  // sa[p] = sum_{p'<p} ne
        const int Etot = warp_exclusive_scan(S.sb, nS, lane);                  // sb[p] = sum_{p'<p} nx
        for (int p = lane; p < nS; p += 32) {
            const int pos = S.procpos[p];
            const int ne = packed[p] & 0xff;
            const uint32_t beg = S.nbeg[a][pos];
            const uint32_t x = S.nx[a][pos];
            const int ulx = (int)(x & 0xffff), urx = (int)(x >> 16);
            const int mx = ulx + ((urx - ulx + 1) >> 1);
            const uint32_t dep = S.ndep[a][pos] + 1;
            const uint32_t pre4 = S.npre[a][pos] << 2;
            const uint32_t c0 = S.cc[4 * p], c1 = S.cc[4 * p + 1], c2 = S.cc[4 * p + 2], c3 = S.cc[4 * p + 3];
            const uint32_t cb[4] = {beg, beg + c0, beg + c0 + c1, beg + c0 + c1 + c2};
            const uint32_t cn[4] = {c0, c1, c2, c3};
            const uint32_t cx[4] = {(uint32_t)ulx | ((uint32_t)mx << 16), (uint32_t)mx | ((uint32_t)urx << 16),
                                    (uint32_t)ulx | ((uint32_t)mx << 16), (uint32_t)mx | ((uint32_t)urx << 16)};
            // group start: groups of later-processed nodes come first
            const int gstart = Stot - (S.sa[p] + ne);
            int slot = gstart, vslot = S.sb[p];
            int posk[4];
#pragma unroll
            for (int k = 3; k >= 0; --k) {            // list order inside the group: n4, n3, n2, n1
                posk[k] = -1;
                if (cn[k] > 0) {
                    S.nbeg[b][slot] = cb[k]; S.ncnt[b][slot] = cn[k]; S.nx[b][slot] = cx[k]; S.ndep[b][slot] = dep;
                    S.npre[b][slot] = pre4 | (uint32_t)k;
                    posk[k] = slot++;
                }
            }
#pragma unroll
            for (int k = 0; k < 4; ++k)               // creation order of vSizeAndPointerToNode: n1..n4 with > 1 key
                if (cn[k] > 1)
                    vout[vslot++] = orbx_sort::make_item(((unsigned long long)cn[k] << 13) | (cx[k] & 0xffff), (uint32_t)posk[k]);
        }
        for (int i = lane; i < nL; i += 32) {
            const int r = S.sc[i];
            if (r >= 0) {
                const int slot = Stot + r;
                S.nbeg[b][slot] = S.nbeg[a][i]; S.ncnt[b][slot] = S.ncnt[a][i]; S.nx[b][slot] = S.nx[a][i];
                S.ndep[b][slot] = S.ndep[a][i]; S.npre[b][slot] = S.npre[a][i];
            }
        }
        if (lane == 0) { s_nL = Stot + nKeep; s_total = Etot; }
        __syncwarp();
    };

    __syncthreads();
    OCT_MARK(2);
    // ---- 3. main loop (src 635-753) ---------------------------------------------------------------------------------
    // One loop body serves both kinds of rounds (one copy of the split / apply code: a single CTA per level is bound by
    // instruction fetch, so the kernel is kept small): a phase-1 sweep processes every expandable node in list order, a
    // phase-2 round processes the std::sort-ed expandable nodes from the back and stops at the split that reaches N.
    bool finish = false, phase2 = false;
    unsigned long long* vprev = S.vec;      // expandable nodes created by the previous round (creation order)
    unsigned long long* vnext = S.vec2;
    int nToExpand = 0;
    while (!finish) {
        const int prevSize = s_nL;
        if (dbg) { if (phase2) { dbg[8] += 1; if (nToExpand > dbg[10]) dbg[10] = nToExpand; } else dbg[7] += 1; }
        bool small = false;
        uint32_t* s32 = reinterpret_cast<uint32_t*>(S.sd);
        if (phase2) {
            // std::sort(compareNodes) (src 709).  For the usual few hundred nodes the replay runs on 32-bit items
            // (dense rank of (count, UL.x) << 16 | creation index): one shared-memory word per move/compare.
            const int m = nToExpand;
            small = m <= 512;
            if (small) {
                for (int i = tid; i < m; i += T) {
                    const unsigned long long ki = vprev[i] >> orbx_sort::kPayloadBits;
                    int rank = 0;
                    for (int j = 0; j < m; ++j) rank += (vprev[j] >> orbx_sort::kPayloadBits) < ki;
                    s32[i] = ((uint32_t)rank << 16) | (uint32_t)i;
                }
                __syncthreads();
                sort_replay_parallel<T>(s32, m, reinterpret_cast<uint32_t*>(S.sa), reinterpret_cast<uint32_t*>(S.sb),
                                        reinterpret_cast<uint32_t*>(S.sc), S.sort_stk);
            } else {
                if (tid == 0) orbx_sort::sort_replay(vprev, m);
            }
            __syncthreads();
            OCT_MARK(4);
        }
        if (warp == 0) {
            const int nL = prevSize;
            int nS;
            if (!phase2) {
                // every node with more than one key, in list order
                for (int i = lane; i < nL; i += 32) S.sc[i] = S.ncnt[a][i] > 1 ? 1 : 0;
                __syncwarp();
                nS = warp_exclusive_scan(S.sc, nL, lane);
                for (int i = lane; i < nL; i += 32)
                    if (S.ncnt[a][i] > 1) S.procpos[S.sc[i]] = i;
            } else {
                // processing order p = 0..m-1 walks the sorted vector from the back (src 710).  s32 lives in sd, which
                // apply_splits reuses: the positions are taken out first.
                nS = nToExpand;
                for (int p = lane; p < nS; p += 32)
                    S.procpos[p] = (int)orbx_sort::payload(small ? vprev[s32[nS - 1 - p] & 0xffffu] : vprev[nS - 1 - p]);
            }
            __syncwarp();
            for (int p = lane; p < nS; p += 32) {
                const int r = split_counts(p, S.procpos[p]);
                S.sa[p] = r & 0xff; S.sb[p] = r >> 8;
                S.sc[p] = (r & 0xff) - 1;                               // list growth of this split
            }
            __syncwarp();
            int cut = nS;
            if (phase2) {
                // cut-off: stop right after the first split that makes size >= N (src 745-746)
                warp_exclusive_scan(S.sc, nS, lane);                    // sc[p] = growth before p
                for (int p = lane; p < nS; p += 32) {
                    const int before = nL + S.sc[p];
                    const int after = before + (S.sa[p] - 1);
                    if (after >= N && before < N) cut = p + 1;          // at most one p satisfies this (growth >= 0)
                }
#pragma unroll
                for (int d = 16; d >= 1; d >>= 1) cut = min(cut, __shfl_xor_sync(0xffffffffu, cut, d));
            }
            apply_splits(nL, cut, vnext);
        }
        a ^= 1;
        __syncthreads();
        const int nL = s_nL;
        nToExpand = s_total;
        { unsigned long long* t = vprev; vprev = vnext; vnext = t; }
        OCT_MARK(phase2 ? 5 : 3);
        if (nL >= N || nL == prevSize) finish = true;                   // src 697-698, 751-752
        else if (!phase2 && nL + nToExpand * 3 > N) phase2 = true;      // src 699: the rest of the work is phase-2 rounds
    }

    // ---- 4. retain the best key per node, in list order (src 756-771) ------------------------------------------------
    // The segment is ordered by sub-path, not by original position, so "first key with maximal response" (src 758-768) = max
    // score, then min rank: the reduction runs on (score << 24 | 0xffffff - rank) << 32 | packed candidate, whose low word is
    // the answer — no dependent look-up.  Four nodes per warp iteration keep four independent loads in flight.
    const int nL = s_nL;
    constexpr int RU = T >= 512 ? 1 : 4;
    for (int i0 = warp * RU; i0 < nL; i0 += (T / 32) * RU) {
        unsigned long long best[RU];
#pragma unroll
        for (int u = 0; u < RU; ++u) {
            best[u] = 0ull;
            const int i = i0 + u;
            if (i < nL) {
                const uint32_t beg = S.nbeg[a][i], cnt = S.ncnt[a][i];
                for (uint32_t j = lane; j < cnt; j += 32) {
                    const uint32_t pl = K[beg + j], kk = K2[beg + j];
                    const unsigned long long v = ((unsigned long long)((pl & 0xff000000u) | (0xffffffu - (pl & 0xffffffu))) << 32) | kk;
                    best[u] = v > best[u] ? v : best[u];
                }
            }
        }
#pragma unroll
        for (int u = 0; u < RU; ++u) {
#pragma unroll
            for (int d = 16; d >= 1; d >>= 1) {
                const unsigned long long o = __shfl_xor_sync(0xffffffffu, best[u], d);
                best[u] = o > best[u] ? o : best[u];
            }
            if (lane == 0 && i0 + u < nL) out_kp[i0 + u] = (uint32_t)best[u];
        }
    }
    if (tid == 0) *out_n = nL;
    OCT_MARK(6);
    if (dbg) dbg[9] = n;
#undef OCT_MARK
#undef OCT_FINE
}

cudaError_t octree_prepare()
{
    cudaError_t e = cudaFuncSetAttribute(octree_kernel<256>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(octree_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
}

size_t octree_smem_for(const FrameGeom& fg, int level_lo, int level_hi)
{
    int M = 1, NB = 1;
    for (int l = level_lo; l < level_hi; ++l) {
        M = M > fg.L[l].kp_cap ? M : fg.L[l].kp_cap;
        const int nb = octree_bins(fg.L[l]);
        NB = NB > nb ? NB : nb;
    }
    return octree_smem_bytes(M, NB);
}

static int* g_err_flag[64] = {nullptr};

// The depth-overflow flag of the last octree launches on the current device (set when two candidates share a pixel: the
// quadtree cannot separate them); reading clears it.  Synchronises the device: test / stand-alone entry points only.
int octree_take_error_flag()
{
    int dev = 0;
    cudaGetDevice(&dev);
    int* p = g_err_flag[dev & 63];
    if (!p) return 0;
    int v = 0;
    if (cudaMemcpy(&v, p, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
    if (v) cudaMemset(p, 0, sizeof(int));
    return v;
}

// Levels [level_lo, level_hi) of n_frames frames (level_hi <= 0: all levels).
cudaError_t launch_octree(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st, int level_lo, int level_hi)
{
    if (level_hi <= 0) level_hi = fg.nlevels;
    if (level_lo >= level_hi) return cudaSuccess;
    int M = 1, NB = 1;
    for (int l = level_lo; l < level_hi; ++l) {
        M = M > fg.L[l].kp_cap ? M : fg.L[l].kp_cap;
        const int nb = octree_bins(fg.L[l]);
        NB = NB > nb ? NB : nb;
    }
    // Batches: 256-thread CTAs (measured on 512-frame batches: 128 threads +7 %, 64 threads +36 %, 512 threads ~30 % slower:
    // the parallel phases need the lanes, the single-lane parts need many resident CTAs).
    // A few frames: the level-0 CTA is the critical path of the whole extraction, so give it more lanes.
    const size_t smem = octree_smem_bytes(M, NB);
    if (smem > 200 * 1024) return cudaErrorInvalidConfiguration;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!g_err_flag[dev & 63]) {
        static std::mutex mu;
        std::lock_guard<std::mutex> lock(mu);
        if (!g_err_flag[dev & 63]) {
            int* p = nullptr;
            cudaError_t e = cudaMalloc(&p, sizeof(int));
            if (e != cudaSuccess) return e;
            cudaMemset(p, 0, sizeof(int));
            g_err_flag[dev & 63] = p;
        }
    }
    dim3 grid(n_frames, level_hi - level_lo);
    if (n_frames >= 8) octree_kernel<256><<<grid, 256, smem, st>>>(fg, ws, M, NB, level_lo, g_err_flag[dev & 63]);
    else octree_kernel<1024><<<grid, 1024, smem, st>>>(fg, ws, M, NB, level_lo, g_err_flag[dev & 63]);
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
