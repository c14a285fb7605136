// kernels_proj.cu — the 64x48 frame grid and the projection-guided window searches of ORBmatcher (SURVEY.md §8(f)2).
//
// Reference semantics reproduced (paths relative to the reference root):
//   * Frame::AssignFeaturesToGrid src/Frame.cc:387-418, Frame::PosInGrid :755-766: feature -> cell (round((x - minX) * wInv), ...).
//   * Frame::GetFeaturesInArea src/Frame.cc:687-753: candidates of a window in the order cell column ix, cell row iy, then the
//     cell's push_back order (= ascending feature index).
//   * ORBmatcher::SearchByProjection(Frame, MapPoints) src/ORBmatcher1.cc:45-215: best / second-best Hamming distance with strict
//     '<' over that order, level-aware ratio test, TH_HIGH.
//   * SearchByProjection(Current, Last) src/ORBmatcher3.cc:256-467 and (Current, KeyFrame) :469-578: 1-NN under a threshold.
//   All three skip features that already hold an observed map point, INCLUDING the ones assigned by earlier queries of the same
//   call — a sequential dependence between queries whose windows overlap.
//
// GPU formulation.  The scan's (best, second) pair equals the two least keys (distance, cell id, feature index): strict '<'
// keeps the earliest candidate of a distance, and bestLevel2 is the level of the earliest candidate that reaches the final
// second-best distance (worked out in DESIGN.md §5b).  So a warp scans a window with lanes across the candidates and reduces a
// top-2 of 64-bit keys; no candidate list is ever materialised or ordered.
// The dependence is resolved by deterministic speculation in rounds: every unresolved query computes its top-2 on the current
// "taken" state and CLAIMS (atomicMin of its index) every candidate it could ever take (distance <= threshold).  A query is
// final when no earlier unresolved query claims its best (and, for the ratio test, its second-best) candidate: nothing that
// is still undecided can change what it sees.  The least unresolved index is always final, so the loop terminates; real
// frames resolve in 2-3 rounds because only near-matches (distance <= TH_HIGH) claim.
// Queries are decided out of order, so "taken" is versioned: taken_by[f] holds the index of the query that took f (-1 = occupied
// on entry) and query q treats f as taken only if taken_by[f] < q — a later query's assignment must stay invisible to an earlier,
// still undecided one (it may be that query's second-best candidate, which feeds the ratio test).  An earlier query can never
// take the same feature afterwards: it would have claimed it, and the later query would not have been final.
//
// Mode 2 = ORBmatcher::SearchForInitialization src/ORBmatcher1.cc:650-765: one query per level-0 feature of F1, a feature of F2
// is skipped when vMatchedDistance[f] <= dist, i.e. when an earlier query accepted it at a distance no larger.  Acceptances of
// one feature happen in query order (the earlier acceptor claims f until it is decided), so they form a chain per feature,
// newest first: last_acc[f] -> prev_acc[q] -> ...; query q reads vMatchedDistance[f] as the acc_dist of the first acceptor
// below q on that chain (DESIGN.md §5b).
//
// ORBmatcher::Fuse src/ORBmatcher2.cc:420-610 (fuse_grid_kernel, fuse_scan_kernel): the candidate loop never reads the key
// frame's map points, so every (key frame, point) pair is independent — one wide launch, no rounds (DESIGN.md §5b).  The Sim3
// Fuse of loop closing (src/ORBmatcher2.cc:612-729) is the same loop without the reprojection gate (fuse_scan_kernel<false>);
// the Sim3 SearchByProjection (src/ORBmatcher1.cc:429-648) is mode 1 above.
#include <climits>

#include "orbx_internal.cuh"

namespace orbx {

namespace {

constexpr int GRID_COLS = ORBX_FRAME_GRID_COLS, GRID_ROWS = ORBX_FRAME_GRID_ROWS, GRID_CELLS = GRID_COLS * GRID_ROWS;
constexpr unsigned long long KEY_NONE = ~0ull;

__device__ __forceinline__ void load_desc(const uint8_t* __restrict__ base, size_t row, uint32_t d[8])
{
    const uint4* p = reinterpret_cast<const uint4*>(base + row * 32);
    const uint4 a = __ldg(p), b = __ldg(p + 1);
    d[0] = a.x; d[1] = a.y; d[2] = a.z; d[3] = a.w; d[4] = b.x; d[5] = b.y; d[6] = b.z; d[7] = b.w;
}
__device__ __forceinline__ int hamming256(const uint32_t a[8], const uint32_t b[8])
{
    int d = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) d += __popc(a[i] ^ b[i]);
    return d;
}

__device__ __forceinline__ void top2_push(unsigned long long& k1, unsigned long long& k2, unsigned long long k)
{
    if (k < k1) { k2 = k1; k1 = k; }
    else if (k < k2) k2 = k;
}
__device__ __forceinline__ void top2_warp_reduce(unsigned long long& k1, unsigned long long& k2)
{
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const unsigned long long o1 = __shfl_xor_sync(0xffffffffu, k1, s), o2 = __shfl_xor_sync(0xffffffffu, k2, s);
        top2_push(k1, k2, o1);
        top2_push(k1, k2, o2);
    }
}

// PosInGrid (src/Frame.cc:755-766): -1 when the rounded position falls outside the grid.
__device__ __forceinline__ int cell_of_point(const ProjArgs& a, float x, float y)
{
    const float px = roundf(__fmul_rn(__fsub_rn(x, a.min_x), a.grid_w_inv));
    const float py = roundf(__fmul_rn(__fsub_rn(y, a.min_y), a.grid_h_inv));
    if (!(px >= 0.0f && px < (float)GRID_COLS && py >= 0.0f && py < (float)GRID_ROWS)) return -1;
    return (int)px * GRID_ROWS + (int)py;
}

struct Window { int x0, x1, y0, y1; };     // cell range of GetFeaturesInArea; x0 > x1 = empty
__device__ __forceinline__ Window window_cells(const ProjArgs& a, float x, float y, float r)
{
    Window w;
    // src/Frame.cc:695-717, evaluated in float exactly as written: ((x - minX) -/+ r) * inv, floor / ceil, clamp
    const float dx = __fsub_rn(x, a.min_x), dy = __fsub_rn(y, a.min_y);
    w.x0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(dx, r), a.grid_w_inv)));
    w.x1 = min(GRID_COLS - 1, (int)ceilf(__fmul_rn(__fadd_rn(dx, r), a.grid_w_inv)));
    w.y0 = max(0, (int)floorf(__fmul_rn(__fsub_rn(dy, r), a.grid_h_inv)));
    w.y1 = min(GRID_ROWS - 1, (int)ceilf(__fmul_rn(__fadd_rn(dy, r), a.grid_h_inv)));
    if (w.x0 >= GRID_COLS || w.x1 < 0 || w.y0 >= GRID_ROWS || w.y1 < 0) { w.x0 = 1; w.x1 = 0; }
    return w;
}

// Is feature idx a member of GetFeaturesInArea(x, y, r, minLevel, maxLevel)?  (level and box tests, src/Frame.cc:733-747)
__device__ __forceinline__ bool in_area(const ProjArgs& a, int idx, float x, float y, float r, int min_level, int max_level)
{
    const orbx_keypoint* kp = a.kp + idx;
    if (min_level > 0 || max_level >= 0) {
        const int oct = __ldg(&kp->octave);
        if (oct < min_level) return false;
        if (max_level >= 0 && oct > max_level) return false;
    }
    const float distx = __fsub_rn(__ldg(&kp->x), x), disty = __fsub_rn(__ldg(&kp->y), y);
    return fabsf(distx) < r && fabsf(disty) < r;
}

// vMatchedDistance[f] as query qi sees it (mode 2): the distance of the latest acceptance of f by a query below qi, INT_MAX if
// none.  The chain is newest first and its distances strictly fall from at most TH_LOW, so the walk is short.
__device__ __forceinline__ int matched_distance(const ProjArgs& a, int f, int qi)
{
    int p = __ldcg(a.last_acc + f);
    while (p >= qi) p = __ldcg(a.prev_acc + p);
    return p < 0 ? INT_MAX : __ldcg(a.acc_dist + p);
}

// One warp evaluates one query on the current taken[] state: top-2 keys over its window, and (claim) atomicMin of the query
// index on every candidate within the distance threshold.
__device__ void scan_query(const ProjArgs& a, int qi, int lane, unsigned long long& k1, unsigned long long& k2)
{
    const ProjQuery q = a.q[qi];
    k1 = k2 = KEY_NONE;
    const Window w = window_cells(a, q.x, q.y, q.r);
    uint32_t qd[8];
    load_desc(a.qdesc, (size_t)qi, qd);
    const bool check_right = (q.flags & PROJ_Q_CHECK_RIGHT) && a.u_right;
    const bool init = a.mode == 2;
    for (int ix = w.x0; ix <= w.x1; ++ix) {
        // cells (ix, y0..y1) are consecutive cell ids: one contiguous item range per grid column
        const int t0 = __ldg(a.cell_start + ix * GRID_ROWS + w.y0), t1 = __ldg(a.cell_start + ix * GRID_ROWS + w.y1 + 1);
        for (int t = t0 + lane; t < t1; t += 32) {
            const int idx = __ldg(a.items + t);
            if (!in_area(a, idx, q.x, q.y, q.r, q.min_level, q.max_level)) continue;
            if (!init && __ldcg(a.taken_by + idx) < qi) continue;          // mvpMapPoints[idx] with Observations() > 0, as query qi sees it
            if (check_right) {                                             // src/ORBmatcher1.cc:95-100, ORBmatcher3.cc:330-336
                const float ur = __ldg(a.u_right + idx);
                if (ur > 0.0f && fabsf(__fsub_rn(q.ur, ur)) > q.r) continue;
            }
            uint32_t d[8];
            load_desc(a.desc, (size_t)idx, d);
            const int dist = hamming256(qd, d);
            if (init && matched_distance(a, idx, qi) <= dist) continue;    // vMatchedDistance[i2] <= dist, before the top-2 update
            top2_push(k1, k2, ((unsigned long long)dist << 48) | ((unsigned long long)__ldg(a.cell_of + idx) << 32) | (unsigned)idx);
            if (dist <= a.th_dist) atomicMin(a.claim + idx, qi);
        }
    }
    top2_warp_reduce(k1, k2);
}

// Decide query qi from its stored keys; returns false if an earlier undecided query may still change what it sees.
__device__ bool decide_query(const ProjArgs& a, int qi)
{
    const unsigned long long k1 = __ldcg(a.keys + 2 * qi), k2 = __ldcg(a.keys + 2 * qi + 1);
    if (k1 == KEY_NONE) return true;                                       // empty window
    const int d1 = (int)(k1 >> 48), f1 = (int)(unsigned)k1;
    if (d1 > a.th_dist) return true;                                       // taking candidates away can only raise the best distance
    if (__ldcg(a.claim + f1) < qi) return false;                           // L2 reads: the claims are L2 atomics
    if (a.mode == 2) {
        // src/ORBmatcher1.cc:650-765: bestDist2 starts at INT_MAX, so a candidate at 256 is a real second-best and a query
        // without one always passes 'bestDist < (float)bestDist2 * mfNNratio'
        const int f2 = k2 == KEY_NONE ? -1 : (int)(unsigned)k2;
        if (f2 >= 0 && __ldcg(a.claim + f2) < qi) return false;
        const int d2 = f2 >= 0 ? (int)(k2 >> 48) : INT_MAX;
        if (!((float)d1 < __fmul_rn((float)d2, a.nn_ratio))) return true;
        // at most one query accepts a feature per decide phase (an earlier acceptor claims it until it is decided)
        __stcg(a.prev_acc + qi, __ldcg(a.last_acc + f1));
        __stcg(a.acc_dist + qi, d1);
        __stcg(a.last_acc + f1, qi);
        a.qmatch[qi] = f1;
        return true;
    }
    const int f2 = (k2 >> 48) >= 256 ? -1 : (int)(unsigned)k2;            // 'dist < bestDist2' never fires for 256: no second-best
    if (a.mode == 0) {
        if (f2 >= 0 && __ldcg(a.claim + f2) < qi) return false;
        // src/ORBmatcher1.cc:125-131: reject when best and second sit on one level and bestDist > mfNNratio * bestDist2
        const int l1 = a.kp[f1].octave, l2 = f2 >= 0 ? a.kp[f2].octave : -1, d2 = f2 >= 0 ? (int)(k2 >> 48) : 256;
        if (l1 == l2 && (float)d1 > __fmul_rn(a.nn_ratio, (float)d2)) return true;
    }
    a.qmatch[qi] = f1;
    if (a.q[qi].flags & PROJ_Q_TAKES) __stcg(a.taken_by + f1, qi);
    return true;
}

// ---- grid build: one CTA per frame, counting sort by cell id (ix * 48 + iy), in-cell order = ascending feature index --------
// Reads a.n, a.kp, the grid geometry; writes a.cell_of, a.cell_start, a.items.  Every thread of the CTA calls it.
__device__ void build_grid(const ProjArgs& a, int* s_cnt, int* s_part)
{
    const int tid = threadIdx.x;
    for (int c = tid; c < GRID_CELLS; c += 1024) s_cnt[c] = 0;
    __syncthreads();
    for (int i = tid; i < a.n; i += 1024) {
        const int c = cell_of_point(a, a.kp[i].x, a.kp[i].y);
        a.cell_of[i] = (unsigned short)(c < 0 ? 0xffff : c);
        if (c >= 0) atomicAdd(&s_cnt[c], 1);
    }
    __syncthreads();
    // exclusive scan of 3072 counters: 3 per thread + block scan of the partial sums
    const int c0 = s_cnt[3 * tid], c1 = s_cnt[3 * tid + 1], c2 = s_cnt[3 * tid + 2];
    s_part[tid] = c0 + c1 + c2;
    __syncthreads();
    for (int s = 1; s < 1024; s <<= 1) {
        const int v = tid >= s ? s_part[tid - s] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    const int base = s_part[tid] - (c0 + c1 + c2);
    a.cell_start[3 * tid] = base; a.cell_start[3 * tid + 1] = base + c0; a.cell_start[3 * tid + 2] = base + c0 + c1;
    if (tid == 1023) a.cell_start[GRID_CELLS] = s_part[1023];
    s_cnt[3 * tid] = base; s_cnt[3 * tid + 1] = base + c0; s_cnt[3 * tid + 2] = base + c0 + c1;      // scatter cursors
    __syncthreads();
    for (int i = tid; i < a.n; i += 1024) {
        const int c = a.cell_of[i];
        if (c != 0xffff) a.items[atomicAdd(&s_cnt[c], 1)] = i;
    }
    __syncthreads();
    // cells hold a handful of features: insertion sort per cell restores the push_back (ascending index) order
    for (int c = tid; c < GRID_CELLS; c += 1024) {
        const int b = a.cell_start[c], e = s_cnt[c];
        for (int i = b + 1; i < e; ++i) {
            const int v = a.items[i];
            int j = i - 1;
            while (j >= b && a.items[j] > v) { a.items[j + 1] = a.items[j]; --j; }
            a.items[j + 1] = v;
        }
    }
}

// The fields of ProjArgs that build_grid / window_cells / in_area read, for one key frame of orbx_fuse.
__device__ __forceinline__ ProjArgs kf_args(const FuseKF& k)
{
    ProjArgs a{};
    a.n = k.n; a.kp = k.kp; a.desc = k.desc; a.u_right = k.u_right;
    a.min_x = k.min_x; a.min_y = k.min_y; a.grid_w_inv = k.grid_w_inv; a.grid_h_inv = k.grid_h_inv;
    a.cell_start = k.cell_start; a.items = k.items; a.cell_of = k.cell_of;
    return a;
}

}  // namespace

__global__ void __launch_bounds__(1024) frame_grid_kernel(ProjArgs a)
{
    __shared__ int s_cnt[GRID_CELLS];
    __shared__ int s_part[1024];
    for (int i = threadIdx.x; i < a.n; i += 1024) {
        a.claim[i] = INT_MAX;
        if (a.last_acc) a.last_acc[i] = -1;
    }
    build_grid(a, s_cnt, s_part);
}

// ---- orbx_fuse: the grids of all key frames of the call in one launch, one CTA per key frame ------------------------------
__global__ void __launch_bounds__(1024) fuse_grid_kernel(FuseArgs f)
{
    __shared__ int s_cnt[GRID_CELLS];
    __shared__ int s_part[1024];
    build_grid(kf_args(f.kfs[blockIdx.x]), s_cnt, s_part);
}

// ---- ORBmatcher::Fuse (src/ORBmatcher2.cc:420-610), the candidate loop: one warp per (key frame, point) pair -----------------
// The loop never reads the key frame's map points, so every pair is independent.  KeyFrame::GetFeaturesInArea is the window of
// Frame::GetFeaturesInArea without levels; the level gate [level - 1, level] comes first in the loop, so it is folded into the
// window's membership test.  The least key (distance, cell id, index) is the earliest candidate at the least distance, which is
// what strict '<' keeps.  kReprojGate = false is the Sim3 Fuse (src/ORBmatcher2.cc:612-729): no reprojection gate, so neither
// inv_sigma2 nor u_right is read (its bestDist starts at INT_MAX instead of 256, which changes nothing under TH_LOW).
template <bool kReprojGate>
__global__ void __launch_bounds__(256) fuse_scan_kernel(FuseArgs f)
{
    const int lane = threadIdx.x & 31;
    const int qi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qi >= f.nq) return;
    const FuseQuery q = f.q[qi];
    const FuseKF& K = f.kfs[q.kf];
    const ProjArgs a = kf_args(K);
    const Window w = window_cells(a, q.u, q.v, q.r);
    uint32_t qd[8];
    load_desc(f.pdesc, (size_t)q.point, qd);
    unsigned long long k1 = KEY_NONE;
    for (int ix = w.x0; ix <= w.x1; ++ix) {
        const int t0 = __ldg(a.cell_start + ix * GRID_ROWS + w.y0), t1 = __ldg(a.cell_start + ix * GRID_ROWS + w.y1 + 1);
        for (int t = t0 + lane; t < t1; t += 32) {
            const int idx = __ldg(a.items + t);
            // kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel (an octave of -1 would index mvInvLevelSigma2[-1])
            if (!in_area(a, idx, q.u, q.v, q.r, max(q.level - 1, 0), q.level)) continue;
            if constexpr (kReprojGate) {
                const orbx_keypoint* kp = a.kp + idx;
                const int oct = __ldg(&kp->octave);
                const float inv = K.inv_sigma2[oct];
                const float ex = __fsub_rn(q.u, __ldg(&kp->x)), ey = __fsub_rn(q.v, __ldg(&kp->y));
                const float kpr = a.u_right ? __ldg(a.u_right + idx) : -1.0f;
                // float e2, every product and sum rounded; 'e2 * inv' rounded to float, then compared with the double constant
                if (kpr >= 0.0f) {
                    const float er = __fsub_rn(q.ur, kpr);
                    const float e2 = __fadd_rn(__fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey)), __fmul_rn(er, er));
                    if ((double)__fmul_rn(e2, inv) > 7.8) continue;
                } else {
                    const float e2 = __fadd_rn(__fmul_rn(ex, ex), __fmul_rn(ey, ey));
                    if ((double)__fmul_rn(e2, inv) > 5.99) continue;
                }
            }
            uint32_t d[8];
            load_desc(a.desc, (size_t)idx, d);
            const unsigned long long key =
                ((unsigned long long)hamming256(qd, d) << 48) | ((unsigned long long)__ldg(a.cell_of + idx) << 32) | (unsigned)idx;
            if (key < k1) k1 = key;
        }
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
        const unsigned long long o = __shfl_xor_sync(0xffffffffu, k1, s);
        if (o < k1) k1 = o;
    }
    if (lane == 0) f.match[qi] = (k1 != KEY_NONE && (int)(k1 >> 48) <= f.th_dist) ? (int)(unsigned)k1 : -1;
}

// ---- round 0, wide: every valid query scans and claims on the initial state -------------------------------------------------
__global__ void __launch_bounds__(256) proj_scan_kernel(ProjArgs a)
{
    const int lane = threadIdx.x & 31;
    const int qi = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (qi >= a.nq) return;
    if (!(a.q[qi].flags & PROJ_Q_VALID)) return;
    unsigned long long k1, k2;
    scan_query(a, qi, lane, k1, k2);
    if (lane == 0) { __stcg(a.keys + 2 * qi, k1); __stcg(a.keys + 2 * qi + 1, k2); }
}

// ---- resolution: one CTA decides what it can, re-scans the rest on the updated state, until nothing is left ----------------
__global__ void __launch_bounds__(1024) proj_resolve_kernel(ProjArgs a)
{
    __shared__ int s_n[2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int* cur = a.list_a;
    int* nxt = a.list_b;
    // round 0 list = all valid queries (order is irrelevant)
    if (tid == 0) { s_n[0] = 0; s_n[1] = 0; }
    __syncthreads();
    for (int i = tid; i < a.nq; i += 1024)
        if (a.q[i].flags & PROJ_Q_VALID) cur[atomicAdd(&s_n[0], 1)] = i;
    __syncthreads();
    int sel = 0, rounds = 0;
    for (;;) {
        const int n_cur = s_n[sel];
        if (n_cur == 0) break;
        for (int t = tid; t < n_cur; t += 1024) {
            const int qi = cur[t];
            if (!decide_query(a, qi)) nxt[atomicAdd(&s_n[sel ^ 1], 1)] = qi;
        }
        __syncthreads();
        const int n_nxt = s_n[sel ^ 1];
        if (tid == 0) s_n[sel] = 0;
        for (int i = tid; i < a.n; i += 1024) __stcg(a.claim + i, INT_MAX);
        __syncthreads();
        for (int t = warp; t < n_nxt; t += 32) {
            const int qi = nxt[t];
            unsigned long long k1, k2;
            scan_query(a, qi, lane, k1, k2);
            if (lane == 0) { __stcg(a.keys + 2 * qi, k1); __stcg(a.keys + 2 * qi + 1, k2); }
        }
        __syncthreads();
        int* tmp = cur; cur = nxt; nxt = tmp;
        sel ^= 1;
        ++rounds;
    }
    if (tid == 0 && a.rounds_out) *a.rounds_out = rounds;
}

// ---- GetFeaturesInArea as a standalone query (tests, adapter): unordered (cell, index) keys, the host orders them ----------
__global__ void __launch_bounds__(256) features_in_area_kernel(ProjArgs a, float x, float y, float r, int min_level, int max_level,
                                                               unsigned long long* out, int capacity, int* n_out)
{
    const Window w = window_cells(a, x, y, r);
    for (int ix = w.x0; ix <= w.x1; ++ix) {
        const int t0 = a.cell_start[ix * GRID_ROWS + w.y0], t1 = a.cell_start[ix * GRID_ROWS + w.y1 + 1];
        for (int t = t0 + threadIdx.x; t < t1; t += blockDim.x) {
            const int idx = a.items[t];
            if (!in_area(a, idx, x, y, r, min_level, max_level)) continue;
            const int slot = atomicAdd(n_out, 1);
            if (slot < capacity) out[slot] = ((unsigned long long)a.cell_of[idx] << 32) | (unsigned)idx;
        }
    }
}

cudaError_t launch_frame_grid(const ProjArgs& a, cudaStream_t st)
{
    frame_grid_kernel<<<1, 1024, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

cudaError_t launch_proj_search(const ProjArgs& a, cudaStream_t st)
{
    if (a.nq <= 0) return cudaSuccess;
    proj_scan_kernel<<<(a.nq + 7) / 8, 256, 0, st>>>(a);
    proj_resolve_kernel<<<1, 1024, 0, st>>>(a);
    count_launch(2);
    return cudaGetLastError();
}

cudaError_t launch_fuse(const FuseArgs& a, bool reproj_gate, cudaStream_t st)
{
    if (a.n_kf > 0) fuse_grid_kernel<<<a.n_kf, 1024, 0, st>>>(a);
    if (a.nq > 0) {
        if (reproj_gate) fuse_scan_kernel<true><<<(a.nq + 7) / 8, 256, 0, st>>>(a);
        else fuse_scan_kernel<false><<<(a.nq + 7) / 8, 256, 0, st>>>(a);
    }
    count_launch((a.n_kf > 0) + (a.nq > 0));
    return cudaGetLastError();
}

cudaError_t launch_features_in_area(const ProjArgs& a, float x, float y, float r, int min_level, int max_level,
                                    unsigned long long* d_out, int capacity, int* d_n_out, cudaStream_t st)
{
    features_in_area_kernel<<<1, 256, 0, st>>>(a, x, y, r, min_level, max_level, d_out, capacity, d_n_out);
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
