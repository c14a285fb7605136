// kernels_match.cu — Hamming matching on the integer pipe (LOP3 + POPC), never tensor cores.
//
//  * knn2_kernel:        brute-force 2-NN (cv::BFMatcher(NORM_HAMMING).knnMatch(k=2), reference src/Frame.cc:1174; same
//                        (d1,i1,d2) as the strict-'<' best/second scans of src/ORBmatcher1.cc:283-300 and
//                        src/ORBmatcher2.cc:84-118).  DescriptorDistance (src/ORBmatcher3.cc:637-653) = 8 x (XOR, POPC).
//  * knn2_merge_kernel:  lexicographic (distance, index) merge of per-chunk / per-shard candidates.
//  * stereo kernels:     Frame::ComputeStereoMatches (src/Frame.cc:841-1011).
//  * popc_bench_kernel:  POPC issue-rate microbenchmark (roofline denominator for the matcher).
#include <limits.h>
#include <stdlib.h>

#include "orbx_internal.cuh"
#include "synth.h"

namespace orbx {

namespace {

constexpr int KNN_THREADS = 128;
constexpr int KNN_QT = 4;                       // queries per thread (8 was measured 11 % slower: 145 registers)
constexpr int KNN_QTILE = KNN_THREADS * KNN_QT; // queries per CTA
constexpr int KNN_DTILE = 256;                  // database rows staged per shared-memory tile (8 KB)

// Out of line on purpose: after the first few thousand rows an update is rare, so the hot loop should pay one compare and
// one (not-taken) branch per distance — inlined, the compiler if-converts this into six ALU-pipe instructions per compare,
// and the ALU pipe is the bound of the matcher.
__device__ __noinline__ int4 top2_insert(int dist, int idx, int4 s)      // s = (d1, i1, d2, i2), by value: stays in registers
{
    if (dist < s.x) return make_int4(dist, idx, s.x, s.y);
    return make_int4(s.x, s.y, dist, idx);
}
__device__ __forceinline__ void top2_update(int dist, int idx, int& d1, int& i1, int& d2, int& i2)
{
    if (dist < d2) {
        const int4 r = top2_insert(dist, idx, make_int4(d1, i1, d2, i2));
        d1 = r.x; i1 = r.y; d2 = r.z; i2 = r.w;
    }
}

// 256-bit Hamming distance with a carry-save front end.  POPC issues at 16 lanes/clk/SM (a quarter of LOP3), so the plain
// 8 x (XOR, POPC) form is POPC-bound at 0.5 clk per compare per SM.  Three full-adder layers (each 2 LOP3) compress the
// eight XOR words to four population counts of weight 1,1,2,4:
//     (c1,s1)=CSA(x0,x1,x2) (c2,s2)=CSA(x3,x4,x5) (c3,s3)=CSA(s1,s2,x6) (d1,t1)=CSA(c1,c2,c3)
//     dist = popc(s3) + popc(x7) + 2*popc(t1) + 4*popc(d1)
// 16 LOP3 + 4 POPC per compare balances the ALU pipe (0.27 clk) against the POPC pipe (0.25 clk).
__device__ __forceinline__ uint32_t lop3_xor3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t lop3_maj(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ void csa(uint32_t a, uint32_t b, uint32_t c, uint32_t& carry, uint32_t& sum)
{
    sum = lop3_xor3(a, b, c);
    carry = lop3_maj(a, b, c);
}

// The same distance plus `bias`: the caller passes bias = -d2 (minus the query's current second-best), so the sign of the
// result says whether the row enters the top 2 — the subtraction rides in the three-input add of the popcounts for free.
__device__ __forceinline__ int hamming256_csa_biased(const uint32_t (&q)[8], const uint4& a, const uint4& b, int bias)
{
    const uint32_t x0 = q[0] ^ a.x, x1 = q[1] ^ a.y, x2 = q[2] ^ a.z, x3 = q[3] ^ a.w;
    const uint32_t x4 = q[4] ^ b.x, x5 = q[5] ^ b.y, x6 = q[6] ^ b.z, x7 = q[7] ^ b.w;
    uint32_t c1, s1, c2, s2, c3, s3, d1, t1;
    csa(x0, x1, x2, c1, s1);
    csa(x3, x4, x5, c2, s2);
    csa(s1, s2, x6, c3, s3);
    csa(c1, c2, c3, d1, t1);
    // one three-input add on the ALU pipe, the two weighted terms as multiply-adds on the (idle) FMA pipe
    int acc = __popc(s3) + __popc(x7) + bias, r;
    asm("mad.lo.s32 %0, %1, 2, %2;" : "=r"(r) : "r"(__popc(t1)), "r"(acc));
    asm("mad.lo.s32 %0, %1, 4, %2;" : "=r"(acc) : "r"(__popc(d1)), "r"(r));
    return acc;
}

__device__ __forceinline__ int hamming256_csa(const uint32_t (&q)[8], const uint4& a, const uint4& b)
{
    const uint32_t x0 = q[0] ^ a.x, x1 = q[1] ^ a.y, x2 = q[2] ^ a.z, x3 = q[3] ^ a.w;
    const uint32_t x4 = q[4] ^ b.x, x5 = q[5] ^ b.y, x6 = q[6] ^ b.z, x7 = q[7] ^ b.w;
    uint32_t c1, s1, c2, s2, c3, s3, d1, t1;
    csa(x0, x1, x2, c1, s1);
    csa(x3, x4, x5, c2, s2);
    csa(s1, s2, x6, c3, s3);
    csa(c1, c2, c3, d1, t1);
    return __popc(s3) + __popc(x7) + 2 * __popc(t1) + 4 * __popc(d1);
}

// lexicographic (d, i) insert used by the merges; idx < 0 = missing
__device__ __forceinline__ void top2_merge(int dist, int idx, int& d1, int& i1, int& d2, int& i2)
{
    if (idx < 0) return;
    const bool lt1 = dist < d1 || (dist == d1 && (i1 < 0 || idx < i1));
    if (lt1) { d2 = d1; i2 = i1; d1 = dist; i1 = idx; return; }
    const bool lt2 = dist < d2 || (dist == d2 && (i2 < 0 || idx < i2));
    if (lt2) { d2 = dist; i2 = idx; }
}

}  // namespace

// grid = (query tiles, db chunks).  Each thread owns KNN_QT queries in registers; the CTA streams its database chunk
// through shared memory (every lane reads the same row -> broadcast LDS.128) and keeps (d1,i1,d2,i2) per query.
template <int MINB>
__global__ void __launch_bounds__(KNN_THREADS, MINB) knn2_kernel(const uint32_t* __restrict__ q, int nq,
                                                          const uint4* __restrict__ db, long long ndb, int index_base,
                                                          long long rows_per_chunk, int32_t* __restrict__ out_idx,
                                                          int32_t* __restrict__ out_dist)
{
    __shared__ uint4 tile[2][KNN_DTILE * 2];
    const int tid = threadIdx.x;
    const int q0 = blockIdx.x * KNN_QTILE;
    const long long r_begin = (long long)blockIdx.y * rows_per_chunk;
    long long r_end = r_begin + rows_per_chunk;
    if (r_end > ndb) r_end = ndb;

    uint32_t qw[KNN_QT][8];
    int d1[KNN_QT], i1[KNN_QT], d2[KNN_QT], i2[KNN_QT];
    int nd2[KNN_QT];                               // -d2: the hot loop computes dist - d2 directly
#pragma unroll
    for (int j = 0; j < KNN_QT; ++j) {
        const int qi = q0 + j * KNN_THREADS + tid;
        const uint4* p = reinterpret_cast<const uint4*>(q + (size_t)(qi < nq ? qi : 0) * 8);
        const uint4 a = __ldg(p), b = __ldg(p + 1);
        qw[j][0] = a.x; qw[j][1] = a.y; qw[j][2] = a.z; qw[j][3] = a.w;
        qw[j][4] = b.x; qw[j][5] = b.y; qw[j][6] = b.z; qw[j][7] = b.w;
        d1[j] = INT_MAX; d2[j] = INT_MAX; i1[j] = -1; i2[j] = -1;
        nd2[j] = -INT_MAX;
    }

    // software pipeline: prefetch tile t+1 into registers while computing tile t
    const long long ntiles = (r_end - r_begin + KNN_DTILE - 1) / KNN_DTILE;
    uint4 pre[4];
    auto fetch = [&](long long t) {
        const long long base = r_begin + t * KNN_DTILE;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int e = k * KNN_THREADS + tid;                 // uint4 index inside the tile (2 per row)
            const long long row = base + (e >> 1);
            pre[k] = row < r_end ? __ldg(db + row * 2 + (e & 1)) : make_uint4(0, 0, 0, 0);
        }
    };
    auto stash = [&](int buf) {
#pragma unroll
        for (int k = 0; k < 4; ++k) tile[buf][k * KNN_THREADS + tid] = pre[k];
    };
    if (ntiles > 0) { fetch(0); stash(0); }
    __syncthreads();
    for (long long t = 0; t < ntiles; ++t) {
        const int buf = (int)(t & 1);
        if (t + 1 < ntiles) fetch(t + 1);
        const long long base = r_begin + t * KNN_DTILE;
        const int rows = (int)((r_end - base) < KNN_DTILE ? (r_end - base) : KNN_DTILE);
#pragma unroll 2
        for (int r = 0; r < rows; ++r) {
            const uint4 a = tile[buf][2 * r], b = tile[buf][2 * r + 1];
            const int gi = index_base + (int)(base + r);
            // ONE guard per row for the thread's four queries: t[j] = dist_j - d2_j, and a row matters only if some t[j] < 0,
            // i.e. if the OR of the four has its sign bit set (after the first few thousand rows that is rare)
            int t[KNN_QT];
#pragma unroll
            for (int j = 0; j < KNN_QT; ++j) t[j] = hamming256_csa_biased(qw[j], a, b, nd2[j]);
            int any = t[0];
#pragma unroll
            for (int j = 1; j < KNN_QT; ++j) any |= t[j];
            if (any < 0) {
#pragma unroll
                for (int j = 0; j < KNN_QT; ++j)
                    if (t[j] < 0) {
                        const int4 rr = top2_insert(t[j] - nd2[j], gi, make_int4(d1[j], i1[j], d2[j], i2[j]));
                        d1[j] = rr.x; i1[j] = rr.y; d2[j] = rr.z; i2[j] = rr.w;
                        nd2[j] = -rr.z;
                    }
            }
        }
        if (t + 1 < ntiles) stash(buf ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < KNN_QT; ++j) {
        const int qi = q0 + j * KNN_THREADS + tid;
        if (qi < nq) {
            const size_t o = ((size_t)blockIdx.y * nq + qi) * 2;
            out_idx[o] = i1[j]; out_idx[o + 1] = i2[j];
            out_dist[o] = d1[j]; out_dist[o + 1] = d2[j];
        }
    }
}

// ---- the same search on the tensor cores (the default; ORBX_KNN_IMMA=0 selects the CSA kernel above) ---------------------------
// Blackwell has no 1-bit MMA (mma.sync b1 compiles into bit-plane LOP3s + IMMA), but Hamming(a, b) = popc(a) + popc(b) - 2 a.b
// with the bits of a and b expanded to {0,1} bytes, and a.b over 256 bytes is eight m16n8k32 u8 MMAs (SASS IMMA.16832.U8.U8,
// 1.39e11 per second on one B200: tools/micro/imma_rate.cu).  A warp keeps the expanded fragments of 32 queries (two m16
// tiles, 64 registers) for the whole chunk; the CTA streams the database through shared memory as the CSA kernel does, every
// warp expands the 8 rows of a group — lane t of a row takes the bits 8 j + t and 8 j + t + 4 of every word, (w >> t) & 0x01010101
// and ((w >> t) >> 4) & 0x01010101: two shifts and two ANDs per word — and issues 16 MMAs per group = 256 compares.  Which bit
// lands on which k index is the same function of (word, lane) for queries and database rows, which is all the dot product needs.  popc(b) per row is computed once per CTA while the tile is stashed.
// Accumulator layout (PTX m16n8k32): c0, c1 = row lane/4, columns 2 (lane%4), +1; c2, c3 = row lane/4 + 8: a thread keeps a top-2
// state per (tile, row half) = 4 states, sees its columns in ascending index order (strict < keeps the earlier row on ties, as
// the reference's scan does), and the four lanes that share a row merge lexicographically at the end.
constexpr int KI_WARPS = 8, KI_QTILE = KI_WARPS * 32, KI_DT = 128;
#ifndef ORBX_KI_UNROLL
#define ORBX_KI_UNROLL 8          // groups of 8 rows in flight per warp: 1 -> 1.40e12, 2 -> 1.48e12, 4 -> 1.51e12, 8 -> 1.53e12 compares/s
#endif
constexpr int kKiUnroll = ORBX_KI_UNROLL;

__global__ void __launch_bounds__(32 * KI_WARPS, 2) knn2_imma_kernel(const uint32_t* __restrict__ q, int nq, const uint4* __restrict__ db,
                                                                    long long ndb, int index_base, long long rows_per_chunk,
                                                                    int32_t* __restrict__ out_idx, int32_t* __restrict__ out_dist)
{
    __shared__ uint4 tile[2][KI_DT * 2];
    __shared__ __align__(16) uint32_t pdq[2][KI_DT * 2];        // popcount of every staged uint4 (two per row)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const long long r_begin = (long long)blockIdx.y * rows_per_chunk;
    long long r_end = r_begin + rows_per_chunk;
    if (r_end > ndb) r_end = ndb;
    const int qw0 = blockIdx.x * KI_QTILE + warp * 32;

    // query fragments: tile T, k-step s: a[T][s][0..3] = rows (g, g+8) x bit sets (8j + t, 8j + t + 4) of word s
    uint32_t a[2][8][4];
    int pq[2][2];
#pragma unroll
    for (int T = 0; T < 2; ++T)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int qi = qw0 + T * 16 + h * 8 + g;
            const uint4* p = reinterpret_cast<const uint4*>(q + (size_t)(qi < nq ? qi : 0) * 8);
            const uint4 x = __ldg(p), y = __ldg(p + 1);
            const uint32_t w[8] = {x.x, x.y, x.z, x.w, y.x, y.y, y.z, y.w};
            int pc = 0;
#pragma unroll
            for (int sidx = 0; sidx < 8; ++sidx) {
                pc += __popc(w[sidx]);
                const uint32_t v = w[sidx] >> t;
                a[T][sidx][h] = v & 0x01010101u;
                a[T][sidx][2 + h] = (v >> 4) & 0x01010101u;
            }
            pq[T][h] = pc;
        }
    // top-2 state per (tile, row half), thresholds in "e space": e = popc(b) - 2 a.b = dist - popc(a)
    int d1[2][2], i1[2][2], d2[2][2], i2[2][2], thr[2][2];
#pragma unroll
    for (int T = 0; T < 2; ++T)
#pragma unroll
        for (int h = 0; h < 2; ++h) { d1[T][h] = INT_MAX; d2[T][h] = INT_MAX; i1[T][h] = -1; i2[T][h] = -1; thr[T][h] = 1 << 20; }

    const long long ntiles = (r_end - r_begin + KI_DT - 1) / KI_DT;
    uint4 pre;
    auto fetch = [&](long long tl) {
        const long long row = r_begin + tl * KI_DT + (tid >> 1);
        pre = row < r_end ? __ldg(db + row * 2 + (tid & 1)) : make_uint4(0, 0, 0, 0);
    };
    auto stash = [&](int buf) {
        tile[buf][tid] = pre;
        pdq[buf][tid] = (uint32_t)(__popc(pre.x) + __popc(pre.y) + __popc(pre.z) + __popc(pre.w));
    };
    if (ntiles > 0) { fetch(0); stash(0); }
    __syncthreads();
    for (long long tl = 0; tl < ntiles; ++tl) {
        const int buf = (int)(tl & 1);
        if (tl + 1 < ntiles) fetch(tl + 1);
        const long long base = r_begin + tl * KI_DT;
#pragma unroll kKiUnroll
        for (int g8 = 0; g8 < KI_DT / 8; ++g8) {
            const uint4 wa = tile[buf][(8 * g8 + g) * 2], wb = tile[buf][(8 * g8 + g) * 2 + 1];
            const uint4 pd4 = *reinterpret_cast<const uint4*>(&pdq[buf][(8 * g8) * 2 + 4 * t]);
            const uint32_t w[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
            int cA[4] = {0, 0, 0, 0}, cB[4] = {0, 0, 0, 0};
#pragma unroll
            for (int sidx = 0; sidx < 8; ++sidx) {
                const uint32_t v = w[sidx] >> t;
                const uint32_t b0 = v & 0x01010101u, b1 = (v >> 4) & 0x01010101u;
                imma_16832_u8(cA, a[0][sidx], b0, b1);
                imma_16832_u8(cB, a[1][sidx], b0, b1);
            }
            const int pd0 = (int)(pd4.x + pd4.y), pd1 = (int)(pd4.z + pd4.w);      // rows base + 8 g8 + 2t, + 1
            int e[2][2][2];                                                      // [tile][row half][column]
            e[0][0][0] = pd0 - 2 * cA[0]; e[0][0][1] = pd1 - 2 * cA[1]; e[0][1][0] = pd0 - 2 * cA[2]; e[0][1][1] = pd1 - 2 * cA[3];
            e[1][0][0] = pd0 - 2 * cB[0]; e[1][0][1] = pd1 - 2 * cB[1]; e[1][1][0] = pd0 - 2 * cB[2]; e[1][1][1] = pd1 - 2 * cB[3];
            int any = 0;
#pragma unroll
            for (int T = 0; T < 2; ++T)
#pragma unroll
                for (int h = 0; h < 2; ++h) any |= min(e[T][h][0], e[T][h][1]) - thr[T][h];
            if (any < 0) {
                const long long row0 = base + 8 * g8 + 2 * t;
#pragma unroll
                for (int T = 0; T < 2; ++T)
#pragma unroll
                    for (int h = 0; h < 2; ++h)
#pragma unroll
                        for (int c = 0; c < 2; ++c)
                            if (e[T][h][c] < thr[T][h] && row0 + c < r_end) {
                                const int4 rr = top2_insert(e[T][h][c] + pq[T][h], index_base + (int)(row0 + c),
                                                            make_int4(d1[T][h], i1[T][h], d2[T][h], i2[T][h]));
                                d1[T][h] = rr.x; i1[T][h] = rr.y; d2[T][h] = rr.z; i2[T][h] = rr.w;
                                if (rr.z != INT_MAX) thr[T][h] = rr.z - pq[T][h];
                            }
            }
        }
        if (tl + 1 < ntiles) stash(buf ^ 1);
        __syncthreads();
    }
    // the four lanes of a row hold disjoint column sets: lexicographic merge, lane t == 0 writes
#pragma unroll
    for (int T = 0; T < 2; ++T)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            int md1 = d1[T][h], mi1 = i1[T][h], md2 = d2[T][h], mi2 = i2[T][h];
#pragma unroll
            for (int x = 1; x <= 2; x <<= 1) {
                const int od1 = __shfl_xor_sync(0xffffffffu, md1, x), oi1 = __shfl_xor_sync(0xffffffffu, mi1, x);
                const int od2 = __shfl_xor_sync(0xffffffffu, md2, x), oi2 = __shfl_xor_sync(0xffffffffu, mi2, x);
                top2_merge(od1, oi1, md1, mi1, md2, mi2);
                top2_merge(od2, oi2, md1, mi1, md2, mi2);
            }
            const int qi = qw0 + T * 16 + h * 8 + g;
            if (t == 0 && qi < nq) {
                const size_t o = ((size_t)blockIdx.y * nq + qi) * 2;
                out_idx[o] = mi1; out_idx[o + 1] = mi2;
                out_dist[o] = md1; out_dist[o + 1] = md2;
            }
        }
}

// shard s holds its [nq][2] candidates at idx_sh + s * shard_stride / dist_sh + s * shard_stride (int32 elements)
__global__ void knn2_merge_kernel(const int32_t* __restrict__ idx_sh, const int32_t* __restrict__ dist_sh, int n_shards,
                                  int nq, int32_t* __restrict__ idx, int32_t* __restrict__ dist, size_t shard_stride)
{
    const int qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    int d1 = INT_MAX, d2 = INT_MAX, i1 = -1, i2 = -1;
    for (int s = 0; s < n_shards; ++s) {
        const size_t o = (size_t)s * shard_stride + (size_t)qi * 2;
        top2_merge(dist_sh[o], idx_sh[o], d1, i1, d2, i2);
        top2_merge(dist_sh[o + 1], idx_sh[o + 1], d1, i1, d2, i2);
    }
    idx[2 * (size_t)qi] = i1; idx[2 * (size_t)qi + 1] = i2;
    dist[2 * (size_t)qi] = d1; dist[2 * (size_t)qi + 1] = d2;
}

// Database chunking of one launch: a few thousand CTAs, every chunk long enough to amortise the query load / result store.
static bool knn2_use_imma()
{
    // default: the tensor-core kernel (1.5e12 compares/s against 8.3e11 of the CSA kernel on 100 k x 10 M); ORBX_KNN_IMMA=0 = CSA kernel
    static const bool on = getenv("ORBX_KNN_IMMA") ? atoi(getenv("ORBX_KNN_IMMA")) != 0 : true;
    return on;
}

static void knn2_plan(int nq, long long ndb, int& qtiles, int& chunks, long long& rows_per_chunk)
{
    qtiles = (nq + (knn2_use_imma() ? KI_QTILE : KNN_QTILE) - 1) / (knn2_use_imma() ? KI_QTILE : KNN_QTILE);
    chunks = 1;
    if (ndb > 0) {
        const long long target_ctas = 148LL * 16;
        long long want = (target_ctas + qtiles - 1) / qtiles;
        const long long max_chunks = (ndb + 4095) / 4096;
        if (want > max_chunks) want = max_chunks;
        if (want < 1) want = 1;
        if (want > 1024) want = 1024;
        chunks = (int)want;
    }
    rows_per_chunk = ndb > 0 ? (ndb + chunks - 1) / chunks : 1;
    rows_per_chunk = (rows_per_chunk + KNN_DTILE - 1) / KNN_DTILE * KNN_DTILE;
    chunks = ndb > 0 ? (int)((ndb + rows_per_chunk - 1) / rows_per_chunk) : 1;
}

size_t knn2_workspace_bytes(int nq, long long ndb)
{
    if (nq <= 0) return 0;
    int qtiles, chunks; long long rpc;
    knn2_plan(nq, ndb, qtiles, chunks, rpc);
    return chunks > 1 ? (size_t)chunks * nq * 2 * sizeof(int32_t) * 2 : 0;
}

// The per-chunk partial results live in `workspace` (>= knn2_workspace_bytes, owned by the caller for the duration of the
// launch) or, with workspace == nullptr, in a stream-ordered allocation made and released on `st` — either way private to
// this call, so concurrent calls from several host threads / streams (Tracking, LocalMapping, LoopClosing all match
// descriptors, SURVEY.md §3.3) never share scratch.
cudaError_t launch_knn2(const uint8_t* d_q, int nq, const uint8_t* d_db, long long ndb, int index_base, int32_t* d_idx,
                        int32_t* d_dist, cudaStream_t st, void* workspace)
{
    if (nq <= 0) return cudaSuccess;
    int qtiles, chunks; long long rows_per_chunk;
    knn2_plan(nq, ndb, qtiles, chunks, rows_per_chunk);
    int32_t* p_idx = d_idx;
    int32_t* p_dist = d_dist;
    void* owned = nullptr;
    if (chunks > 1) {
        if (!workspace) {
            cudaError_t e = cudaMallocAsync(&owned, knn2_workspace_bytes(nq, ndb), st);
            if (e != cudaSuccess) return e;
            workspace = owned;
        }
        p_idx = reinterpret_cast<int32_t*>(workspace);
        p_dist = p_idx + (size_t)chunks * nq * 2;
    }
    dim3 grid(qtiles, chunks);
    // register budget for 5 or 6 CTAs per SM (ORBX_KNN_MINB: A/B switch for measurements)
    static const int minb = getenv("ORBX_KNN_MINB") ? atoi(getenv("ORBX_KNN_MINB")) : 6;     // measured: 8.29e11 (6) vs 8.07e11 (5) compares/s
    if (knn2_use_imma())
        knn2_imma_kernel<<<grid, 32 * KI_WARPS, 0, st>>>(reinterpret_cast<const uint32_t*>(d_q), nq, reinterpret_cast<const uint4*>(d_db), ndb,
                                                         index_base, rows_per_chunk, p_idx, p_dist);
    else if (minb == 6)
        knn2_kernel<6><<<grid, KNN_THREADS, 0, st>>>(reinterpret_cast<const uint32_t*>(d_q), nq, reinterpret_cast<const uint4*>(d_db), ndb,
                                                     index_base, rows_per_chunk, p_idx, p_dist);
    else
        knn2_kernel<5><<<grid, KNN_THREADS, 0, st>>>(reinterpret_cast<const uint32_t*>(d_q), nq, reinterpret_cast<const uint4*>(d_db), ndb,
                                                     index_base, rows_per_chunk, p_idx, p_dist);
    count_launch();
    if (chunks > 1) {
        knn2_merge_kernel<<<(nq + 255) / 256, 256, 0, st>>>(p_idx, p_dist, chunks, nq, d_idx, d_dist, (size_t)nq * 2);
        count_launch();
    }
    cudaError_t e = cudaGetLastError();
    if (owned) { cudaError_t e2 = cudaFreeAsync(owned, st); if (e == cudaSuccess) e = e2; }
    return e;
}

cudaError_t launch_knn2_merge(const int32_t* d_idx_sh, const int32_t* d_dist_sh, int n_shards, int nq, int32_t* d_idx,
                              int32_t* d_dist, cudaStream_t st, size_t shard_stride)
{
    if (nq <= 0) return cudaSuccess;
    knn2_merge_kernel<<<(nq + 255) / 256, 256, 0, st>>>(d_idx_sh, d_dist_sh, n_shards, nq, d_idx, d_dist,
                                                        shard_stride ? shard_stride : (size_t)nq * 2);
    count_launch();
    return cudaGetLastError();
}

// ---- POPC issue-rate microbenchmark: 8 independent dependent-chains per thread ------------------------------------
__global__ void __launch_bounds__(256) popc_bench_kernel(unsigned long long* sink, int iters)
{
    uint32_t x[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) x[k] = (threadIdx.x * 2654435761u) ^ (blockIdx.x * 40503u + k * 0x9E3779B9u);
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = __popc(x[k]) ^ (0xA5A5A5A5u << k);
    }
    uint32_t s = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += x[k];
    if (s == 0x12345678u) sink[0] = s;   // practically never; keeps the chain alive
}

cudaError_t launch_popc_bench(unsigned long long* d_sink, int iters, int blocks, cudaStream_t st)
{
    popc_bench_kernel<<<blocks, 256, 0, st>>>(d_sink, iters);
    count_launch();
    return cudaGetLastError();
}

// ---- stereo ---------------------------------------------------------------------------------------------------------
namespace {

__device__ __forceinline__ int hamming256(const uint32_t* a, const uint32_t* b)
{
    int d = 0;
#pragma unroll
    for (int k = 0; k < 8; ++k) d += __popc(a[k] ^ b[k]);
    return d;
}

}  // namespace

// one warp per left keypoint (src/Frame.cc:881-995); blockIdx.y = pair
__global__ void __launch_bounds__(256) stereo_match_kernel(const __grid_constant__ FrameGeom fg, StereoArgs A)
{
    __shared__ int s_sad[8][12];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int iL = blockIdx.x * 8 + warp;
    const int p = blockIdx.y;
    // pair p: rows p * nL (left side and outputs) / p * nR (right side) of every per-pair array
    const size_t rowL = (size_t)p * A.nL, rowR = (size_t)p * A.nR;
    // device-resident counts: a frame that overflowed its capacity (count > bound) has no valid rows
    int nL = A.nL, nR = A.nR;
    if (A.d_nL) { const int c = __ldg(A.d_nL + p); nL = c > A.nL ? 0 : c; }
    if (A.d_nR) { const int c = __ldg(A.d_nR + p); nR = c > A.nR ? 0 : c; }
    if (iL >= nL) return;
    const orbx_keypoint* kpR = A.kpR + rowR;
    const uint8_t* descR = A.descR + rowR * 32;
    const int TH_HIGH = 100, TH_LOW = 50;
    const int thOrbDist = (TH_HIGH + TH_LOW) / 2;
    const orbx_keypoint kL = A.kpL[rowL + iL];
    const int levelL = min(max(kL.octave, 0), fg.nlevels - 1);      // host entry points validate; device-resident input is clamped
    const float vL = kL.y, uL = kL.x;
    float out_u = -1.0f, out_d = -1.0f;
    int out_sad = -1;
    const float minD = 0.f, maxD = A.maxD;
    const float minU = __fsub_rn(uL, maxD), maxU = __fsub_rn(uL, minD);
    if (!(maxU < 0)) {
        const int row = (int)vL;
        uint32_t dl[8];
        const uint32_t* pl = reinterpret_cast<const uint32_t*>(A.descL + (rowL + iL) * 32);
#pragma unroll
        for (int k = 0; k < 8; ++k) dl[k] = __ldg(pl + k);
        // best = min over (dist, iR): the reference scans row buckets in ascending iR with strict '<'
        unsigned best = 0xffffffffu;
        for (int iR = lane; iR < nR; iR += 32) {
            const orbx_keypoint kR = kpR[iR];
            if ((unsigned)kR.octave >= (unsigned)fg.nlevels) continue;
            const float r = __fmul_rn(2.0f, fg.L[kR.octave].scale);
            const int maxr = (int)ceilf(__fadd_rn(kR.y, r));
            const int minr = (int)floorf(__fsub_rn(kR.y, r));
            if (row < minr || row > maxr) continue;
            if (kR.octave < levelL - 1 || kR.octave > levelL + 1) continue;
            if (kR.x >= minU && kR.x <= maxU) {
                const int dist = hamming256(dl, reinterpret_cast<const uint32_t*>(descR + (size_t)iR * 32));
                if (dist < TH_HIGH) best = min(best, ((unsigned)dist << 20) | (unsigned)iR);
            }
        }
#pragma unroll
        for (int d = 16; d >= 1; d >>= 1) best = min(best, __shfl_xor_sync(0xffffffffu, best, d));
        const int bestDist = best == 0xffffffffu ? TH_HIGH : (int)(best >> 20);
        if (bestDist < thOrbDist) {
            const int bestIdxR = (int)(best & 0xfffffu);
            const float uR0 = kpR[bestIdxR].x;
            const LevelGeom& g = fg.L[levelL];
            const float sf = g.inv_scale;
            const float scaleduL = roundf(__fmul_rn(kL.x, sf));
            const float scaledvL = roundf(__fmul_rn(kL.y, sf));
            const float scaleduR0 = roundf(__fmul_rn(uR0, sf));
            const int w = 5, L = 5;
            const float iniu = scaleduR0 + L - w;
            const float endu = scaleduR0 + L + w + 1;
            if (!(iniu < 0 || endu >= g.w)) {
                const uint8_t* IL = level_interior(A.pyrL, g, A.frameL + p);
                const uint8_t* IR = A.pyrR + A.offR[levelL] + (unsigned long long)(A.frameR + p) * g.pyr_frame_stride +
                                    (unsigned long long)kEdge * g.pitch + kXPad;
                if (lane < 11) s_sad[warp][lane] = 0;
                __syncwarp();
                const int cu = (int)scaleduL, cv = (int)scaledvL, cr = (int)scaleduR0;
                for (int task = lane; task < 121; task += 32) {
                    const int inc = task / 11 - L, dy = task % 11 - w;
                    const uint8_t* pl2 = IL + (ptrdiff_t)(cv + dy) * g.pitch + (cu - w);
                    const uint8_t* pr2 = IR + (ptrdiff_t)(cv + dy) * g.pitch + (cr + inc - w);
                    int acc = 0;
#pragma unroll
                    for (int dx = 0; dx < 11; ++dx) acc += abs((int)__ldg(pl2 + dx) - (int)__ldg(pr2 + dx));
                    atomicAdd(&s_sad[warp][inc + L], acc);
                }
                __syncwarp();
                int bestS = INT_MAX, bestinc = 0;
                for (int k = 0; k < 11; ++k) {
                    const float dist = (float)s_sad[warp][k];
                    if (dist < (float)bestS) { bestS = (int)dist; bestinc = k - L; }
                }
                if (!(bestinc == -L || bestinc == L)) {
                    const float dist1 = (float)s_sad[warp][L + bestinc - 1];
                    const float dist2 = (float)s_sad[warp][L + bestinc];
                    const float dist3 = (float)s_sad[warp][L + bestinc + 1];
                    const float deltaR = __fdiv_rn(__fsub_rn(dist1, dist3),
                                                   __fmul_rn(2.0f, __fsub_rn(__fadd_rn(dist1, dist3), __fmul_rn(2.0f, dist2))));
                    if (!(deltaR < -1 || deltaR > 1)) {
                        float bestuR = __fmul_rn(g.scale, __fadd_rn(__fadd_rn(scaleduR0, (float)bestinc), deltaR));
                        float disparity = __fsub_rn(uL, bestuR);
                        if (disparity >= minD && disparity < maxD) {
                            if (disparity <= 0) { disparity = 0.01f; bestuR = (float)((double)uL - 0.01); }
                            out_d = __fdiv_rn(A.bf, disparity);
                            out_u = bestuR;
                            out_sad = bestS;
                        }
                    }
                }
            }
        }
    }
    if (lane == 0) { A.uRight[rowL + iL] = out_u; A.depth[rowL + iL] = out_d; A.sad[rowL + iL] = out_sad; }
}

// one CTA per pair: median filter of src/Frame.cc:997-1010.  The accepted matches (a few hundred of ~1200 left keypoints) are compacted
// into shared memory first; the median of the (SAD, iL)-sorted list is found by rank counting over that list (the first version
// counted over all keypoints in global memory: 89 us of the 300 us of a stereo pair; now a few us).
constexpr int kMedianCap = 4096;          // accepted matches held in shared memory (more: rank counting over global memory)
__global__ void __launch_bounds__(1024) stereo_median_kernel(StereoArgs A)
{
    __shared__ int s_n, s_median;
    __shared__ int s_sad[kMedianCap];
    __shared__ int s_idx[kMedianCap];
    const int tid = threadIdx.x;
    const size_t rowL = (size_t)blockIdx.x * A.nL;      // pair blockIdx.x
    const int* sad = A.sad + rowL;
    int nL = A.nL;
    if (A.d_nL) { const int c = __ldg(A.d_nL + blockIdx.x); nL = c > A.nL ? 0 : c; }
    if (tid == 0) { s_n = 0; s_median = -1; }
    __syncthreads();
    for (int i = tid; i < nL; i += 1024) {
        const int si = sad[i];
        if (si >= 0) {
            const int slot = atomicAdd(&s_n, 1);         // order is irrelevant: ranks use (sad, original index)
            if (slot < kMedianCap) { s_sad[slot] = si; s_idx[slot] = i; }
        }
    }
    __syncthreads();
    const int n = s_n;
    if (n == 0) return;
    const int target = n / 2;
    if (n <= kMedianCap) {
        for (int e = tid; e < n; e += 1024) {
            const int si = s_sad[e], ii = s_idx[e];
            int rank = 0;
            for (int j = 0; j < n; ++j) {
                const int sj = s_sad[j];
                rank += (sj < si) || (sj == si && s_idx[j] < ii);
            }
            if (rank == target) s_median = si;
        }
    } else {
        // rank of element i in the sorted (sad, iL) list, counted over global memory
        for (int i = tid; i < nL; i += 1024) {
            const int si = sad[i];
            if (si < 0) continue;
            int rank = 0;
            for (int j = 0; j < nL; ++j) {
                const int sj = sad[j];
                if (sj < 0) continue;
                rank += (sj < si) || (sj == si && j < i);
            }
            if (rank == target) s_median = si;
        }
    }
    __syncthreads();
    const float median = (float)s_median;
    const float thDist = 1.5f * 1.4f * median;
    for (int i = tid; i < nL; i += 1024) {
        const int si = sad[i];
        if (si >= 0 && !((float)si < thDist)) { A.uRight[rowL + i] = -1.f; A.depth[rowL + i] = -1.f; }
    }
}

cudaError_t launch_stereo(const FrameGeom& fg, const StereoArgs& a, cudaStream_t st)
{
    if (a.nL <= 0 || a.n_pairs <= 0) return cudaSuccess;
    stereo_match_kernel<<<dim3((a.nL + 7) / 8, a.n_pairs), 256, 0, st>>>(fg, a);
    count_launch();
    stereo_median_kernel<<<a.n_pairs, 1024, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

// ---- synthetic inputs ---------------------------------------------------------------------------------------------------
__global__ void synth_images_kernel(uint32_t seed0, int view, int cols, int rows, int max_disp, uint8_t* dst, size_t pitch,
                                    size_t frame_stride)
{
    const int x4 = (blockIdx.x * blockDim.x + threadIdx.x) * 4;
    const int y = blockIdx.y, f = blockIdx.z;
    if (x4 >= cols) return;
    uint8_t* row = dst + (size_t)f * frame_stride + (size_t)y * pitch;
    for (int j = 0; j < 4 && x4 + j < cols; ++j) row[x4 + j] = orbx_synth::image_pixel(seed0 + (uint32_t)f, view, x4 + j, y, max_disp);
}

cudaError_t launch_synth_images(uint32_t seed0, int view, int n_frames, int cols, int rows, int max_disp, uint8_t* d_dst,
                                size_t pitch, size_t frame_stride, cudaStream_t st)
{
    dim3 grid(((cols + 3) / 4 + 127) / 128, rows, n_frames);
    synth_images_kernel<<<grid, 128, 0, st>>>(seed0, view, cols, rows, max_disp, d_dst, pitch, frame_stride);
    count_launch();
    return cudaGetLastError();
}

__global__ void synth_desc_kernel(uint32_t seed, int is_query, long long first_row, long long n_rows, long long ndb,
                                  int plant_every, uint32_t* dst)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;   // word index
    if (i >= n_rows * 8) return;
    const uint32_t row = (uint32_t)(first_row + (i >> 3)), w = (uint32_t)(i & 7);
    dst[i] = is_query ? orbx_synth::query_word(seed, row, w, (uint32_t)ndb, (uint32_t)plant_every)
                      : orbx_synth::desc_word(seed, row, w);
}

cudaError_t launch_synth_desc(uint32_t seed, int is_query, long long first_row, long long n_rows, long long ndb,
                              int plant_every, uint8_t* d_dst, cudaStream_t st)
{
    if (n_rows <= 0) return cudaSuccess;
    const long long words = n_rows * 8;
    synth_desc_kernel<<<(unsigned)((words + 255) / 256), 256, 0, st>>>(seed, is_query, first_row, n_rows, ndb, plant_every,
                                                                       reinterpret_cast<uint32_t*>(d_dst));
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
