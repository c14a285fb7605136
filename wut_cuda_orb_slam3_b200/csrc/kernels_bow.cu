// kernels_bow.cu — vocabulary-tree descent (DBoW2 transform) and the vocabulary-guided Hamming searches of ORBmatcher.
//
// Reference semantics reproduced (paths relative to the reference root):
//   * TemplatedVocabulary::transform(feature, word_id, weight, nid, levelsup) — Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h:1217-1259
//     with FORB::distance (Thirdparty/DBoW2/DBoW2/FORB.cpp:81-101): greedy descent, least Hamming distance, ties -> first child.
//   * ORBmatcher::SearchByBoW(KF, Frame) src/ORBmatcher1.cc:225-427 and SearchByBoW(KF, KF) src/ORBmatcher2.cc:36-171: per common
//     vocabulary node, the A features are visited IN ORDER, each scans the node's B features for best / second-best distance
//     (strict '<': the earlier candidate keeps a tie) and B features matched earlier are skipped — a sequential dependence
//     inside a node, none across nodes (a feature belongs to exactly one node) and none across the key frames of a batch.
//   * ORBmatcher::SearchForTriangulation src/ORBmatcher2.cc:173-471 (single pinhole camera): independent 1-NN per A feature
//     with the epipole gate and Pinhole::epipolarConstrain (src/CameraModels/Pinhole.cpp:107-129).
//
// All three are integer XOR/POPC work on a few thousand descriptors: one warp per unit of independence, lanes across the
// candidates, warp-shuffle reductions that reproduce the reference's scan-order tie rules.
#include "orbx_internal.cuh"

namespace orbx {

namespace {

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

}  // namespace

// ---- vocabulary descent -------------------------------------------------------------------------------------------------
// One warp per feature; lane c evaluates child c of the current node (k <= 32), a warp arg-min over (distance, child order)
// picks the next node.  Children descriptors of a node are contiguous in `cdesc` (re-packed on the host).
__global__ void __launch_bounds__(128) bow_descend_kernel(VocabDev v, const uint8_t* __restrict__ desc, int n, int nid_level,
                                                          uint32_t* __restrict__ word_id, double* __restrict__ weight,
                                                          uint32_t* __restrict__ node_id)
{
    const int lane = threadIdx.x & 31;
    const int f = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (f >= n) return;
    uint32_t q[8];
    load_desc(desc, (size_t)f, q);
    int node = 0, level = 0;
    uint32_t nid = 0;                                   // root when nid_level <= 0 (TemplatedVocabulary.h:1227)
    int cnt = __ldg(v.child_count);
    while (cnt > 0) {                                   // do { ... } while(!isLeaf): the root of a non-empty vocabulary has children
        ++level;
        const int beg = __ldg(v.child_begin + node);
        uint32_t key = 0xffffffffu;                     // (distance << 8) | child order: min == least distance, first child on ties
        for (int c0 = 0; c0 < cnt; c0 += 32) {
            const int c = c0 + lane;
            if (c < cnt) {
                uint32_t d[8];
                load_desc(v.cdesc, (size_t)(beg + c), d);
                key = min(key, ((uint32_t)hamming256(q, d) << 8) | (uint32_t)c);
            }
        }
#pragma unroll
        for (int s = 16; s >= 1; s >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, s));
        node = __ldg(v.child_id + beg + (int)(key & 0xff));
        if (level == nid_level) nid = (uint32_t)node;
        cnt = __ldg(v.child_count + node);
    }
    if (lane == 0) {
        if (word_id) word_id[f] = (uint32_t)__ldg(v.word_of_node + node);
        if (weight) weight[f] = __ldg(v.weight + node);
        if (node_id) node_id[f] = nid;
    }
}

cudaError_t launch_bow_descend(const VocabDev& v, const uint8_t* d_desc, int n, int nid_level, uint32_t* d_word, double* d_weight,
                               uint32_t* d_node, cudaStream_t st)
{
    if (n <= 0) return cudaSuccess;
    bow_descend_kernel<<<(n + 3) / 4, 128, 0, st>>>(v, d_desc, n, nid_level, d_word, d_weight, d_node);
    count_launch();
    return cudaGetLastError();
}

// ---- SearchByBoW ----------------------------------------------------------------------------------------------------------
namespace {

struct Best2 {
    int b1, t1, b2;     // least distance, its list position (first on ties), second-least distance (multiset sense)
};
__device__ __forceinline__ void best2_init(Best2& s) { s.b1 = 256; s.t1 = 0x7fffffff; s.b2 = 256; }   // src/ORBmatcher1.cc:267-269
__device__ __forceinline__ void best2_push(Best2& s, int dist, int t)
{
    if (dist < s.b1) { s.b2 = s.b1; s.b1 = dist; s.t1 = t; }     // src/ORBmatcher1.cc:296-305
    else if (dist < s.b2) s.b2 = dist;
}
// merge of two partial scans over disjoint position sets == the scan over their union in position order
__device__ __forceinline__ void best2_merge(Best2& s, int ob1, int ot1, int ob2)
{
    const bool other_wins = ob1 < s.b1 || (ob1 == s.b1 && ot1 < s.t1);
    const int loser = other_wins ? s.b1 : ob1;
    s.b2 = min(min(s.b2, ob2), loser);
    if (other_wins) { s.b1 = ob1; s.t1 = ot1; }
}
__device__ __forceinline__ void best2_warp_reduce(Best2& s)
{
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        const int ob1 = __shfl_xor_sync(0xffffffffu, s.b1, d), ot1 = __shfl_xor_sync(0xffffffffu, s.t1, d);
        const int ob2 = __shfl_xor_sync(0xffffffffu, s.b2, d);
        best2_merge(s, ob1, ot1, ob2);
    }
}

}  // namespace

// Job build of key frame blockIdx.x: its row of the fixed side and its own per-feature rows = -1, then the common nodes of the
// two ascending node lists (a node of the fixed side is looked up in the key frame's list by binary search: the node ids are
// strictly ascending, so the equal pairs are those of the lock-step walk, src/ORBmatcher1.cc:247-251, 397-404), one job per
// common node with features on both sides.  A node of the fixed side gives at most one job, so key frame k has at most
// job_stride jobs; the order of the jobs is irrelevant (different nodes hold different features of both sides).
__global__ void __launch_bounds__(256) bow_jobs_kernel(BowBatchArgs a)
{
    const int k = blockIdx.x;
    const BowKF& K = a.kfs[k];
    __shared__ int s_count;
    if (threadIdx.x == 0) s_count = 0;
    int* row = a.row + (size_t)k * a.n;
    for (int i = threadIdx.x; i < a.n; i += blockDim.x) row[i] = -1;
    for (int i = threadIdx.x; i < K.n; i += blockDim.x) {
        if (a.feat) a.feat[K.base + i] = -1;
        if (a.feat_right) a.feat_right[K.base + i] = -1;
    }
    __syncthreads();
    const int nb = K.n_nodes;
    int4* jobs = a.jobs + (size_t)k * a.job_stride;
    for (int p = threadIdx.x; p < a.n_nodes; p += blockDim.x) {
        const uint32_t id = __ldg(a.node_ids + p);
        int lo = 0, hi = nb;                                 // first position of the key frame's list with node id >= id
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(K.node_ids + mid) < id) lo = mid + 1;
            else hi = mid;
        }
        if (lo == nb || __ldg(K.node_ids + lo) != id) continue;
        const int f0 = __ldg(a.offsets + p), f1 = __ldg(a.offsets + p + 1), k0 = __ldg(K.offsets + lo), k1 = __ldg(K.offsets + lo + 1);
        if (f0 == f1 || k0 == k1) continue;                  // no A feature to walk or no B feature to scan: no match either way
        const int slot = atomicAdd(&s_count, 1);
        jobs[slot] = a.mode == 0 ? make_int4(k0, k1, f0, f1) : make_int4(f0, f1, k0, k1);
    }
    __syncthreads();
    if (threadIdx.x == 0) a.job_count[k] = s_count;
}

// One warp per job (a common vocabulary node) of key frame blockIdx.y.  match_b doubles as the "already matched" state of B
// (mode 0: the key frame's row of vpMapPointMatches, mode 1: the key frame's vbMatched2); it is read/written through L2
// (ld.cg / st.cg) and ordered by __syncwarp between A features.  kf_frame = mode 0.
template <bool kf_frame>
__global__ void __launch_bounds__(128) search_by_bow_kernel(BowBatchArgs a)
{
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.y;
    const int jb = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (jb >= __ldg(a.job_count + k)) return;
    const BowKF* K = a.kfs + k;
    const int4 pr = __ldg(a.jobs + (size_t)k * a.job_stride + jb);      // (a_begin, a_end, b_begin, b_end) into idx_a / idx_b
    const size_t base = K->base;
    const uint32_t* __restrict__ idx_a = kf_frame ? K->indices : a.indices;
    const uint32_t* __restrict__ idx_b = kf_frame ? a.indices : K->indices;
    const uint8_t* __restrict__ desc_a = kf_frame ? K->desc : a.desc;
    const uint8_t* __restrict__ desc_b = kf_frame ? a.desc : K->desc;
    const uint8_t* __restrict__ valid_a = kf_frame ? K->valid : a.valid;
    const uint8_t* __restrict__ valid_b = K->valid;                         // read in mode 1 only
    int* row = a.row + (size_t)k * a.n;
    int* match_b = kf_frame ? row : a.feat + base;
    int* match_a = kf_frame ? (a.feat ? a.feat + base : nullptr) : row;
    int* match_a_right = kf_frame && a.feat_right ? a.feat_right + base : nullptr;
    const int TH_LOW = 50;                                   // src/ORBmatcher1.cc:37
    for (int ia = pr.x; ia < pr.y; ++ia) {
        const int iA = (int)__ldg(idx_a + ia);
        if (!__ldg(valid_a + iA)) continue;                  // !pMP || pMP->isBad()   (src/ORBmatcher1.cc:259-265)
        uint32_t q[8];
        load_desc(desc_a, (size_t)iA, q);
        Best2 L, R;
        best2_init(L); best2_init(R);
        for (int t = pr.z + lane; t < pr.w; t += 32) {
            const int j = (int)__ldg(idx_b + t);
            if (__ldcg(match_b + j) >= 0) continue;          // vpMapPointMatches[realIdxF] / vbMatched2[idx2]
            if (!kf_frame && !__ldg(valid_b + j)) continue;  // !pMP2 || pMP2->isBad()   (src/ORBmatcher2.cc:95-103)
            uint32_t d[8];
            load_desc(desc_b, (size_t)j, d);
            const int dist = hamming256(q, d);
            if (a.nleft < 0 || j < a.nleft) best2_push(L, dist, t);
            else best2_push(R, dist, t);                     // src/ORBmatcher1.cc:323-330
        }
        best2_warp_reduce(L);
        if (a.nleft >= 0) best2_warp_reduce(R);
        // acceptance (identical on all lanes); lane 0 writes
        int jL = -1, jR = -1;
        if (kf_frame) {
            if (L.b1 <= TH_LOW) {                                                            // src/ORBmatcher1.cc:336
                if ((float)L.b1 < __fmul_rn(a.nn_ratio, (float)L.b2)) jL = (int)__ldg(idx_b + L.t1);            // :338
                if (a.nleft >= 0 && R.b1 <= TH_LOW) jR = (int)__ldg(idx_b + R.t1);           // :366-368 ('|| true')
            }
        } else {
            if (L.b1 < TH_LOW && (float)L.b1 < __fmul_rn(a.nn_ratio, (float)L.b2)) jL = (int)__ldg(idx_b + L.t1);    // ORBmatcher2.cc:120-122
        }
        if (lane == 0) {
            if (jL >= 0) { __stcg(match_b + jL, iA); if (match_a) match_a[iA] = jL; }
            if (jR >= 0) { __stcg(match_b + jR, iA); if (match_a_right) match_a_right[iA] = jR; }
        }
        __syncwarp();
    }
}

cudaError_t launch_search_by_bow_batch(const BowBatchArgs& a, cudaStream_t st)
{
    if (a.n_kf <= 0 || a.n <= 0) return cudaSuccess;
    bow_jobs_kernel<<<a.n_kf, 256, 0, st>>>(a);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess || a.job_stride <= 0) return e;
    const dim3 grid((a.job_stride + 3) / 4, a.n_kf);
    if (a.mode == 0) search_by_bow_kernel<true><<<grid, 128, 0, st>>>(a);
    else search_by_bow_kernel<false><<<grid, 128, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

// ---- SearchForTriangulation -------------------------------------------------------------------------------------------------
namespace {

// The scan of one (A feature, common node) job by one warp: the least distance <= TH_LOW among gate-passing candidates
// idx_b[b_begin, b_end), the LAST one in list order on ties ('dist > bestDist' is the skip test, src/ORBmatcher2.cc:289).
// Returns the KF2 index or -1 (on every lane).  F / scale_b / sigma2_b are the pair's tables (global: the neighbour's TriKF).
__device__ __forceinline__ int tri_scan(int lane, const uint32_t q[8], const orbx_keypoint& k1, bool stereo1, const float* F, float ep0,
                                        float ep1, const float* scale_b, const float* sigma2_b, bool only_stereo, bool coarse,
                                        const uint32_t* __restrict__ idx_b, const uint8_t* __restrict__ free_b,
                                        const uint8_t* __restrict__ stereo_b, const uint8_t* __restrict__ desc_b,
                                        const orbx_keypoint* kp_b, int b_begin, int b_end)
{
    const int TH_LOW = 50;
    // epipolar line of kp1 in image 2: l = x1' F12 = [la lb lc]   (src/CameraModels/Pinhole.cpp:115-117), float, no FMA
    const float la = __fadd_rn(__fadd_rn(__fmul_rn(k1.x, F[0]), __fmul_rn(k1.y, F[3])), F[6]);
    const float lb = __fadd_rn(__fadd_rn(__fmul_rn(k1.x, F[1]), __fmul_rn(k1.y, F[4])), F[7]);
    const float lc = __fadd_rn(__fadd_rn(__fmul_rn(k1.x, F[2]), __fmul_rn(k1.y, F[5])), F[8]);
    const float den = __fadd_rn(__fmul_rn(la, la), __fmul_rn(lb, lb));
    uint32_t key = 0xffffffffu;                              // (distance << 24) | (0xffffff - relative list position): min == least distance, last position
    for (int t = b_begin + lane; t < b_end; t += 32) {
        const int j = (int)__ldg(idx_b + t);
        if (!__ldg(free_b + j)) continue;                    // vbMatched2[idx2] (never set) || pMP2   (src/ORBmatcher2.cc:276)
        const bool stereo2 = __ldg(stereo_b + j) != 0;
        if (only_stereo && !stereo2) continue;               // :281-283
        uint32_t d[8];
        load_desc(desc_b, (size_t)j, d);
        const int dist = hamming256(q, d);
        if (dist > TH_LOW) continue;                         // :289
        const orbx_keypoint k2 = kp_b[j];
        if (!stereo1 && !stereo2) {                          // :299-307 (single camera: !pKF1->mpCamera2)
            const float dx = __fsub_rn(ep0, k2.x), dy = __fsub_rn(ep1, k2.y);
            if (__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)) < __fmul_rn(100.0f, scale_b[k2.octave])) continue;
        }
        if (!coarse) {                                       // Pinhole::epipolarConstrain (Pinhole.cpp:119-128)
            const float num = __fadd_rn(__fadd_rn(__fmul_rn(la, k2.x), __fmul_rn(lb, k2.y)), lc);
            if (den == 0.0f) continue;
            const float dsqr = __fdiv_rn(__fmul_rn(num, num), den);
            if (!((double)dsqr < 3.84 * (double)sigma2_b[k2.octave])) continue;
        }
        key = min(key, ((uint32_t)dist << 24) | (uint32_t)(0xffffff - (t - b_begin)));
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, s));
    return key == 0xffffffffu ? -1 : (int)__ldg(idx_b + b_begin + (int)(0xffffff - (key & 0xffffff)));
}

}  // namespace

// Job build of neighbour blockIdx.x: match row k = -1, then the common nodes of the two ascending node lists (a node of A is
// looked up in B's list by binary search: the node ids are strictly ascending, so the equal pairs are those of the lock-step
// walk, src/ORBmatcher2.cc:226-236, 458-467) and one job per A feature of a common node that is free (and stereo under
// only_stereo).  A feature sits in one node of A, so neighbour k has at most n_a jobs; the order of the jobs is irrelevant
// (each writes its own feature's slot).
__global__ void __launch_bounds__(256) tri_jobs_kernel(TriBatchArgs a)
{
    const int k = blockIdx.x;
    const TriKF& K = a.kfs[k];
    __shared__ int s_count;
    if (threadIdx.x == 0) s_count = 0;
    int* match = a.match + (size_t)k * a.n_a;
    for (int i = threadIdx.x; i < a.n_a; i += blockDim.x) match[i] = -1;
    __syncthreads();
    const int nb = K.n_nodes;
    int4* jobs = a.jobs + (size_t)k * a.n_a;
    if (K.n > 0) {
        for (int p = threadIdx.x; p < a.a_nodes; p += blockDim.x) {
            const uint32_t id = __ldg(a.a_node_ids + p);
            int lo = 0, hi = nb;                             // first position of B with node id >= id
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(K.node_ids + mid) < id) lo = mid + 1;
                else hi = mid;
            }
            if (lo == nb || __ldg(K.node_ids + lo) != id) continue;
            const int b0 = __ldg(K.offsets + lo), b1 = __ldg(K.offsets + lo + 1);
            for (int t = __ldg(a.a_offsets + p), te = __ldg(a.a_offsets + p + 1); t < te; ++t) {
                const int iA = (int)__ldg(a.a_indices + t);
                if (!__ldg(a.free_a + iA)) continue;         // already has a MapPoint (src/ORBmatcher2.cc:246-252)
                if (a.only_stereo && !__ldg(a.stereo_a + iA)) continue;       // :256-258
                const int slot = atomicAdd(&s_count, 1);
                if (slot < a.n_a) jobs[slot] = make_int4(iA, b0, b1, 0);    // (bound: a feature listed in two nodes of A)
            }
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) a.job_count[k] = min(s_count, a.n_a);
}

// One warp per job slot of neighbour blockIdx.y; the neighbour's F12, epipole, scale / sigma2 tables and coarse flag are read
// from its TriKF.
__global__ void __launch_bounds__(128) tri_batch_scan_kernel(TriBatchArgs a)
{
    const int lane = threadIdx.x & 31;
    const int k = blockIdx.y;
    const int jb = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (jb >= __ldg(a.job_count + k)) return;
    const TriKF* __restrict__ K = a.kfs + k;
    const int4 job = __ldg(a.jobs + (size_t)k * a.n_a + jb);  // (iA, b_begin, b_end, unused)
    const int iA = job.x;
    const orbx_keypoint k1 = a.kp_a[iA];
    const bool stereo1 = __ldg(a.stereo_a + iA) != 0;
    uint32_t q[8];
    load_desc(a.desc_a, (size_t)iA, q);
    const int m = tri_scan(lane, q, k1, stereo1, K->F12, __ldg(K->ep), __ldg(K->ep + 1), K->scale, K->sigma2, a.only_stereo, __ldg(&K->coarse),
                           K->indices, K->free, K->stereo, K->desc, K->kp, job.y, job.z);
    if (lane == 0) a.match[(size_t)k * a.n_a + iA] = m;
}

cudaError_t launch_search_triangulation_batch(const TriBatchArgs& a, cudaStream_t st)
{
    if (a.n_kf <= 0 || a.n_a <= 0) return cudaSuccess;
    tri_jobs_kernel<<<a.n_kf, 256, 0, st>>>(a);
    count_launch();
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    tri_batch_scan_kernel<<<dim3((a.n_a + 3) / 4, a.n_kf), 128, 0, st>>>(a);
    count_launch();
    return cudaGetLastError();
}

}  // namespace orbx
