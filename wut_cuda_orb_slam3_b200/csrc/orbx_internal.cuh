// orbx_internal.cuh — shared definitions between the host API (api.cu) and the sm_100a kernels.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

#include "../../include/orbx.h"

namespace orbx {

constexpr int kEdge = ORBX_EDGE_THRESHOLD;   // 19
constexpr int kXPad = 32;                     // left pad of a pyramid row: interior pixel 0 is 16-byte aligned
constexpr int kWinBorder = 16;                // EDGE_THRESHOLD - 3: FAST window origin (src/ORBextractor.cc:960-962)
constexpr int kMaxLevels = ORBX_MAX_LEVELS;
constexpr int kMaxCellDim = 70;               // wCell/hCell < 70 whenever the grid has >= 1 cell
constexpr int kMaxDim = 4128;                 // packed 12-bit window coordinates
constexpr int kHalfPatch = 15;
// window of a blurred level staged per keypoint for rBRIEF: |dx|, |dy| <= 19, + 15 bytes of alignment; a row pitch of 80 bytes spreads
// the rows over 8 shared-memory bank offsets (64 bytes: 2)
constexpr int kDescBoxW = 80, kDescBoxH = 40;
// box of the blur's tensor maps over a bordered level: 128 output columns + 16-byte aligned halo (columns x0 - 16 .. x0 + 159) by
// 32 output rows + 3 above + 5 below (blur_mma_kernel works in 8-row blocks); a pitch of 176 bytes (44 words, 12 mod 32) puts the
// 32-bit loads of 8 rows x 4 consecutive words on distinct banks
constexpr int kBlurBoxW = 176, kBlurBoxH = 40;

// Geometry of one pyramid level for the current image shape (host-computed, passed to kernels by value).
struct LevelGeom {
    int w, h;                 // interior size
    int pitch;                // bytes per row of the bordered buffer (multiple of 16)
    int rows_alloc;           // h + 2*19
    unsigned long long pyr_off;       // byte offset of this level's slab inside the pyramid allocation
    unsigned long long pyr_frame_stride;
    int bpitch;               // blurred level pitch
    unsigned long long blur_off, blur_frame_stride;
    // FAST cell grid (src/ORBextractor.cc:873-886)
    int nCols, nRows, wCell, hCell;
    int cell_base;            // first global cell id of this level (cells of all levels are numbered consecutively)
    int cell_cap;             // staging slots per cell = ceil(wCell/2)*ceil(hCell/2)
    unsigned long long cand_off;      // u32 offset of this level's staging slab inside one frame's staging area
    int cand_max;             // nCols*nRows*cell_cap
    unsigned long long oct_off;       // u32 offset of this level's octree scratch inside one frame's scratch area
    // octree
    int nfeat;                // mnFeaturesPerLevel[level]
    int nIni;                 // round(width/height)
    float hX;                 // width / nIni
    int depth;                // quadtree depth needed to separate distinct pixels
    int root_bits;
    int kp_base;              // first slot of this level in the per-frame level-keypoint arrays
    int kp_cap;               // nfeat + 4
    // resize tables (device pointers): entry = {src offset, a0 | a1<<16}
    const uint2* xtab;        // [w + 2*19 + pad] indexed by bordered column
    const uint2* ytab;        // [h + 2*19] indexed by bordered row
    int area2x;               // 1 if this level is an exact 2x decimation (OpenCV INTER_AREA fast path)
    float scale;              // mvScaleFactor[level]
    float inv_scale;          // mvInvScaleFactor[level]
    float kp_size;            // (float)(int)(31*scale)
    int tma_box_w, tma_box_h; // box of THIS level's resize-source descriptor (when it is the source of level+1)
    int rp_box_w, rp_box_h;   // the same for the warp-streaming resize kernel (128-column x 16-row items of the BORDERED level + 1); 0 = not applicable
    // tables of the warp-streaming resize kernel for THIS level as the destination (api.cu: configure)
    const uint2* rp_xlane;    // [column tile][lane] 32-byte records: a0..a3 | selA + selB << 16, qA + qB << 16 | keep mask, box start column
    const uint2* rp_ysched;   // [strip][rp_box_h + 1] 16-byte records: {first source row, rows in the box, 0, 0}, then per pair of source rows {b0, b1, out rows, 0}
};

struct FrameGeom {
    int nlevels;
    int rows, cols;
    int total_cells;          // per frame
    int kp_slots;             // per frame = sum kp_cap
    unsigned long long cand_frame_stride;  // u32 per frame
    unsigned long long oct_frame_stride;   // u32 per frame
    int iniTh, minTh;
    const uint32_t* cell_tab;  // [total_cells] level | cell_row << 4 | cell_col << 16   (device)
    LevelGeom L[kMaxLevels];
};

// Device workspace pointers of one extractor (one "slot").
struct Workspace {
    uint8_t* pyr;             // bordered pyramid, [level][frame][rows_alloc][pitch]
    uint8_t* blur;            // blurred levels
    uint32_t* cand;           // per-cell candidate staging (packed x | y<<12 | score<<24, window-relative)
    int* cell_count;          // [frame][total_cells]
    uint32_t* oct;            // octree scratch
    uint32_t* lvl_kp;         // [frame][kp_slots] packed retained keypoints (window-relative)
    int* lvl_n;               // [frame][nlevels]
    float* lvl_angle;         // [frame][kp_slots]
    uint8_t* lvl_desc;        // [frame][kp_slots][32]
    int* lvl_ncand;           // [frame][nlevels] number of FAST candidates (probe)
    long long* dbg;           // optional octree phase timing (nullptr in production)
    const CUtensorMap* tmap_resize;   // [nlevels] TMA descriptors of the pyramid levels, box = resize source window (or nullptr)
    const CUtensorMap* tmap_blur;     // [nlevels] TMA descriptors of the pyramid levels, box = blur input tile (or nullptr)
    const CUtensorMap* tmap_rpipe;    // [nlevels] TMA descriptors of the pyramid levels, box = source window of pyr_resize_pipe_kernel (or nullptr)
    const CUtensorMap* tmap_desc;     // [nlevels] TMA descriptors of the BLURRED levels, box = the 64 x 40 window around a keypoint's rBRIEF patch (or nullptr)
    int dbg_level;
};

inline __host__ __device__ uint8_t* level_interior(uint8_t* pyr, const LevelGeom& g, int frame)
{
    return pyr + g.pyr_off + (unsigned long long)frame * g.pyr_frame_stride + (unsigned long long)kEdge * g.pitch + kXPad;
}
inline __host__ __device__ const uint8_t* level_interior(const uint8_t* pyr, const LevelGeom& g, int frame)
{
    return pyr + g.pyr_off + (unsigned long long)frame * g.pyr_frame_stride + (unsigned long long)kEdge * g.pitch + kXPad;
}

// ---- TMA / mbarrier helpers (sm_90+ PTX; SASS: UTMALDG, SYNCS) ----------------------------------------------------------
#if defined(__CUDACC__)
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(bar);
    uint32_t ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
}
// 3-D tiled load: coordinates (byte column, row, frame) of the bordered level buffer; out-of-range elements are zero-filled
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z)
{
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(map), "r"(x), "r"(y), "r"(z),
                 "r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
}
// c += A . B, int8 MMA m16n8k32 (u8 x u8 -> s32; SASS IMMA.16832.U8.U8).  PTX fragment layout, g = lane / 4, t = lane % 4:
// a[q] = A row g + 8 (q & 1), k = 16 (q >> 1) + 4 t + byte;  b0 / b1 = B k = 4 t + byte / + 16, n = g;
// c0, c1 = C row g, n = 2 t, 2 t + 1;  c2, c3 = row g + 8.
__device__ __forceinline__ void imma_16832_u8(int (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
#endif

// Where the frames of a chunk read their image and write their results.  The frames form one or two sets: frames [0, split)
// are set 0, frames [split, n) set 1, and frame f is element f - (set ? split : 0) of its set.  A mono batch is one set
// (split >= n); a stereo chunk of P pairs has split = P: the pairs' left images, then their right images, each side read
// from and written to the caller's own arrays.
// (Named fields and selects, not [2] arrays: a dynamically indexed kernel parameter is copied to the stack.)
struct ChunkIO {
    const uint8_t* img0; const uint8_t* img1;  // frame i of a set: img + i * frame_stride, `pitch` bytes per row
    size_t frame_stride, pitch;
    orbx_keypoint* kps0; orbx_keypoint* kps1;  // [capacity] rows per frame
    uint8_t* desc0; uint8_t* desc1;            // [capacity][32] per frame
    int* n_out0; int* n_out1; int* n_mono0; int* n_mono1;   // one count per frame
    int capacity;
    int split;
    __host__ __device__ size_t index(int f) const { return (size_t)(f >= split ? f - split : f); }
    __host__ __device__ const uint8_t* image(int f) const { return (f >= split ? img1 : img0) + index(f) * frame_stride; }
    __host__ __device__ orbx_keypoint* kps(int f) const { return (f >= split ? kps1 : kps0) + index(f) * capacity; }
    __host__ __device__ uint8_t* desc(int f) const { return (f >= split ? desc1 : desc0) + index(f) * capacity * 32; }
    __host__ __device__ int* n_out(int f) const { return (f >= split ? n_out1 : n_out0) + index(f); }
    __host__ __device__ int* n_mono(int f) const { return (f >= split ? n_mono1 : n_mono0) + index(f); }
};
inline ChunkIO one_set_io(const uint8_t* images, size_t frame_stride, size_t pitch, orbx_keypoint* kps, uint8_t* desc, int capacity,
                          int* n_out, int* n_mono)
{
    ChunkIO io{};
    io.img0 = io.img1 = images; io.frame_stride = frame_stride; io.pitch = pitch;
    io.kps0 = io.kps1 = kps; io.desc0 = io.desc1 = desc; io.n_out0 = io.n_out1 = n_out; io.n_mono0 = io.n_mono1 = n_mono;
    io.capacity = capacity; io.split = 1 << 30;
    return io;
}

// ---- launchers (defined in the kernel translation units) ---------------------------------------------------
void count_launch(int n = 1);

cudaError_t launch_pyramid(const FrameGeom& fg, const Workspace& ws, const ChunkIO& io, int n_frames, cudaStream_t st, int level_lo = 0,
                           int level_hi = 0);
cudaError_t launch_cvt_gray(const uint8_t* d_src, size_t src_pitch, size_t src_frame_stride, int channels, int rgb, int n_frames,
                            int rows, int cols, uint8_t* d_dst, size_t dst_pitch, size_t dst_frame_stride, cudaStream_t st);
cudaError_t launch_fast(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st, int level_lo = 0, int level_hi = 0);
cudaError_t launch_blur(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st);
cudaError_t launch_octree(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st, int level_lo = 0, int level_hi = 0);
cudaError_t launch_orient_describe(const FrameGeom& fg, const Workspace& ws, int n_frames, cudaStream_t st, int lap0, int lap1,
                                   const ChunkIO& io, bool* fused);
cudaError_t launch_pack(const FrameGeom& fg, const Workspace& ws, int n_frames, int lap0, int lap1, const ChunkIO& io, cudaStream_t st);
size_t octree_smem_for(const FrameGeom& fg, int level_lo, int level_hi);   // dynamic shared memory of octree_kernel for these levels
int octree_take_error_flag();   // depth-overflow flag of the current device (duplicate pixels); reading clears it; synchronises
cudaError_t octree_prepare();   // opt in to large dynamic shared memory

cudaError_t launch_knn2(const uint8_t* d_q, int nq, const uint8_t* d_db, long long ndb, int index_base, int32_t* d_idx,
                        int32_t* d_dist, cudaStream_t st, void* workspace = nullptr);
size_t knn2_workspace_bytes(int nq, long long ndb);
cudaError_t launch_knn2_merge(const int32_t* d_idx_sh, const int32_t* d_dist_sh, int n_shards, int nq, int32_t* d_idx,
                              int32_t* d_dist, cudaStream_t st, size_t shard_stride = 0);   // stride in int32 elements, 0 = 2 * nq
cudaError_t launch_popc_bench(unsigned long long* d_sink, int iters, int blocks, cudaStream_t st);

// Frame::ComputeStereoMatches over n_pairs pairs (blockIdx.y of the match kernel, blockIdx.x of the median kernel).  Pair p
// reads pyramid frames frameL + p / frameR + p, keypoints / descriptors at row p * nL (left) and p * nR (right), counts
// d_nL[p] / d_nR[p], and writes rows p * nL of uRight / depth / sad.
struct StereoArgs {
    const uint8_t* pyrL; const uint8_t* pyrR;       // pyramid allocations: same level sizes and pitches, but each extractor lays its
    unsigned long long offR[kMaxLevels];            // level slabs out for its own slot capacity -> the right pyramid's level offsets
    int frameL, frameR;
    int n_pairs;
    const orbx_keypoint* kpL; const uint8_t* descL; int nL;      // nL / nR: counts, or (with d_nL / d_nR) the capacity bound
    const orbx_keypoint* kpR; const uint8_t* descR; int nR;
    const int* d_nL; const int* d_nR;               // optional device-resident counts (results of an extraction still in flight)
    float bf, maxD;
    float* uRight; float* depth;                    // [n_pairs][nL]
    int* sad;                                       // [n_pairs][nL] scratch: SAD of accepted matches, -1 otherwise
};
cudaError_t launch_stereo(const FrameGeom& fg, const StereoArgs& a, cudaStream_t st);

// ---- bag-of-words / vocabulary-guided matching (kernels_bow.cu, api_bow.cu) ---------------------------------------------
struct VocabDev {
    const int* child_begin;      // [n_nodes] first child slot of a node
    const int* child_count;      // [n_nodes] 0 for leaves
    const int* child_id;         // [n_nodes - 1] node id of a child slot (children of a node are contiguous slots)
    const uint8_t* cdesc;        // [n_nodes - 1][32] descriptor of a child slot
    const int* word_of_node;     // [n_nodes] word id of a leaf, -1 otherwise
    const double* weight;        // [n_nodes]
};
cudaError_t launch_bow_descend(const VocabDev& v, const uint8_t* d_desc, int n, int nid_level, uint32_t* d_word, double* d_weight,
                               uint32_t* d_node, cudaStream_t st);

// SearchByBoW of one fixed side against many key frames.  Mode 0 (KF -> Frame, src/ORBmatcher1.cc:225-427): the fixed side is B
// and each key frame an A side; mode 1 (KF -> KF, src/ORBmatcher2.cc:36-171): the fixed side is A and each key frame a B side.
// A job-build kernel (one CTA per key frame) sets key frame k's rows to -1 and writes its common nodes as jobs into
// jobs[k * job_stride, k * job_stride + job_count[k]); the search kernel takes the key frame as blockIdx.y.  Feature indices
// inside a key frame are its own (0 .. n - 1); its arrays point into the packed upload, its per-feature rows start at `base`.
struct BowKF {
    const uint8_t* desc; const uint8_t* valid;
    const uint32_t* node_ids; const int32_t* offsets; const uint32_t* indices;   // mFeatVec in CSR form
    int n, n_nodes;
    size_t base;                 // first feature of this key frame in the packed per-feature arrays
};
struct BowBatchArgs {
    int mode;
    int n_kf; const BowKF* kfs;
    int n; const uint8_t* desc; const uint8_t* valid;                          // the fixed side (valid: mode 1 only)
    int n_nodes; const uint32_t* node_ids; const int32_t* offsets; const uint32_t* indices;
    int nleft;                   // mode 0: F.Nleft (separate left / right best for j < nleft and j >= nleft), else -1
    float nn_ratio;
    int4* jobs;                  // [n_kf][job_stride] (a_begin, a_end, b_begin, b_end) into the A / B index arrays
    int* job_count;              // [n_kf]
    int job_stride;              // n_nodes of the fixed side: a key frame has at most that many common nodes
    int* row;                    // [n_kf][n] per feature of the fixed side: mode 0 match_b (also the "already matched" state),
                                 //           mode 1 match_a
    int* feat;                   // [sum n] per key-frame feature: mode 1 match_b (vbMatched2), mode 0 match_a (may be null)
    int* feat_right;             // [sum n] mode 0 with nleft >= 0: match_a of the right camera (may be null)
};
cudaError_t launch_search_by_bow_batch(const BowBatchArgs& a, cudaStream_t st);

// SearchForTriangulation of one KF1 against many neighbours: a job-build kernel (one CTA per neighbour) writes the jobs of
// neighbour k into jobs[k * n_a, k * n_a + job_count[k]) and sets match row k to -1; the scan kernel takes the neighbour as
// blockIdx.y.  Feature indices inside a neighbour are its own (0 .. n - 1); its arrays point into the packed upload.
struct TriKF {
    const orbx_keypoint* kp; const uint8_t* desc; const uint8_t* free; const uint8_t* stereo;
    const uint32_t* node_ids; const int32_t* offsets; const uint32_t* indices;   // mFeatVec in CSR form
    int n, n_nodes, coarse, pad;
    float F12[9]; float ep[2]; float scale[kMaxLevels]; float sigma2[kMaxLevels];
};
struct TriBatchArgs {
    int n_kf; const TriKF* kfs;
    int n_a; const orbx_keypoint* kp_a; const uint8_t* desc_a; const uint8_t* free_a; const uint8_t* stereo_a;
    int a_nodes; const uint32_t* a_node_ids; const int32_t* a_offsets; const uint32_t* a_indices;
    int only_stereo;
    int4* jobs;                  // [n_kf][n_a] (iA, b_begin, b_end, 0), b_* into the neighbour's indices
    int* job_count;              // [n_kf]
    int* match;                  // [n_kf][n_a]
};
cudaError_t launch_search_triangulation_batch(const TriBatchArgs& a, cudaStream_t st);


// ---- frame grid + projection-guided window searches (kernels_proj.cu, api_proj.cu) ----------------------------------------
enum { PROJ_Q_VALID = 1, PROJ_Q_CHECK_RIGHT = 2, PROJ_Q_TAKES = 4 };
struct ProjQuery {               // one GetFeaturesInArea window + what the scan needs (32 bytes)
    float x, y, r;               // window centre and half size (already multiplied by the level's scale factor)
    float ur;                    // predicted right-image coordinate for the mvuRight gate (PROJ_Q_CHECK_RIGHT)
    int min_level, max_level;    // GetFeaturesInArea minLevel / maxLevel (-1 = open)
    int flags;                   // PROJ_Q_*: VALID = passes the reference's pre-checks; TAKES = the assigned map point has Observations() > 0
    int pad;
};
struct ProjArgs {
    int n;                       // features of the frame
    const orbx_keypoint* kp; const uint8_t* desc; const float* u_right;   // u_right may be null
    float min_x, min_y, grid_w_inv, grid_h_inv;
    int* cell_start;             // [64*48 + 1] CSR over cell id = ix * 48 + iy
    int* items;                  // [n] feature indices by cell, ascending inside a cell
    unsigned short* cell_of;     // [n] cell id or 0xffff
    int* taken_by;               // [n] INT_MAX = free, -1 = holds an observed map point on entry, else the query that took it
    int* claim;                  // [n] least undecided query index that could take the feature
    int nq; const ProjQuery* q; const uint8_t* qdesc;
    int mode;                    // 0: best/second + level-aware ratio (ORBmatcher1.cc:45-215); 1: 1-NN (ORBmatcher3.cc:256-578);
                                 // 2: SearchForInitialization (ORBmatcher1.cc:650-765): vMatchedDistance skip, no level test in the ratio
    int th_dist; float nn_ratio;
    unsigned long long* keys;    // [nq][2] top-2 (distance << 48 | cell << 32 | index)
    int* qmatch;                 // [nq] init -1: feature assigned to the query
    int* list_a; int* list_b;    // [nq] undecided queries, ping-pong
    int* rounds_out;             // speculation rounds used (diagnostics; may be null)
    // mode 2: the acceptances of each feature as a chain, newest first (vMatchedDistance as every query sees it)
    int* last_acc;               // [n] latest query that accepted the feature, -1 = none (null outside mode 2)
    int* prev_acc;               // [nq] the acceptance of the same feature before this query's, -1 = none
    int* acc_dist;               // [nq] the distance this query accepted at
};
cudaError_t launch_frame_grid(const ProjArgs& a, cudaStream_t st);
cudaError_t launch_proj_search(const ProjArgs& a, cudaStream_t st);
// ORBmatcher::Fuse (ORBmatcher2.cc:420-610) over many key frames: one grid per key frame, one warp per (key frame, point) pair.
// The Sim3 Fuse (ORBmatcher2.cc:612-729) runs the same launch without the reprojection gate (u_right / inv_sigma2 unused).
struct FuseKF {                  // one key frame on the device
    const orbx_keypoint* kp; const uint8_t* desc; const float* u_right;   // u_right null = monocular (mvuRight all -1)
    int n;
    float min_x, min_y, grid_w_inv, grid_h_inv;
    int* cell_start;             // [64*48 + 1]
    int* items;                  // [n]
    unsigned short* cell_of;     // [n]
    float inv_sigma2[kMaxLevels];   // mvInvLevelSigma2
};
struct FuseQuery {               // one pair that passed the caller's pre-checks and IsInImage (32 bytes)
    float u, v, r, ur;           // projection, window half size th * mvScaleFactors[level], ur = u - bf * invz
    int kf, point, level, pad;
};
struct FuseArgs {
    int n_kf; const FuseKF* kfs;
    int nq; const FuseQuery* q;
    const uint8_t* pdesc;        // [n_desc][32] map point descriptors, indexed by FuseQuery::point
    int th_dist;                 // TH_LOW
    int* match;                  // [nq] bestIdx or -1
};
cudaError_t launch_fuse(const FuseArgs& a, bool reproj_gate, cudaStream_t st);   // reproj_gate = false: the Sim3 Fuse
cudaError_t launch_features_in_area(const ProjArgs& a, float x, float y, float r, int min_level, int max_level,
                                    unsigned long long* d_out, int capacity, int* d_n_out, cudaStream_t st);

// ---- preparation steps either side of the extractor (kernels_prep.cu, api_prep.cu) ------------------------------------------
struct UndistortParams {
    double fx, fy, cx, cy;       // K of the distorted camera
    double nfx, nfy, ncx, ncy;   // P = new camera matrix (mK)
    double k[14];                // k1 k2 p1 p2 k3 k4 k5 k6 s1..s4 (tilt unused); missing = 0
    int n_dist;
};
cudaError_t launch_undistort(const orbx_keypoint* d_in, int n, const UndistortParams& p, orbx_keypoint* d_out, cudaStream_t st);
// mvKeysUn + ComputeStereoFromRGBD of n_frames frames.  Frame f: counts n[f], keypoint rows f * capacity of kp / kp_un / uRight /
// depth_out, depth map at depth + f * depth_frame_stride (depth_pitch bytes per row, u16 or f32 elements).
struct RgbdArgs {
    const orbx_keypoint* kp; const int* n; int capacity;
    orbx_keypoint* kp_un; float* uRight; float* depth_out;
    const uint8_t* depth; size_t depth_pitch, depth_frame_stride;
    int depth_type;              // 0: CV_16U, 1: CV_32F
    int convert;                 // GrabImageRGBD's predicate, evaluated on the host: multiply the sample by `factor`
    float factor, bf;
    int undistort;               // 0: mvKeysUn = mvKeys (mDistCoef[0] == 0, src/Frame.cc:779-783)
    UndistortParams p;
};
cudaError_t launch_rgbd_frame(const RgbdArgs& a, int n_frames, cudaStream_t st);
cudaError_t launch_remap_quantise(const float* d_mapx, const float* d_mapy, size_t map_step, int dw, int dh, uint2* d_packed, cudaStream_t st);
cudaError_t launch_remap(const uint8_t* d_src, int sw, int sh, size_t spitch, size_t sframe, const uint2* d_packed, uint8_t* d_dst, int dw,
                         int dh, size_t dpitch, size_t dframe, int n_frames, cudaStream_t st);
cudaError_t launch_resize(const uint8_t* d_src, size_t spitch, size_t sframe, const uint2* d_xtab, const uint2* d_ytab, int area2x,
                          uint8_t* d_dst, int dw, int dh, size_t dpitch, size_t dframe, int n_frames, cudaStream_t st);

// Per-device grow-only scratch of every call that takes host buffers (api.cu): device memory, a pinned staging buffer and a
// non-blocking stream.  One call = one Lease: a bump allocator that hands out matching (pinned host, device) ranges so that all
// inputs travel in one cudaMemcpyAsync.  Inputs are allocated first (the upload range), device-only scratch and outputs after.
// The call queues everything on A.st and ends with one cudaStreamSynchronize(A.st), so the arena is idle whenever it is leased.
// Each thread of an ORB-SLAM3 system has its own set, so a call never waits for another thread's lock or work.
struct ProjArena {
    std::mutex mu;
    unsigned char* d = nullptr; size_t d_bytes = 0;
    unsigned char* h = nullptr; size_t h_bytes = 0;
    cudaStream_t st = nullptr;
};
// tracking: the Frame / KF->Frame searches, orbx_knn2, orbx_stereo_match, orbx_undistort_keypoints, orbx_bow_transform,
// orbx_search_by_bow mode 0
extern ProjArena g_arena[64];
// local mapping: orbx_fuse, orbx_search_for_triangulation(_batch), orbx_distinctive_descriptors
extern ProjArena g_fuse_arena[64];
// loop closing: the Sim3 searches, orbx_search_by_bow mode 1
extern ProjArena g_loop_arena[64];
struct Lease {
    ProjArena& A;
    std::unique_lock<std::mutex> lock;
    size_t off = 0, upload_end = 0;
    explicit Lease(int device, ProjArena* arenas = g_arena) : A(arenas[device & 63]), lock(A.mu) {}
    // Device bytes for the whole layout; only its first `staged` bytes have a pinned host mirror (a large device-only tail, such
    // as orbx_knn2's database, is not pinned twice).
    int reserve(size_t bytes, size_t staged = SIZE_MAX);
    template <typename T> size_t take(size_t count)
    {
        off = (off + 255) & ~(size_t)255;
        const size_t o = off;
        off += (count > 1 ? count : 1) * sizeof(T);
        return o;
    }
    template <typename T> T* dev(size_t o) const { return reinterpret_cast<T*>(A.d + o); }
    template <typename T> T* host(size_t o) const { return reinterpret_cast<T*>(A.h + o); }
};
inline size_t lease_pad(size_t bytes) { return ((bytes + 255) & ~(size_t)255) + 256; }   // bytes of one take() in reserve()

// host helpers shared by api.cu / api_bow.cu / api_proj.cu
int fail(int code, const char* fmt, ...);
int set_device(int device);
void three_maxima(const int* count, int L, int& ind1, int& ind2, int& ind3);   // ORBmatcher::ComputeThreeMaxima (src/ORBmatcher3.cc:592-633)
int rotation_bin(float angle_a, float angle_b);                                 // src/ORBmatcher1.cc:344-351; -1 if out of range

cudaError_t launch_synth_images(uint32_t seed0, int view, int n_frames, int cols, int rows, int max_disp, uint8_t* d_dst,
                                size_t pitch, size_t frame_stride, cudaStream_t st);
cudaError_t launch_synth_desc(uint32_t seed, int is_query, long long first_row, long long n_rows, long long ndb,
                              int plant_every, uint8_t* d_dst, cudaStream_t st);

}  // namespace orbx
