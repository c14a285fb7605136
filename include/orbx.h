/* orbx.h — C ABI of the B200-native ORB front end (liborbx.so).
 *
 * Drop-in boundary for the hot path of kpmrozowski/wut-cuda-orb-slam3 (an ORB-SLAM3 v1.0 fork):
 * ORB_SLAM3::ORBextractor (pyramid -> FAST -> octree -> orientation -> blur -> rBRIEF -> packing),
 * ORBmatcher::DescriptorDistance / brute-force 2-NN Hamming matching, and Frame::ComputeStereoMatches.
 * The reference has no FFI layer (the boundary is a C++ class linked into libORB_SLAM3.so), so the entry
 * points below are what a maintainer's thin C++ adapter binds; the adapter with the reference's exact
 * signatures is wut_cuda_orb_slam3_b200/csrc/adapter/ORBextractor.h (see INTEGRATION.md).
 *
 * Every entry point cites the reference interface it replaces (paths relative to the reference root).
 * POD only: plain pointers and sizes, no OpenCV / torch types.  All functions return ORBX_OK (0) or a
 * negative orbx_status; none aborts the process (the reference exit(1)s on OpenCL init failure,
 * src/OpenCL/Manager.cpp:13-20, and throws on launch failure, src/ORBextractor.cc:498,861,973,1212).
 * There is NO CPU fallback: compute entry points fail with ORBX_ERR_NO_DEVICE without a CUDA device.
 *
 * Threading: one extractor handle is used by one thread at a time; different handles may be used
 * concurrently (the reference runs the left/right extractors on two std::threads, src/Frame.cc:124-127).
 */
#ifndef ORBX_H_
#define ORBX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ORBX_VERSION 100 /* 0.1.0 */
#define ORBX_MAX_LEVELS 16
#define ORBX_EDGE_THRESHOLD 19 /* src/ORBextractor.cc:101 */
#define ORBX_DESC_BYTES 32

typedef enum orbx_status {
    ORBX_OK = 0,
    ORBX_ERR_EMPTY_IMAGE = -1, /* ORBextractor::operator() returns -1 on an empty image (src/ORBextractor.cc:1231-1232) */
    ORBX_ERR_INVALID_ARG = -2,
    ORBX_ERR_NO_DEVICE = -3,
    ORBX_ERR_CUDA = -4,
    ORBX_ERR_CAPACITY = -5,    /* caller's output buffer too small; *n_out holds the needed count */
    ORBX_ERR_UNSUPPORTED = -6, /* image larger than 4128 px per side, > ORBX_MAX_LEVELS levels, ... */
    ORBX_ERR_OOM = -7
} orbx_status;

/* cv::KeyPoint == key_point_t, 28-byte POD (include/OpenCL/Kernel/key_point.hpp:22-29; the reference relies on
 * the reinterpret-cast equivalence at src/ORBextractor.cc:839-841). */
typedef struct orbx_keypoint {
    float x, y;      /* pt, in level-0 pixel coordinates */
    float size;      /* (float)(int)(31 * mvScaleFactor[octave]) */
    float angle;     /* degrees, [0,360) */
    float response;  /* FAST score */
    int32_t octave;
    int32_t class_id; /* -1 */
} orbx_keypoint;

typedef struct orbx_extractor orbx_extractor; /* opaque; owns a CUDA stream + device workspace */

/* Thread-local description of the last error on the calling thread ("" if none). */
const char* orbx_last_error(void);
int orbx_version(void);
/* Number of visible CUDA devices (0 without a driver/GPU; never fails). */
int orbx_device_count(void);

/* ---- construction / accessors -------------------------------------------------------------------------- */

/* ORBextractor::ORBextractor(nfeatures, scaleFactor, nlevels, iniThFAST, minThFAST) — include/ORBextractor.h:58-59,
 * src/ORBextractor.cc:410-468.  `device` = CUDA ordinal.  max_cols/max_rows/max_batch pre-size the workspace
 * (0 = size lazily on first use; the workspace grows on demand either way). */
int orbx_create(int nfeatures, float scaleFactor, int nlevels, int iniThFAST, int minThFAST, int device,
                int max_cols, int max_rows, int max_batch, orbx_extractor** out);
void orbx_destroy(orbx_extractor* ex);

/* GetLevels / GetScaleFactor — include/ORBextractor.h:70-74. */
int orbx_get_levels(const orbx_extractor* ex);
float orbx_get_scale_factor(const orbx_extractor* ex);
/* GetScaleFactors / GetInverseScaleFactors / GetScaleSigmaSquares / GetInverseScaleSigmaSquares (include/ORBextractor.h:76-90)
 * plus mnFeaturesPerLevel (src/ORBextractor.cc:436-447).  Any output pointer may be NULL; arrays hold nlevels entries. */
int orbx_get_tables(const orbx_extractor* ex, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2,
                    int* nfeatures_per_level);
/* Same tables without a handle or a GPU (host arithmetic of src/ORBextractor.cc:418-447). */
int orbx_compute_tables(int nfeatures, float scaleFactor, int nlevels, float* scale, float* inv_scale, float* sigma2,
                        float* inv_sigma2, int* nfeatures_per_level);
/* Level size for an input of cols x rows: cvRound(cols * mvInvScaleFactor[level]) (src/ORBextractor.cc:1312-1313). */
int orbx_level_size(const orbx_extractor* ex, int cols, int rows, int level, int* level_cols, int* level_rows);
/* Upper bound on keypoints per frame for the shape the handle is configured for (sum over levels of
 * max(mnFeaturesPerLevel + 4, 4 * nIni + 1)); before the first image it cannot know nIni = round(width / height) of
 * DistributeOctTree (src/ORBextractor.cc:589) and returns the sum of mnFeaturesPerLevel + 4 only. */
int orbx_max_keypoints(const orbx_extractor* ex);
/* The same bound for a rows x cols image, from the shape alone (host arithmetic, handle unchanged): size outputs with
 * this.  Wide images matter: the octree's first sweep splits all nIni roots into four before it compares with N. */
int orbx_max_keypoints_for(const orbx_extractor* ex, int rows, int cols);

/* ---- extraction ------------------------------------------------------------------------------------------ */

/* int ORBextractor::operator()(image, mask, keypoints, descriptors, vLappingArea) — include/ORBextractor.h:66-68,
 * src/ORBextractor.cc:1227-1307.  image: CV_8UC1 rows x cols, `step` bytes per row, HOST memory.  (lap0, lap1) =
 * vLappingArea.  Writes *n_out keypoints (28 B) + descriptors (32 B) in the reference's packing order (non-lapping
 * from the front, lapping from the back) and *n_mono = the reference's return value (monoIndex).
 * `capacity` = room in keypoints / descriptors, sized with orbx_max_keypoints_for(ex, rows, cols); a frame with more
 * keypoints than that fails with ORBX_ERR_CAPACITY and writes nothing past the buffers.
 * Returns ORBX_ERR_EMPTY_IMAGE for a NULL/empty image. */
int orbx_extract(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int lap0, int lap1,
                 orbx_keypoint* keypoints, uint8_t* descriptors, int capacity, int* n_out, int* n_mono);

/* Image prep of Tracking::GrabImageStereo / GrabImageMonocular / GrabImageRGBD (src/Tracking2.cc:289-316, 347-361, 392-406):
 * cv::cvtColor(im, im, COLOR_{RGB,BGR,RGBA,BGRA}2GRAY) chosen by the channel count and mbRGB, fused in front of operator():
 * `image` is a HOST rows x cols image of `channels` (3 or 4) interleaved 8-bit channels, `rgb` != 0 means channel 0 is red
 * (mbRGB).  8U arithmetic of OpenCV: (R*9798 + G*19235 + B*3735 + 2^14) >> 15.  The grey image is level 0 of the pyramid
 * (orbx_get_pyramid_level) — the reference keeps it as mImGray. */
int orbx_extract_color(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int channels, int rgb, int lap0,
                       int lap1, orbx_keypoint* keypoints, uint8_t* descriptors, int capacity, int* n_out, int* n_mono);
/* The conversion alone on device-resident frames (frame f at d_src + f*src_frame_stride, src_pitch bytes per row). */
int orbx_cvt_gray_device(int device, const uint8_t* d_src, size_t src_pitch, size_t src_frame_stride, int channels, int rgb,
                         int n_frames, int rows, int cols, uint8_t* d_dst, size_t dst_pitch, size_t dst_frame_stride, void* stream);

/* Batched operator(): n_frames HOST images of identical shape (images[i] -> rows x cols, `step` bytes per row).
 * Outputs are [n_frames][capacity] slabs; n_out / n_mono are [n_frames].  Host<->device copies are pipelined
 * against compute when the host buffers are page-locked. */
int orbx_extract_batch(orbx_extractor* ex, const uint8_t* const* images, int n_frames, int rows, int cols, size_t step,
                       int lap0, int lap1, orbx_keypoint* keypoints, uint8_t* descriptors, int capacity, int* n_out,
                       int* n_mono);

/* Device-resident batched operator(): frame f starts at d_images + f*frame_stride, `pitch` bytes per row; all
 * output pointers are DEVICE memory with the same slab layout.  Asynchronous on `stream` (a cudaStream_t, or NULL
 * for the extractor's own stream).  orbx_sync waits for it whichever stream was used (an event is recorded behind the last
 * launch), and so do the probes, orbx_stereo_match and the next call on this handle. */
int orbx_extract_batch_device(orbx_extractor* ex, const uint8_t* d_images, size_t frame_stride, int n_frames, int rows,
                              int cols, size_t pitch, int lap0, int lap1, orbx_keypoint* d_keypoints,
                              uint8_t* d_descriptors, int capacity, int* d_n_out, int* d_n_mono, void* stream);
int orbx_sync(orbx_extractor* ex);

/* std::vector<cv::Mat> mvImagePyramid (include/ORBextractor.h:92), read by Frame::ComputeStereoMatches
 * (src/Frame.cc:848,938-953): lazy device->host copy of one level of frame `frame` of the LAST call.
 * with_border = 0: interior (level_rows x level_cols); 1: the whole (rows+38) x (cols+38) bordered buffer. */
int orbx_get_pyramid_level(orbx_extractor* ex, int frame, int level, uint8_t* dst, size_t dst_step, int with_border);

/* The same member kept current without a blocking copy per level: with the mirror enabled every orbx_extract also sends the
 * bordered levels to pinned host storage owned by the handle, level by level on a copy branch that overlaps FAST, the octree
 * and the descriptors (the call returns when everything has arrived).  orbx_get_pyramid_mirror hands out the storage of one
 * level: `bordered` = top-left of the (rows + 38) x (cols + 38) buffer, `step` bytes per row; the interior (the cv::Mat of
 * mvImagePyramid[level]) starts at bordered + 19 * step + 19.  Valid until the next call on the handle. */
int orbx_set_pyramid_mirror(orbx_extractor* ex, int enable);
int orbx_get_pyramid_mirror(orbx_extractor* ex, int level, const uint8_t** bordered, size_t* step, int* level_cols, int* level_rows);

/* Stage probes for parity tests (results of the LAST call, copied to host):
 *  blurred level (cv::GaussianBlur 7x7 sigma 2, src/ORBextractor.cc:1270-1273),
 *  FAST candidates handed to DistributeOctTree (vToDistributeKeys, src/ORBextractor.cc:867-950; window-relative),
 *  per-level keypoints after octree + orientation (allKeypoints[level], level coordinates) and their descriptors. */
int orbx_get_blurred_level(orbx_extractor* ex, int frame, int level, uint8_t* dst, size_t dst_step);
int orbx_get_candidates(orbx_extractor* ex, int frame, int level, int* xs, int* ys, int* scores, int capacity);
int orbx_get_level_keypoints(orbx_extractor* ex, int frame, int level, orbx_keypoint* keypoints, uint8_t* descriptors,
                             int capacity);

/* Stand-alone DistributeOctTree (src/ORBextractor.cc:584-774) on host candidate arrays, run on the GPU kernel:
 * returns in out_idx the indices (into the input) of the retained keypoints in the reference's output order. */
int orbx_distribute_octree(int device, const int* xs, const int* ys, const int* scores, int n, int minX, int maxX,
                           int minY, int maxY, int nFeatures, int* out_idx, int capacity, int* n_out);

/* ---- matching -------------------------------------------------------------------------------------------- */

/* static int ORBmatcher::DescriptorDistance(a, b) — include/ORBmatcher.h:43, src/ORBmatcher3.cc:637-653.
 * Host inline popcount (a GPU launch per pair would be absurd); pure and re-entrant. */
int orbx_descriptor_distance(const uint8_t* a, const uint8_t* b);

/* Brute-force 2-NN (cv::BFMatcher(NORM_HAMMING).knnMatch(k=2), src/Frame.cc:45,1174; identical (d1,i1,d2) to the
 * strict-'<' best/second scan of src/ORBmatcher1.cc:283-300 and src/ORBmatcher2.cc:84-118 over the whole set).
 * HOST buffers; idx/dist are [nq][2], ascending distance, ties -> lower database index; missing = (-1, INT32_MAX).  Uses the
 * tracking thread's device scratch; the database is copied straight from `database` (it is not staged in pinned memory). */
int orbx_knn2(int device, const uint8_t* queries, int nq, const uint8_t* database, int64_t ndb, int32_t* idx,
              int32_t* dist);
/* Device-resident variant on `stream`; database rows are numbered index_base + row (for sharded databases).  Re-entrant:
 * scratch is a stream-ordered allocation private to the call, so Tracking / LocalMapping / LoopClosing threads (all of which
 * match descriptors, src/ORBmatcher3.cc:637-653 callers) may run it concurrently on their own streams. */
int orbx_knn2_device(int device, const uint8_t* d_queries, int nq, const uint8_t* d_database, int64_t ndb,
                     int32_t index_base, int32_t* d_idx, int32_t* d_dist, void* stream);
/* Merge per-shard 2-NN candidates (e.g. after an NCCL all-gather): inputs [n_shards][nq][2]; lexicographic
 * (distance, index) order reproduces the single-GPU / BFMatcher tie rule exactly. */
int orbx_knn2_merge_device(int device, const int32_t* d_idx_shards, const int32_t* d_dist_shards, int n_shards, int nq,
                           int32_t* d_idx, int32_t* d_dist, void* stream);

/* ---- database-sharded 2-NN over several GPUs (BASELINE config 5; SURVEY.md §8(b) "a sharded variant taking an
 * ncclComm_t/rank/world", §8(e)) --------------------------------------------------------------------------------------------
 * The reference's brute-force matcher (cv::BFMatcher(NORM_HAMMING).knnMatch(k=2) + the ratio test, src/Frame.cc:45, 1174-1181)
 * on a database too large for one GPU: queries replicated, database rows split in contiguous shards (orbx_shard_rows), one
 * process per GPU.  NCCL is bound at run time (the copy already loaded into the process, else libnccl.so.2 / $ORBX_NCCL_LIB). */
typedef struct orbx_comm orbx_comm;
#define ORBX_COMM_ID_BYTES 128
/* ncclGetUniqueId: call on one rank, hand the 128 bytes to every rank by any means (MPI, torch.distributed, a file). */
int orbx_comm_unique_id(uint8_t id[ORBX_COMM_ID_BYTES]);
/* ncclCommInitRank on `device`; collective: every rank of `world` must call it with the same id. */
int orbx_comm_create(int device, int rank, int world, const uint8_t id[ORBX_COMM_ID_BYTES], orbx_comm** out);
/* Wrap a communicator the caller already owns (an ncclComm_t from the SAME libnccl the process has loaded); not destroyed by
 * orbx_comm_destroy. */
int orbx_comm_from_nccl(int device, void* nccl_comm, int rank, int world, orbx_comm** out);
void orbx_comm_destroy(orbx_comm* comm);
int orbx_comm_info(const orbx_comm* comm, int* rank, int* world, int* nccl_version);
/* The contiguous shard [first, first + count) of n_rows that `rank` of `world` owns (trailing shards may be empty). Host. */
void orbx_shard_rows(int64_t n_rows, int world, int rank, int64_t* first, int64_t* count);
/* One collective call per rank: d_db_shard holds rows [first_row, first_row + n_shard_rows) of the global database; every rank
 * passes the same nq queries.  On return (asynchronously on `stream`) EVERY rank's d_idx / d_dist [nq][2] hold the 2-NN over the
 * whole database with GLOBAL row indices: local scan, ONE ncclAllGather of the packed 16 B / query candidates, lexicographic
 * (distance, index) merge = the single-GPU / BFMatcher answer bit for bit.  Calls on one communicator are serialised. */
int orbx_knn2_sharded(orbx_comm* comm, const uint8_t* d_queries, int nq, const uint8_t* d_db_shard, int64_t n_shard_rows,
                      int64_t first_row, int32_t* d_idx, int32_t* d_dist, void* stream);

/* Ratio-test acceptance on 2-NN output, host: mode 0 = src/ORBmatcher1.cc:329-333 (d1 <= th_low && (float)d1 <
 * ratio*(float)d2), mode 1 = src/ORBmatcher2.cc:120-125 (d1 < th_low && ...), mode 2 = src/Frame.cc:1181
 * (d1 < d2 * ratio, no gate).  accept[i] = 0/1. */
int orbx_ratio_test(const int32_t* dist, int nq, float ratio, int th_low, int mode, uint8_t* accept);

/* Rotation-consistency filter applied to accepted matches by SearchByBoW / SearchByProjection (src/ORBmatcher1.cc:344-356
 * histogram of round((angleA-angleB [+360]) * (1/HISTO_LENGTH)) over HISTO_LENGTH=30 bins, src/ORBmatcher1.cc:408-427 removal,
 * ComputeThreeMaxima src/ORBmatcher3.cc:592-633): keep[i] = 1 iff match i falls in one of the (up to) three dominant bins. Host. */
int orbx_rotation_consistency(const float* angle_a, const float* angle_b, int n, uint8_t* keep);

/* MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cc:329-401): N x N Hamming distances, per-row median at index
 * (int)(0.5*(N-1)) of the sorted row, first row with the least median.  Host (N is a handful of observations). */
int orbx_distinctive_descriptor(const uint8_t* descriptors, int n, int* best_idx);

/* The same for MANY map points in one call, on the GPU (one warp per map point): the observations of point p are the
 * descriptors [offsets[p], offsets[p + 1]) of `descriptors` (HOST, rows of 32 bytes; offsets[0] == 0).  best_idx[p] = index
 * INSIDE the point's own list, -1 for a point without observations.  What LocalMapping does point by point after every key
 * frame (src/LocalMapping.cc -> MapPoint::ComputeDistinctiveDescriptors, src/MapPoint.cc:329-401).  Uses local mapping's
 * device scratch. */
int orbx_distinctive_descriptors(int device, const uint8_t* descriptors, const int32_t* offsets, int n_points, int32_t* best_idx);

/* ---- the on-disk form of descriptors and key points (SURVEY.md §8(f)4) --------------------------------------------------
 * serializeMatrix / serializeVectorKeyPoints of include/SerializationUtils.h:76-153 as applied to KeyFrame::mDescriptors,
 * MapPoint::mDescriptor, KeyFrame::mvKeys / mvKeysUn / mvKeysRight (include/KeyFrame.h:120-128, 180, include/MapPoint.h:92) by
 * System::SaveAtlas / LoadAtlas (src/System.cc:1339-1475).  `text` != 0: the primitive stream of a boost text archive
 * (space-separated tokens), else of a boost binary archive (native little-endian).  Only the stream these two helpers emit is
 * produced / parsed — the archive header and class records around it are boost's.  Writers return the stream length (call
 * with dst == NULL to size it); readers return the bytes consumed; negative = orbx_status. */
int64_t orbx_serialize_matrix_u8(int text, const uint8_t* data, int rows, int cols, size_t step, uint8_t* dst, size_t dst_capacity);
int64_t orbx_deserialize_matrix_u8(int text, const uint8_t* src, size_t src_len, int* rows, int* cols, uint8_t* dst, size_t dst_step,
                                   size_t dst_capacity);
int64_t orbx_serialize_keypoints(int text, const orbx_keypoint* kps, int n, uint8_t* dst, size_t dst_capacity);
int64_t orbx_deserialize_keypoints(int text, const uint8_t* src, size_t src_len, int* n_out, orbx_keypoint* kps, int capacity);

/* void Frame::ComputeStereoMatches() — src/Frame.cc:841-1011.  Uses the un-blurred pyramids of frame `frameL` /
 * `frameR` of the LAST calls on exL / exR (which must live on the same device; they may be the same handle) and
 * HOST keypoints/descriptors as returned by orbx_extract.  bf = mbf; maxD = mbf/mb is explicit because the
 * reference reads mb before it is assigned (src/Frame.cc:143 vs 176).  Outputs mvuRight / mvDepth (-1 = no match).  Uses the
 * tracking thread's device scratch. */
int orbx_stereo_match(orbx_extractor* exL, int frameL, orbx_extractor* exR, int frameR, const orbx_keypoint* kpL,
                      const uint8_t* descL, int nL, const orbx_keypoint* kpR, const uint8_t* descR, int nR, float bf,
                      float maxD, float* uRight, float* depth);

/* The same on DEVICE-resident features, asynchronous on `stream`: d_kp* / d_desc* are [cap*] rows as written by
 * orbx_extract_batch_device (or any device copy of orbx_extract's output), *d_nL / *d_nR the device-resident counts (read by the
 * kernel, so the call can be queued behind an extraction that is still running on the same stream); d_uRight / d_depth receive
 * capL floats (rows >= *d_nL are left untouched).  No host round trip, no re-upload. */
int orbx_stereo_match_device(orbx_extractor* exL, int frameL, orbx_extractor* exR, int frameR, const orbx_keypoint* d_kpL,
                             const uint8_t* d_descL, const int* d_nL, int capL, const orbx_keypoint* d_kpR, const uint8_t* d_descR,
                             const int* d_nR, int capR, float bf, float maxD, float* d_uRight, float* d_depth, void* stream);
/* The stereo Frame constructor in one call — src/Frame.cc:124-143: ExtractORB(0, imLeft) and ExtractORB(1, imRight) (two
 * std::threads in the reference, two CUDA streams here, vLappingArea = {0, 0}) followed by ComputeStereoMatches().  HOST images
 * in; HOST keypoints / descriptors of both sides (capacity rows each, *nL / *nR valid), mvuRight / mvDepth [capacity] out.
 * The matcher reads keypoints, descriptors and pyramids where the extractors left them on the device; its outputs and scratch
 * are exL's stereo staging (that of orbx_extract_stereo_batch).  Every argument is checked before any work is queued:
 * capacity >= 2^20 returns ORBX_ERR_UNSUPPORTED with the outputs untouched. */
int orbx_extract_stereo(orbx_extractor* exL, orbx_extractor* exR, const uint8_t* imageL, const uint8_t* imageR, int rows, int cols,
                        size_t step, orbx_keypoint* kpL, uint8_t* descL, int* nL, orbx_keypoint* kpR, uint8_t* descR, int* nR,
                        int capacity, float bf, float maxD, float* uRight, float* depth);

/* orbx_extract_stereo over a batch of rectified pairs of one shape, with ONE handle for both sides: the reference builds its
 * left and right extractors from the same settings, and results depend only on those and the image.  For every pair the
 * outputs equal what orbx_extract_stereo returns for it, bit for bit.  n_pairs HOST pairs imagesL[i] / imagesR[i] (rows x cols,
 * `step` bytes per row).  Outputs are [n_pairs][capacity] slabs: keypoints (28 B), descriptors (32 B) and mvuRight / mvDepth
 * floats; nL / nR are [n_pairs].  Only the first nL[i] rows of a pair's uRight / depth are defined.  Host<->device copies are
 * pipelined against compute when the host buffers are page-locked.
 * n_pairs == 0 returns ORBX_OK and does nothing; n_pairs < 0, a NULL output, capacity <= 0 or step < cols: ORBX_ERR_INVALID_ARG;
 * a NULL image array or image, rows or cols <= 0: ORBX_ERR_EMPTY_IMAGE; capacity >= 2^20: ORBX_ERR_UNSUPPORTED; a pair with more
 * than `capacity` keypoints on either side: ORBX_ERR_CAPACITY (the rows of that pair are undefined; nothing is written past the
 * slabs).
 * The pyramids of a stereo batch are not kept for inspection: afterwards the stage probes, orbx_get_pyramid_level and
 * orbx_stereo_match refuse every frame index (ORBX_ERR_INVALID_ARG) until the next extraction. */
int orbx_extract_stereo_batch(orbx_extractor* ex, const uint8_t* const* imagesL, const uint8_t* const* imagesR, int n_pairs,
                              int rows, int cols, size_t step, float bf, float maxD, orbx_keypoint* kpL, uint8_t* descL, int* nL,
                              orbx_keypoint* kpR, uint8_t* descR, int* nR, int capacity, float* uRight, float* depth);
/* The same on DEVICE-resident pairs: pair i at d_imagesL + i * frame_stride and d_imagesR + i * frame_stride (`pitch` bytes per
 * row); every output is DEVICE memory with the slab layout above.  Asynchronous on `stream` (NULL = the extractor's own):
 * orbx_sync and the next call on the handle wait for it, exactly as for orbx_extract_batch_device.  A pair over capacity is
 * reported only through its device counts (*d_nL / *d_nR > capacity; the rows of that pair are undefined), as in
 * orbx_extract_batch_device.  Rows
 * of d_uRight / d_depth at or past a pair's *d_nL are left untouched. */
int orbx_extract_stereo_batch_device(orbx_extractor* ex, const uint8_t* d_imagesL, const uint8_t* d_imagesR, size_t frame_stride,
                                     int n_pairs, int rows, int cols, size_t pitch, float bf, float maxD, orbx_keypoint* d_kpL,
                                     uint8_t* d_descL, int* d_nL, orbx_keypoint* d_kpR, uint8_t* d_descR, int* d_nR, int capacity,
                                     float* d_uRight, float* d_depth, void* stream);

/* ---- RGB-D frames ------------------------------------------------------------------------------------------------ */

/* What the RGB-D Frame constructor reads besides the images (src/Frame.cc:202-260, Tracking::GrabImageRGBD in src/Tracking2.cc). */
typedef struct orbx_rgbd_calib {
    float K[4];           /* fx, fy, cx, cy = Pinhole::toK() == mK */
    const float* dist;    /* mDistCoef: k1 k2 p1 p2 [k3 [k4 k5 k6 [s1..s4]]], n_dist in {0, 4, 5, 8, 12} */
    int n_dist;
    float bf;             /* mbf */
    float depth_factor;   /* Tracking::mDepthMapFactor: already the multiplier (1 / RGBD.DepthMapFactor, or 1) */
} orbx_rgbd_calib;

/* The RGB-D Frame constructor in one call — Tracking::GrabImageRGBD's colour conversion and depth conversion, then
 * Frame::Frame(imGray, imDepth, ...) (src/Frame.cc:202-260): ExtractORB(0, imGray, 0, 0), UndistortKeyPoints() and
 * ComputeStereoFromRGBD(imDepth).  HOST inputs: `image` rows x cols of `channels` (1, 3 or 4; `rgb` as in orbx_extract_color),
 * `depth` the RAW rows x cols depth map, depth_type 0 = CV_16U, 1 = CV_32F, depth_step bytes per row.  GrabImageRGBD's
 * convertTo(CV_32F, depth_factor) applies when |depth_factor - 1| > 1e-5 or the map is not CV_32F; it is evaluated on the
 * sampled pixels only (it is element-wise), so the caller passes the map unconverted.  HOST outputs, capacity rows each:
 * mvKeys, mvKeysUn, descriptors, *n_out = N, mvuRight and mvDepth (-1 where the depth is not > 0).  Rows past *n_out are
 * undefined.  Every argument is checked before any work is queued: a NULL handle, output, depth or calib, a bad depth_type,
 * depth_step < cols * element size, channels not 1 / 3 / 4, step < cols * channels, capacity <= 0, n_dist not in
 * {0, 4, 5, 8, 12} or a NULL dist with n_dist > 0: ORBX_ERR_INVALID_ARG; a NULL image, rows or cols <= 0:
 * ORBX_ERR_EMPTY_IMAGE; more than `capacity` keypoints: ORBX_ERR_CAPACITY.  Frame 0 stays inspectable through the probes and
 * the pyramid mirror is filled, as after orbx_extract. */
int orbx_extract_rgbd(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int channels, int rgb,
                      const void* depth, int depth_type, size_t depth_step, const orbx_rgbd_calib* calib, orbx_keypoint* kp,
                      orbx_keypoint* kp_un, uint8_t* desc, int capacity, int* n_out, float* uRight, float* depth_out);
/* orbx_extract_rgbd over n_frames HOST grey frames images[i] (rows x cols, `step` bytes per row) and depth maps depths[i] of one
 * type and shape.  Outputs are [n_frames][capacity] slabs; n_out is [n_frames]; for every frame they equal what
 * orbx_extract_rgbd returns, bit for bit.  Copies are pipelined against compute when the host buffers are page-locked.
 * n_frames == 0 returns ORBX_OK and does nothing; a frame over capacity: ORBX_ERR_CAPACITY (its rows are undefined; nothing is
 * written past the slabs).  Afterwards the probes refuse every frame index until the next extraction, as after a stereo batch. */
int orbx_extract_rgbd_batch(orbx_extractor* ex, const uint8_t* const* images, const void* const* depths, int n_frames, int rows,
                            int cols, size_t step, int depth_type, size_t depth_step, const orbx_rgbd_calib* calib, orbx_keypoint* kp,
                            orbx_keypoint* kp_un, uint8_t* desc, int capacity, int* n_out, float* uRight, float* depth_out);
/* The same on DEVICE-resident grey frames (frame f at d_images + f * frame_stride, `pitch` bytes per row) and depth maps (at
 * d_depths + f * depth_frame_stride, depth_pitch bytes per row; base, pitch and stride multiples of the element size); every
 * output is DEVICE memory with the slab layout above.  Asynchronous on `stream` (NULL = the extractor's own): orbx_sync and the
 * next call on the handle wait for it, as for orbx_extract_batch_device.  A frame over capacity shows only in its device count
 * (*d_n_out > capacity; its rows are undefined).  Rows of d_kp_un / d_uRight / d_depth at or past a frame's count are left
 * untouched.  Colour frames: run
 * orbx_cvt_gray_device in front on the same stream. */
int orbx_extract_rgbd_batch_device(orbx_extractor* ex, const uint8_t* d_images, size_t frame_stride, size_t pitch, const void* d_depths,
                                   size_t depth_frame_stride, size_t depth_pitch, int depth_type, int n_frames, int rows, int cols,
                                   const orbx_rgbd_calib* calib, orbx_keypoint* d_kp, orbx_keypoint* d_kp_un, uint8_t* d_desc,
                                   int capacity, int* d_n_out, float* d_uRight, float* d_depth, void* stream);

/* ---- bag-of-words transform and vocabulary-guided matching (SURVEY.md §8 rows A13, A14 and (f)1) -------------------- */

/* DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB> (Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h): a k-ary tree of
 * 256-bit node descriptors.  Nodes are numbered as in m_nodes (0 = root, children in creation order = ascending id,
 * TemplatedVocabulary.h:1340-1398 loadFromTextFile); leaves carry a word id and a weight.  The handle owns a device copy. */
typedef struct orbx_vocabulary orbx_vocabulary;
typedef enum orbx_weighting { ORBX_TF_IDF = 0, ORBX_TF = 1, ORBX_IDF = 2, ORBX_BINARY = 3 } orbx_weighting;     /* BowVector.h:27-33 */
typedef enum orbx_scoring { ORBX_L1_NORM = 0, ORBX_L2_NORM = 1, ORBX_CHI_SQUARE = 2, ORBX_KL = 3, ORBX_BHATTACHARYYA = 4,
                            ORBX_DOT_PRODUCT = 5 } orbx_scoring;                                              /* BowVector.h:43-51 */
/* (the scoring type selects how orbx_compute_bow normalises; orbx_bow_score implements L1_NORM, the ORBvoc.txt setting) */
/* parent[0] = -1; descriptors [n_nodes][32]; weights [n_nodes] (leaf weight = idf, TemplatedVocabulary.h:1393);
 * a node is a leaf iff it has no children; word ids are assigned to leaves in ascending node id (TemplatedVocabulary.h:1388-1392). */
int orbx_vocab_create(int device, int n_nodes, const int32_t* parent, const uint8_t* descriptors, const double* weights, int k,
                      int L, int scoring, int weighting, orbx_vocabulary** out);
/* TemplatedVocabulary::loadFromTextFile (TemplatedVocabulary.h:1340-1398; the ORBvoc.txt format: "k L scoring weighting",
 * then per node "parent is_leaf b0 .. b31 weight"). */
int orbx_vocab_load_text(int device, const char* path, orbx_vocabulary** out);
void orbx_vocab_destroy(orbx_vocabulary* voc);
int orbx_vocab_info(const orbx_vocabulary* voc, int* n_nodes, int* n_words, int* k, int* L);

/* transform(feature, word_id, weight, &nid, levelsup) for every feature (TemplatedVocabulary.h:1217-1259): greedy descent,
 * the child with the least Hamming distance wins, ties -> the first child; node_id = the node met at level L - levelsup
 * (0 = root when L - levelsup <= 0).  HOST arrays of n entries; any output may be NULL.  Runs on the GPU, in the tracking
 * thread's device scratch (Frame::ComputeBoW). */
int orbx_bow_transform(const orbx_vocabulary* voc, const uint8_t* descriptors, int n, int levelsup, uint32_t* word_id,
                       double* weight, uint32_t* node_id);
/* Frame::ComputeBoW / KeyFrame::ComputeBoW (src/Frame.cc:768-775): transform(features, BowVector, FeatureVector, levelsup)
 * (TemplatedVocabulary.h:1126-1204, BowVector.cpp:34-90, FeatureVector.cpp:32-46).
 *   BowVector    -> bow_ids[*n_bow] ascending, bow_vals[*n_bow] (weighted + normalised exactly as the std::map code does);
 *   FeatureVector -> CSR: fv_nodes[*n_fv] ascending node ids, fv_offsets[*n_fv + 1], fv_indices[n] (feature ids ascending per node).
 * bow_* need capacity n, fv_nodes n, fv_offsets n + 1, fv_indices n. */
int orbx_compute_bow(const orbx_vocabulary* voc, const uint8_t* descriptors, int n, int levelsup, uint32_t* bow_ids,
                     double* bow_vals, int* n_bow, uint32_t* fv_nodes, int32_t* fv_offsets, uint32_t* fv_indices, int* n_fv);
/* DBoW2 score between two BowVectors for the vocabulary's scoring type (ScoringObject.cpp; L1: 1 - 0.5*sum|a-b| computed as
 * sum(|a-b| - |a| - |b|) over common words, ScoringObject.cpp:24-62).  Host. */
int orbx_bow_score(const orbx_vocabulary* voc, const uint32_t* ids_a, const double* vals_a, int na, const uint32_t* ids_b,
                   const double* vals_b, int nb, double* score);

/* A DBoW2::FeatureVector (std::map<NodeId, std::vector<unsigned>>, FeatureVector.h:23-25) in CSR form, node ids ascending. */
typedef struct orbx_feature_vector {
    int n_nodes;
    const uint32_t* node_ids;    /* [n_nodes] */
    const int32_t* offsets;      /* [n_nodes + 1] */
    const uint32_t* indices;     /* [offsets[n_nodes]] feature indices */
} orbx_feature_vector;

/* int ORBmatcher::SearchByBoW(KeyFrame* pKF, Frame& F, vector<MapPoint*>& vpMapPointMatches) — src/ORBmatcher1.cc:225-427
 * (mode 0) and SearchByBoW(KeyFrame* pKF1, KeyFrame* pKF2, vector<MapPoint*>& vpMatches12) — src/ORBmatcher2.cc:36-171 (mode 1).
 * A = the key frame whose features drive the outer loop (pKF / pKF1), B = the searched set (F / pKF2).
 *   valid_a[i] != 0  <=> feature i of A has a usable map point (non-NULL, !isBad(); mode 1 also folds the NLeft test of :77-79)
 *   valid_b[j] != 0  <=> mode 1 only: pKF2's map point j is usable (:95-103); ignored (may be NULL) in mode 0
 *   nleft_b          = F.Nleft (-1 for anything but a two-fisheye rig): mode 0 keeps separate best/second for j < Nleft and
 *                      j >= Nleft and accepts the right one without a ratio test (the reference's '|| true', :381)
 * Features of B already matched are skipped by later features of A inside the same vocabulary node (:289, :98): that
 * sequential dependence is honoured (one warp walks a node's A-list in order; lanes scan the B-list).
 * Outputs: mode 0: match_b[nB] = index of the A feature whose map point was assigned to B's feature j (vpMapPointMatches),
 *          mode 1: match_a[nA] = index of the B feature matched to A's feature i (vpMatches12), -1 = none; the other array
 *          (may be NULL) receives the inverse map.  *n_matches = the reference's return value (after the rotation filter).
 * Mode 0 uses the tracking thread's device scratch, mode 1 the loop-closing thread's.
 * orbx_search_by_bow_batch with one key frame (pKF in mode 0, pKF2 in mode 1): the same checks, results and device scratch. */
int orbx_search_by_bow(int device, int mode, const uint8_t* desc_a, const float* angle_a, const uint8_t* valid_a, int n_a,
                       const orbx_feature_vector* fv_a, const uint8_t* desc_b, const float* angle_b, const uint8_t* valid_b,
                       int n_b, const orbx_feature_vector* fv_b, int nleft_b, float nn_ratio, int check_orientation,
                       int32_t* match_a, int32_t* match_b, int* n_matches);

/* One key frame of orbx_search_by_bow_batch: the side that changes from search to search (HOST pointers). */
typedef struct orbx_bow_view {
    int n;                       /* N of the key frame */
    const uint8_t* desc;         /* mDescriptors, n x 32 */
    const float* angle;          /* mvKeysUn[i].angle; may be NULL without check_orientation */
    const uint8_t* valid;        /* [n] != 0 <=> the feature's map point is non-NULL and !isBad() */
    orbx_feature_vector fv;      /* mFeatVec */
} orbx_bow_view;
/* orbx_search_by_bow of one fixed side against n_kf key frames in one call.  The two place-recognition loops of ORB-SLAM3:
 *   mode 0, Tracking::Relocalization (src/Tracking5.cc:63-83): SearchByBoW(vpCandidateKFs[i], mCurrentFrame, ...) per candidate.
 *           The fixed side is B, the Frame (valid is not read, may be NULL; nleft = F.Nleft as nleft_b); kfs[k] is an A side.
 *           match[k * n + j] = index in kfs[k] whose map point the Frame's feature j received (match_b of the single call).
 *   mode 1, LoopClosing::DetectCommonRegionsFromBoW (src/LoopClosing1.cc:591-662): SearchByBoW(mpCurrentKF, vpCovKFi[j], ...)
 *           per covisible.  The fixed side is A, KF1 (nleft must be -1); kfs[k] is a B side, KF2.
 *           match[k * n + i] = index in kfs[k] matched to KF1's feature i (match_a of the single call).
 * n_matches[k] = the return value for key frame k.  Row k is bit-identical to orbx_search_by_bow on that key frame with the same
 * nn_ratio and check_orientation (rotation filter included): neither loop changes map state between its searches, so the
 * searches are independent.  The fixed side is uploaded once and every key frame's arrays in one packed copy; the common
 * vocabulary nodes are found on the GPU and one launch searches every key frame (DESIGN.md §5f).
 * n_kf == 0 does nothing; n_kf > 65535 is ORBX_ERR_UNSUPPORTED.  ORBX_ERR_INVALID_ARG, before any work is queued, for the single
 * call's argument errors on the fixed side or on any view (null arrays, a malformed feature vector, an index out of range,
 * angles missing under check_orientation).  Mode 0 uses the tracking thread's device scratch, mode 1 the loop-closing thread's. */
int orbx_search_by_bow_batch(int device, int mode, const uint8_t* desc, const float* angle, const uint8_t* valid, int n,
                             const orbx_feature_vector* fv, int nleft, int n_kf, const orbx_bow_view* kfs, float nn_ratio,
                             int check_orientation, int32_t* match, int* n_matches);

/* int ORBmatcher::SearchForTriangulation(pKF1, pKF2, vMatchedPairs, bOnlyStereo, bCoarse) — src/ORBmatcher2.cc:173-471, the
 * single-camera (pinhole, !mpCamera2) path.  Per feature of KF1 without a map point: scan the features of KF2 in the same
 * vocabulary node, keep the candidate of least distance <= TH_LOW (a later candidate of EQUAL distance replaces the
 * earlier one, :289) that passes the epipole-distance gate (:299-307) and Pinhole::epipolarConstrain
 * (src/CameraModels/Pinhole.cpp:107-129) unless coarse.  vbMatched2 is never set by the reference, so queries are independent.
 *   kp_a / kp_b      = mvKeysUn (pt, octave, angle are read)
 *   free_a / free_b  != 0 <=> the feature has no map point yet (:246-252, :273-277)
 *   stereo_a / stereo_b != 0 <=> mvuRight[i] >= 0 (:254, :279)
 *   F12[9]           = row-major K1^-T [t12]x R12 K2^-1 computed by the caller exactly as Pinhole.cpp:109-112 does
 *   ep[2]            = projection of KF1's camera centre into KF2 (:186-189); scale_b / sigma2_b = mvScaleFactors and mvLevelSigma2
 *                      of KF2, n_levels entries (Pinhole::epipolarConstrain ignores its sigmaLevel argument, KF1's sigma)
 * Output: match_a[nA] = index in B or -1 (vMatches12 after the rotation filter); *n_matches = the return value.
 * orbx_search_for_triangulation_batch with this one neighbour: the same checks, results and device scratch. */
int orbx_search_for_triangulation(int device, const orbx_keypoint* kp_a, const uint8_t* desc_a, const uint8_t* free_a,
                                  const uint8_t* stereo_a, int n_a, const orbx_feature_vector* fv_a, const orbx_keypoint* kp_b,
                                  const uint8_t* desc_b, const uint8_t* free_b, const uint8_t* stereo_b, int n_b,
                                  const orbx_feature_vector* fv_b, const float* F12, const float* ep, const float* scale_b,
                                  const float* sigma2_b, int n_levels, int only_stereo, int coarse, int check_orientation,
                                  int32_t* match_a, int* n_matches);

/* One neighbour (pKF2) of orbx_search_for_triangulation_batch: the KF2 arguments of orbx_search_for_triangulation, plus the
 * neighbour's own bCoarse (HOST pointers). */
typedef struct orbx_triangulation_view {
    int n;                          /* KF2's N */
    const orbx_keypoint* kp;        /* mvKeysUn */
    const uint8_t* desc;            /* mDescriptors, n x 32 */
    const uint8_t* free;            /* [n] != 0 <=> no map point yet */
    const uint8_t* stereo;          /* [n] != 0 <=> mvuRight[j] >= 0 */
    orbx_feature_vector fv;         /* mFeatVec */
    float F12[9];                   /* row-major K1^-T [t12]x R12 K2^-1 (Pinhole.cpp:109-112) */
    float ep[2];                    /* KF1's camera centre projected into KF2 */
    const float* scale;             /* mvScaleFactors, n_levels entries */
    const float* sigma2;            /* mvLevelSigma2, n_levels entries */
    int n_levels;
    int coarse;                     /* bCoarse */
} orbx_triangulation_view;
/* orbx_search_for_triangulation of KF1 against n_kf neighbours in one call (the neighbour loop of
 * LocalMapping::CreateNewMapPoints, src/LocalMapping.cc): KF1 is uploaded once, the neighbours in one packed copy, the
 * jobs are built on the GPU and one launch scans them all.  For every neighbour k the result is bit-identical to
 * orbx_search_for_triangulation(KF1, kfs[k], ..., only_stereo, kfs[k].coarse, check_orientation):
 *   match[k * n_a + i] = index in kfs[k] or -1 (after the rotation filter when check_orientation), n_matches[k] = its return value.
 * The neighbours are searched against the same free_a: the caller that adds map points to KF1 between neighbours drops the
 * later neighbours' matches of those features itself (the C++ adapter does; DESIGN.md §5d).  n_kf == 0 does nothing.
 * ORBX_ERR_INVALID_ARG per neighbour as the single call: null arrays, a malformed feature vector, n_levels outside
 * [1, ORBX_MAX_LEVELS], an octave outside [0, n_levels).  Uses local mapping's device scratch (that of orbx_fuse), so it never
 * waits on the tracking thread's searches. */
int orbx_search_for_triangulation_batch(int device, const orbx_keypoint* kp_a, const uint8_t* desc_a, const uint8_t* free_a,
                                        const uint8_t* stereo_a, int n_a, const orbx_feature_vector* fv_a, int n_kf,
                                        const orbx_triangulation_view* kfs, int only_stereo, int check_orientation,
                                        int32_t* match, int* n_matches);

/* ---- the frame grid and the projection-guided searches (SURVEY.md §8(f)2) ---------------------------------- */

#define ORBX_FRAME_GRID_ROWS 48   /* include/Frame.h:44 */
#define ORBX_FRAME_GRID_COLS 64   /* include/Frame.h:45 */

/* The slice of ORB_SLAM3::Frame the searches read (HOST pointers; Nleft == -1: one camera, rectified stereo or RGB-D). */
typedef struct orbx_frame_view {
    int n;                          /* Frame::N */
    const orbx_keypoint* keys_un;   /* mvKeysUn (pt, octave, angle are read) */
    const uint8_t* descriptors;     /* mDescriptors, n x 32 */
    const float* u_right;           /* mvuRight, NULL = none (monocular: all -1) */
    const uint8_t* occupied;        /* [n] or NULL: the feature's map point on entry makes later queries skip it (each function
                                     * says what that means: Observations() > 0, or merely non-NULL) */
    float min_x, min_y, max_x, max_y;   /* mnMinX, mnMinY, mnMaxX, mnMaxY (src/Frame.cc:150-162) */
    float grid_w_inv, grid_h_inv;   /* mfGridElementWidthInv / HeightInv = 64 / (maxX - minX), 48 / (maxY - minY) */
    const float* scale_factors;     /* mvScaleFactors, n_levels entries */
    int n_levels;
} orbx_frame_view;

/* Frame::AssignFeaturesToGrid (src/Frame.cc:387-418, PosInGrid :755-766) as CSR over cell id = ix * 48 + iy:
 * cell_start[64*48 + 1], items[n] (only cell_start[64*48] entries are written: features outside the grid are dropped), the
 * features of a cell in push_back order = ascending index.  Runs on the GPU (the same kernel the searches use). */
int orbx_assign_features_to_grid(int device, const orbx_frame_view* frame, int32_t* cell_start, int32_t* items);
/* vector<size_t> Frame::GetFeaturesInArea(x, y, r, minLevel, maxLevel) (src/Frame.cc:687-753): indices in the reference's
 * order (cell column, cell row, in-cell order).  ORBX_ERR_CAPACITY with *n_out = needed count if out is too small. */
int orbx_get_features_in_area(int device, const orbx_frame_view* frame, float x, float y, float r, int min_level, int max_level,
                              int32_t* out, int capacity, int* n_out);

/* The map points of Tracking::SearchLocalPoints as the fields SearchByProjection reads (HOST arrays of n entries). */
typedef struct orbx_track_points {
    int n;
    const uint8_t* in_view;         /* pMP->mbTrackInView */
    const uint8_t* bad;             /* pMP->isBad() */
    const float* proj_x;            /* mTrackProjX */
    const float* proj_y;            /* mTrackProjY */
    const float* proj_xr;           /* mTrackProjXR */
    const float* view_cos;          /* mTrackViewCos */
    const float* track_depth;       /* mTrackDepth (read only with far_points) */
    const int32_t* scale_level;     /* mnTrackScaleLevel */
    const int32_t* n_obs;           /* Observations() */
    const uint8_t* descriptors;     /* GetDescriptor(), n x 32 */
} orbx_track_points;

/* int ORBmatcher::SearchByProjection(Frame& F, const vector<MapPoint*>& vpMapPoints, th, bFarPoints, thFarPoints)
 * — src/ORBmatcher1.cc:45-215 (Nleft == -1).  frame->occupied[idx] != 0 <=> F.mvpMapPoints[idx] && Observations() > 0 on entry.
 * Window radius = RadiusByViewingCos(viewCos) [* th] * mvScaleFactors[level] (:68-74), levels [level-1, level], mvuRight gate
 * (:95-100), best/second with the same-level ratio test against nn_ratio (mfNNratio) and TH_HIGH (:125-131).  Features taken by
 * an earlier map point of the call are skipped by later ones exactly as the sequential loop does.
 * Output: match_f[frame->n] = index of the map point assigned to the feature by THIS call, -1 = untouched;
 * *n_matches = the return value. */
int orbx_search_by_projection_map(int device, const orbx_frame_view* frame, const orbx_track_points* points, float th,
                                  int far_points, float th_far_points, float nn_ratio, int32_t* match_f, int* n_matches);

/* int ORBmatcher::SearchByProjection(Frame& CurrentFrame, const Frame& LastFrame, th, bMono) — src/ORBmatcher3.cc:256-467
 * (Nleft == -1).  The Sophus/Eigen part stays with the caller: per last-frame feature i
 *   valid[i]   = LastFrame.mvpMapPoints[i] && !LastFrame.mvbOutlier[i]           (:278-281)
 *   u, v, invz = mpCamera->project(Tcw * x3Dw) and 1 / x3Dc(2)                   (:284-294)
 *   octave, angle = the last frame's key point (:304, :358-365), n_obs = pMP->Observations(), desc = pMP->GetDescriptor()
 *   forward / backward = bForward / bBackward (:272-273); mbf = CurrentFrame.mbf
 * cur->occupied as above.  Output: match_f[cur->n] = last-frame index i assigned to the feature (after the rotation filter),
 * *n_matches = the return value. */
int orbx_search_by_projection_last(int device, const orbx_frame_view* cur, float mbf, int n_last, const uint8_t* valid,
                                   const float* u, const float* v, const float* invz, const int32_t* octave, const float* angle,
                                   const int32_t* n_obs, const uint8_t* desc, float th, int forward, int backward,
                                   int check_orientation, int32_t* match_f, int* n_matches);

/* int ORBmatcher::SearchByProjection(Frame& CurrentFrame, KeyFrame* pKF, sAlreadyFound, th, ORBdist) — src/ORBmatcher3.cc:469-578.
 *   valid[i] = pMP && !pMP->isBad() && !sAlreadyFound.count(pMP); u, v = projection by the caller; dist3d = |x3Dw - Ow| with the
 *   map point's min/max distance invariance (:508-514); level = pMP->PredictScale(dist3D, &CurrentFrame) (:516); angle = pKF->mvKeysUn[i].angle.
 * cur->occupied[idx] != 0 <=> CurrentFrame.mvpMapPoints[idx] != NULL (:533), and every assignment of the call occupies. */
int orbx_search_by_projection_kf(int device, const orbx_frame_view* cur, int n_kf, const uint8_t* valid, const float* u,
                                 const float* v, const float* dist3d, const float* min_dist, const float* max_dist,
                                 const int32_t* level, const float* angle, const uint8_t* desc, float th, int orb_dist,
                                 int check_orientation, int32_t* match_f, int* n_matches);
/* int ORBmatcher::SearchForInitialization(Frame &F1, Frame &F2, vector<cv::Point2f> &vbPrevMatched, vector<int> &vnMatches12,
 * int windowSize) — src/ORBmatcher1.cc:650-765, as Tracking::MonocularInitialization calls it (src/Tracking3.cc:740-741).
 *   kp1 / desc1 = F1.mvKeysUn / F1.mDescriptors (n1 rows); only features with octave <= 0 search (the reference skips level1 > 0),
 *   in GetFeaturesInArea(vbPrevMatched[i1], windowSize, level1, level1) of f2 (f2->u_right, f2->occupied and the scale factors
 *   are not read).  Best / second-best with the vMatchedDistance skip, TH_LOW and 'bestDist < (float)bestDist2 * mfNNratio' (no
 *   second-best always passes); a later feature of F1 that reaches an F2 feature at a smaller distance takes it over.
 *   prev_matched = vbPrevMatched [n1][2] (x, y), in/out: matched entries become F2.mvKeysUn[vnMatches12[i1]].pt.
 * Output: matches12[n1] = vnMatches12 (after the rotation filter when check_orientation), *n_matches = the return value.
 * ORBX_ERR_INVALID_ARG for a keypoint angle pair outside the histogram (the reference asserts). */
int orbx_search_for_initialization(int device, const orbx_keypoint* kp1, const uint8_t* desc1, int n1, const orbx_frame_view* f2,
                                   float* prev_matched, int window_size, float nn_ratio, int check_orientation, int32_t* matches12,
                                   int* n_matches);
/* The slice of ORB_SLAM3::KeyFrame that ORBmatcher::Fuse reads (HOST pointers; NLeft == -1). */
typedef struct orbx_keyframe_view {
    orbx_frame_view frame;          /* mvKeysUn, mDescriptors, mvuRight (NULL = monocular), bounds, grid, mvScaleFactors; frame.occupied is not read */
    const float* inv_level_sigma2;  /* mvInvLevelSigma2, frame.n_levels entries */
    float bf;                       /* mbf */
} orbx_keyframe_view;
/* int ORBmatcher::Fuse(KeyFrame* pKF, const vector<MapPoint*>& vpMapPoints, th, bRight = false) — src/ORBmatcher2.cc:420-610, as
 * LocalMapping::SearchInNeighbors calls it (src/LocalMapping.cc:766-803), for n_kf key frames in one call: the search part.
 *   Pairs [kf_offsets[k], kf_offsets[k + 1]) belong to key frame kfs[k]; kf_offsets[0] = 0, nq = kf_offsets[n_kf].  Pair q is
 *   map point point[q] (its descriptor = point_desc row point[q], 0 <= point[q] < n_desc) projected to (u[q], v[q]) with
 *   invz[q] = 1 / p3Dc(2) and level[q] = pMP->PredictScale(dist3D, pKF).  valid[q] folds the caller's pre-checks: pMP &&
 *   !isBad() && !IsInKeyFrame(pKF), p3Dc(2) >= 0, the distance window and the viewing angle (Eigen arithmetic, with the caller).
 *   This call applies IsInImage (x >= mnMinX && x < mnMaxX, the same for y; upper bounds strict), the window
 *   GetFeaturesInArea(u, v, th * mvScaleFactors[level]), the level gate [level - 1, level], the reprojection gate (mvuRight >= 0:
 *   e2 * mvInvLevelSigma2 > 7.8 with ur = u - bf * invz, else > 5.99) and the 1-NN by Hamming distance (earliest in the window's
 *   order on ties) under TH_LOW (50).  Pairs are independent: the candidate loop never reads the key frame's map points.
 * Output: match[nq] = bestIdx when bestDist <= 50, else -1; n_fused[n_kf] = matches per key frame (the reference's return value
 *   when no point changes state during the call).  The bookkeeping (AddMapPoint / Replace) stays with the caller.
 * ORBX_ERR_INVALID_ARG for null arrays, a missing inv_level_sigma2, non-monotone offsets, point[q] outside [0, n_desc) or a level
 * outside [0, n_levels) on a valid pair.  Uses local mapping's device scratch, so it never waits on the tracking thread's searches. */
int orbx_fuse(int device, int n_kf, const orbx_keyframe_view* kfs, const int32_t* kf_offsets, int n_desc, const uint8_t* point_desc,
              const int32_t* point, const uint8_t* valid, const float* u, const float* v, const float* invz, const int32_t* level,
              float th, int32_t* match, int* n_fused);
/* int ORBmatcher::SearchByProjection(KeyFrame* pKF, Sophus::Sim3f& Scw, const vector<MapPoint*>& vpPoints,
 * [const vector<KeyFrame*>& vpPointsKFs,] vector<MapPoint*>& vpMatched, [vector<KeyFrame*>& vpMatchedKF,] int th,
 * float ratioHamming) — src/ORBmatcher1.cc:429-648 (NLeft == -1), as loop closing calls it (LoopClosing::DetectCommonRegionsFromBoW,
 * FindMatchesByProjection).  Point i is vpPoints[i] projected with Tcw = SE3(Scw.rotationMatrix(), Scw.translation() / Scw.scale())
 * to (u[i], v[i]), level[i] = pMP->PredictScale(dist, pKF), desc = pMP->GetDescriptor() (n_points x 32).
 *   valid[i] folds the caller's checks: !isBad(), not in spAlreadyFound (the non-NULL entries of vpMatched on entry),
 *   p3Dc(2) >= 0, the distance window and the viewing angle (Eigen arithmetic, with the caller).
 *   kf->occupied[idx] != 0 <=> vpMatched[idx] != NULL on entry; kf->u_right is not read.
 *   This call applies IsInImage (x >= mnMinX && x < mnMaxX, the same for y; upper bounds strict), the window
 *   GetFeaturesInArea(u, v, th * mvScaleFactors[level]), the level gate [level - 1, level] and the 1-NN by Hamming distance
 *   (earliest in the window's order on ties) accepted when bestDist <= TH_LOW * ratio_hamming (in float).  A feature taken by an
 *   earlier point of the call is skipped by later ones exactly as the sequential loop does.
 * Output: match_f[kf->n] = index of the point assigned to the feature by THIS call, -1 = untouched; *n_matches = the return value.
 * Sets orbx_projection_rounds().  ORBX_ERR_INVALID_ARG for null arrays, a level outside [0, n_levels) on a valid point, and
 * 50 * ratio_hamming >= 256 or NaN (where the reference would write vpMatched[-1]).  Uses the loop-closing thread's own device
 * scratch. */
int orbx_search_by_projection_sim3(int device, const orbx_frame_view* kf, int n_points, const uint8_t* valid, const float* u,
                                   const float* v, const int32_t* level, const uint8_t* desc, float th, float ratio_hamming,
                                   int32_t* match_f, int* n_matches);
/* int ORBmatcher::Fuse(KeyFrame* pKF, Sophus::Sim3f& Scw, const vector<MapPoint*>& vpPoints, float th,
 * vector<MapPoint*>& vpReplacePoint) — src/ORBmatcher2.cc:612-729, as LoopClosing::SearchAndFuse calls it (both overloads), for
 * n_kf key frames in one call: the search part.  The layout of orbx_fuse without invz: pairs [kf_offsets[k], kf_offsets[k + 1])
 * belong to kfs[k]; pair q is point point[q] (a row of point_desc) at (u[q], v[q]) with level[q] = PredictScale.  valid[q] folds
 * the caller's pre-checks: !isBad(), not in pKF->GetMapPoints() on entry, p3Dc(2) >= 0, the distance window, the viewing angle.
 *   This call applies IsInImage (upper bounds strict), the window GetFeaturesInArea(u, v, th * mvScaleFactors[level]), the level
 *   gate [level - 1, level] and the 1-NN by Hamming distance (earliest in the window's order on ties) under TH_LOW (50).  There is
 *   no reprojection gate: kfs[k].inv_level_sigma2, kfs[k].bf and kfs[k].frame.u_right are not read and may be NULL / 0.
 * Output: match[nq] = bestIdx when bestDist <= 50, else -1; n_fused[n_kf] = acceptances per key frame (the reference's return
 *   value).  The bookkeeping (vpReplacePoint, AddMapPoint, the Replace loop of SearchAndFuse) stays with the caller.
 * ORBX_ERR_INVALID_ARG as orbx_fuse (without the inv_level_sigma2 case).  Uses the loop-closing thread's own device scratch, so
 * it never waits on the tracking thread's searches or on orbx_fuse. */
int orbx_fuse_sim3(int device, int n_kf, const orbx_keyframe_view* kfs, const int32_t* kf_offsets, int n_desc, const uint8_t* point_desc,
                   const int32_t* point, const uint8_t* valid, const float* u, const float* v, const int32_t* level, float th,
                   int32_t* match, int* n_fused);
/* Speculation rounds the last projection search on this thread needed (diagnostics; 0 = every query was final at once). */
int orbx_projection_rounds(void);

/* ---- preparation steps either side of the extractor (SURVEY.md §8(f)3) ------------------------------------- */

/* void Frame::UndistortKeyPoints() — src/Frame.cc:777-810 = cv::undistortPoints(mvKeys, K, mDistCoef, cv::Mat(), mK).
 *   K[4] / new_K[4] = (fx, fy, cx, cy) of Pinhole::toK() and of mK; dist = mDistCoef (CV_32F: k1 k2 p1 p2 [k3 [k4 k5 k6]]),
 *   n_dist in {0, 4, 5, 8, 12}.  dist[0] == 0 (or n_dist == 0) copies the key points, as the reference does (:779-783).
 * HOST arrays; out may alias keypoints.  Computes on the GPU in double, bit-identical to OpenCV's scalar code, in the tracking
 * thread's device scratch. */
int orbx_undistort_keypoints(int device, const orbx_keypoint* keypoints, int n, const float* K, const float* dist, int n_dist,
                             const float* new_K, orbx_keypoint* out);

/* Stereo rectification of System::TrackStereo (src/System.cc:253-260): cv::remap(im, out, M1, M2, cv::INTER_LINEAR) with the
 * CV_32FC1 maps of cv::initUndistortRectifyMap (src/Settings.cc:488-491), BORDER_CONSTANT 0.  The maps are quantised to
 * OpenCV's 1/32-pixel fixed point once, at creation, and stay on the device. */
typedef struct orbx_rectifier orbx_rectifier;
int orbx_rectifier_create(int device, const float* map_x, const float* map_y, size_t map_step_bytes, int dst_rows, int dst_cols,
                          orbx_rectifier** out);
/* The other branch of System::TrackStereo / TrackMonocular / TrackRGBD (src/System.cc:261-263, 330, 407, settings_->needToResize()):
 * cv::resize(im, out, newImSize) — INTER_LINEAR on 8UC1 (OpenCV's 11-bit fixed point; exact 2x takes the INTER_AREA average).
 * Returns a rectifier whose orbx_remap / orbx_remap_device calls resize src_rows x src_cols images to dst_rows x dst_cols. */
int orbx_resizer_create(int device, int src_rows, int src_cols, int dst_rows, int dst_cols, orbx_rectifier** out);
void orbx_rectifier_destroy(orbx_rectifier* r);
/* One HOST image (src_rows x src_cols, 8UC1) -> HOST dst (dst_rows x dst_cols of the rectifier). */
int orbx_remap(orbx_rectifier* r, const uint8_t* src, int src_rows, int src_cols, size_t src_step, uint8_t* dst, size_t dst_step);
/* Device-resident frames (frame f at d_src + f * src_frame_stride), on `stream` (a cudaStream_t or NULL); chain it in front of
 * orbx_extract_batch_device on the same stream to keep the rectified images on the device. */
int orbx_remap_device(orbx_rectifier* r, const uint8_t* d_src, int src_rows, int src_cols, size_t src_pitch, size_t src_frame_stride,
                      int n_frames, uint8_t* d_dst, size_t dst_pitch, size_t dst_frame_stride, void* stream);

/* ---- measurement helpers ----------------------------------------------------------------------------------- */

/* Per-stage device timing: between begin and end every extraction on `ex` records CUDA events around its stages on the
 * launching stream; end() waits for them and returns the summed milliseconds of the 6 stages
 * {pyramid, fast, blur, octree, orient+describe, pack} and the number of chunks timed. */
#define ORBX_NUM_STAGES 6
int orbx_profile_begin(orbx_extractor* ex);
int orbx_profile_end(orbx_extractor* ex, float* stage_ms, int* n_chunks);

/* POPC.b32 issue-rate microbenchmark on `device`: returns popc instructions (per 32-bit lane) per second. */
int orbx_measure_popc_peak(int device, double* popc_per_second);
/* Number of kernel launches issued by this library on the calling process since load (for bench gpu_launches). */
int64_t orbx_launch_count(void);

/* ---- synthetic inputs (integer-only, bit-identical on host and device; csrc/synth.h) ----------------------- */
void orbx_synth_image_host(uint32_t seed, int view, int cols, int rows, int max_disp, uint8_t* dst, size_t step);
int orbx_synth_images_device(int device, uint32_t seed0, int view, int n_frames, int cols, int rows, int max_disp,
                             uint8_t* d_dst, size_t pitch, size_t frame_stride, void* stream);
void orbx_synth_descriptors_host(uint32_t seed, int is_query, int64_t first_row, int64_t n_rows, int64_t ndb,
                                 int plant_every, uint8_t* dst);
int orbx_synth_descriptors_device(int device, uint32_t seed, int is_query, int64_t first_row, int64_t n_rows,
                                  int64_t ndb, int plant_every, uint8_t* d_dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ORBX_H_ */
