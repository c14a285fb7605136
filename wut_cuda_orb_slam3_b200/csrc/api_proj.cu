// api_proj.cu — host side of the frame grid and the projection-guided searches (C ABI of include/orbx.h).
//
// Reference interfaces replaced (paths relative to the reference root):
//   Frame::AssignFeaturesToGrid / PosInGrid / GetFeaturesInArea          src/Frame.cc:387-418, 755-766, 687-753
//   ORBmatcher::SearchByProjection(Frame&, vector<MapPoint*>&, ...)      src/ORBmatcher1.cc:45-215   (Tracking::SearchLocalPoints)
//   ORBmatcher::SearchByProjection(Frame& Current, const Frame& Last..)  src/ORBmatcher3.cc:256-467  (Tracking::TrackWithMotionModel)
//   ORBmatcher::SearchByProjection(Frame& Current, KeyFrame*, ...)       src/ORBmatcher3.cc:469-578  (Tracking::Relocalization)
//   ORBmatcher::SearchForInitialization(F1, F2, vbPrevMatched, ...)      src/ORBmatcher1.cc:650-765  (Tracking::MonocularInitialization)
//   ORBmatcher::Fuse(KeyFrame*, const vector<MapPoint*>&, th, bRight)     src/ORBmatcher2.cc:420-610  (LocalMapping::SearchInNeighbors)
//   ORBmatcher::SearchByProjection(KeyFrame*, Sim3f&, vpPoints, .., th, ratioHamming)   src/ORBmatcher1.cc:429-648 (LoopClosing)
//   ORBmatcher::Fuse(KeyFrame*, Sim3f&, vpPoints, th, vpReplacePoint)      src/ORBmatcher2.cc:612-729  (LoopClosing::SearchAndFuse)
// Each entry point turns the reference's per-map-point pre-checks into window queries (float arithmetic in the reference's
// order, on the host: a handful of operations per point), ships everything in ONE pinned staging copy, runs the grid build and
// the window search (kernels_proj.cu) and reads the per-query assignment back in one copy.  The 30-bin rotation histogram runs
// on the host afterwards (it depends on the accepted matches only).  These calls sit on the tracking thread's per-frame path,
// so the device scratch, the pinned staging buffer and the stream live in a per-device grow-only arena (no cudaMalloc per call).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>
#include <mutex>
#include <vector>

#include "orbx_internal.cuh"

namespace orbx {

ProjArena g_arena[64];
// orbx_fuse and orbx_search_for_triangulation_batch run on the local-mapping thread: their own arenas, so a large Fuse never
// holds the lock a tracking-thread search waits on
ProjArena g_fuse_arena[64];
// the Sim3 searches run on the loop-closing thread: a third set, so they never hold a lock the other two threads wait on
ProjArena g_loop_arena[64];

int Lease::reserve(size_t bytes)
{
    bytes += 8192;
    if (!A.st) {
        cudaError_t e = cudaStreamCreateWithFlags(&A.st, cudaStreamNonBlocking);
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
    }
    if (A.d_bytes < bytes) {
        if (A.d) cudaFree(A.d);
        if (A.h) cudaFreeHost(A.h);
        A.d = A.h = nullptr; A.d_bytes = A.h_bytes = 0;
        const size_t want = bytes + bytes / 2;
        cudaError_t e = cudaMalloc((void**)&A.d, want);
        if (e == cudaSuccess) e = cudaMallocHost((void**)&A.h, want);
        if (e != cudaSuccess) return fail(ORBX_ERR_OOM, "projection scratch (%zu bytes): %s", want, cudaGetErrorString(e));
        A.d_bytes = A.h_bytes = want;
    }
    return ORBX_OK;
}

namespace {

constexpr int GRID_CELLS = ORBX_FRAME_GRID_COLS * ORBX_FRAME_GRID_ROWS;
thread_local int t_rounds = 0;

int check_frame(const orbx_frame_view* f, bool need_desc)
{
    if (!f || f->n < 0) return fail(ORBX_ERR_INVALID_ARG, "bad frame view");
    if (f->n > 0 && (!f->keys_un || (need_desc && !f->descriptors))) return fail(ORBX_ERR_INVALID_ARG, "frame view: keys_un / descriptors missing");
    if (f->n >= (1 << 24)) return fail(ORBX_ERR_UNSUPPORTED, "frame view: too many features");
    if (!(f->grid_w_inv > 0.0f) || !(f->grid_h_inv > 0.0f)) return fail(ORBX_ERR_INVALID_ARG, "frame view: grid element sizes must be positive");
    if (need_desc && (!f->scale_factors || f->n_levels < 1 || f->n_levels > kMaxLevels)) return fail(ORBX_ERR_INVALID_ARG, "frame view: scale factors missing");
    return ORBX_OK;
}

// A frame + a set of window queries on the device.
struct Session {
    Lease L;
    ProjArgs A{};
    size_t o_kp = 0, o_desc = 0, o_ur = 0, o_taken = 0, o_q = 0, o_qd = 0, o_cs = 0, o_items = 0, o_cellof = 0, o_claim = 0, o_keys = 0,
           o_qm = 0, o_la = 0, o_lb = 0, o_rounds = 0, o_area = 0, o_area_n = 0, o_last_acc = 0, o_prev_acc = 0, o_acc_dist = 0;
    int n = 0, nq = 0, area_cap = 0;
    explicit Session(int device, ProjArena* arenas = g_arena) : L(device, arenas) {}

    // Lay out and reserve; afterwards queries()/qdesc() point into the pinned staging buffer for the caller to fill.
    int begin(int device, const orbx_frame_view* f, int n_queries, bool with_desc, int area_capacity = 0)
    {
        int rc;
        if ((rc = set_device(device))) return rc;
        n = f->n; nq = n_queries; area_cap = area_capacity;
        const size_t total = lease_pad((size_t)n * 28) + lease_pad((size_t)n * 32) + lease_pad((size_t)n * 4) + lease_pad((size_t)n * 4) + lease_pad((size_t)nq * sizeof(ProjQuery)) +
                             lease_pad((size_t)nq * 32) + lease_pad((GRID_CELLS + 1) * 4) + lease_pad((size_t)n * 4) + lease_pad((size_t)n * 2) + lease_pad((size_t)n * 4) +
                             lease_pad((size_t)nq * 16) + 3 * lease_pad((size_t)nq * 4) + lease_pad(4) + lease_pad((size_t)area_cap * 8) + lease_pad(4) +
                             lease_pad((size_t)n * 4) + 2 * lease_pad((size_t)nq * 4);
        if ((rc = L.reserve(total))) return rc;
        // upload range
        o_kp = L.take<orbx_keypoint>(n);
        o_desc = L.take<uint8_t>((size_t)n * 32);
        o_ur = L.take<float>(n);
        o_taken = L.take<int>(n);
        o_q = L.take<ProjQuery>(nq);
        o_qd = L.take<uint8_t>((size_t)nq * 32);
        o_qm = L.take<int>(nq);
        o_area_n = L.take<int>(1);
        L.upload_end = L.off;
        // device-only scratch / outputs
        o_cs = L.take<int>(GRID_CELLS + 1);
        o_items = L.take<int>(n);
        o_cellof = L.take<unsigned short>(n);
        o_claim = L.take<int>(n);
        o_keys = L.take<unsigned long long>((size_t)nq * 2);
        o_la = L.take<int>(nq);
        o_lb = L.take<int>(nq);
        o_rounds = L.take<int>(1);
        o_area = L.take<unsigned long long>(area_cap);
        o_last_acc = L.take<int>(n);
        o_prev_acc = L.take<int>(nq);
        o_acc_dist = L.take<int>(nq);
        if (n) memcpy(L.host<orbx_keypoint>(o_kp), f->keys_un, (size_t)n * sizeof(orbx_keypoint));
        if (n && with_desc) memcpy(L.host<uint8_t>(o_desc), f->descriptors, (size_t)n * 32);
        if (n && f->u_right) memcpy(L.host<float>(o_ur), f->u_right, (size_t)n * 4);
        for (int i = 0; i < n; ++i) L.host<int>(o_taken)[i] = f->occupied && f->occupied[i] ? -1 : INT_MAX;
        for (int i = 0; i < nq; ++i) L.host<int>(o_qm)[i] = -1;
        *L.host<int>(o_area_n) = 0;
        A.n = n; A.kp = L.dev<orbx_keypoint>(o_kp); A.desc = L.dev<uint8_t>(o_desc); A.u_right = f->u_right ? L.dev<float>(o_ur) : nullptr;
        A.min_x = f->min_x; A.min_y = f->min_y; A.grid_w_inv = f->grid_w_inv; A.grid_h_inv = f->grid_h_inv;
        A.cell_start = L.dev<int>(o_cs); A.items = L.dev<int>(o_items); A.cell_of = L.dev<unsigned short>(o_cellof);
        A.taken_by = L.dev<int>(o_taken); A.claim = L.dev<int>(o_claim);
        A.nq = nq; A.q = L.dev<ProjQuery>(o_q); A.qdesc = L.dev<uint8_t>(o_qd);
        A.keys = L.dev<unsigned long long>(o_keys); A.qmatch = L.dev<int>(o_qm); A.list_a = L.dev<int>(o_la); A.list_b = L.dev<int>(o_lb);
        A.rounds_out = L.dev<int>(o_rounds);
        return ORBX_OK;
    }
    // Mode 2 keeps the acceptances of each feature as a chain; the grid build resets last_acc (before upload_and_grid()).
    void enable_chains()
    {
        A.last_acc = L.dev<int>(o_last_acc); A.prev_acc = L.dev<int>(o_prev_acc); A.acc_dist = L.dev<int>(o_acc_dist);
    }
    ProjQuery* queries() { return L.host<ProjQuery>(o_q); }
    uint8_t* qdesc() { return L.host<uint8_t>(o_qd); }
    cudaStream_t stream() const { return L.A.st; }

    int upload_and_grid()
    {
        cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, stream());
        if (e == cudaSuccess) e = launch_frame_grid(A, stream());
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "frame grid: %s", cudaGetErrorString(e));
        return ORBX_OK;
    }
    // Run the search; on return qmatch()[i] = feature assigned to query i or -1.
    int search(int mode, int th_dist, float nn_ratio)
    {
        int rc;
        if ((rc = upload_and_grid())) return rc;
        A.mode = mode; A.th_dist = th_dist; A.nn_ratio = nn_ratio;
        cudaError_t e = launch_proj_search(A, stream());
        // qmatch and the round counter come back through the staging buffer (device-only offsets map 1:1 into it)
        if (e == cudaSuccess && nq) e = cudaMemcpyAsync(L.host<int>(o_qm), L.dev<int>(o_qm), (size_t)nq * 4, cudaMemcpyDeviceToHost, stream());
        if (e == cudaSuccess && nq) e = cudaMemcpyAsync(L.host<int>(o_rounds), L.dev<int>(o_rounds), 4, cudaMemcpyDeviceToHost, stream());
        if (e == cudaSuccess) e = cudaStreamSynchronize(stream());
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "projection search: %s", cudaGetErrorString(e));
        t_rounds = nq ? *L.host<int>(o_rounds) : 0;
        return ORBX_OK;
    }
    const int* qmatch() const { return L.host<int>(o_qm); }
};

// src/ORBmatcher1.cc:217-223
float radius_by_viewing_cos(const float& viewCos)
{
    if (viewCos > 0.998) return 2.5;
    else return 4.0;
}

// Shared tail of the two 1-NN variants: assignments in query order, then the rotation filter (src/ORBmatcher3.cc:442-464, 555-575).
int finish_1nn(const Session& S, const orbx_frame_view* cur, const float* angle_q, int check_orientation, int32_t* match_f, int* n_matches)
{
    const int H = 30;
    int nm = 0;
    for (int i = 0; i < cur->n; ++i) match_f[i] = -1;
    std::vector<int> rot[H];
    for (int i = 0; i < S.nq; ++i) {
        const int f = S.qmatch()[i];
        if (f < 0) continue;
        match_f[f] = i;
        ++nm;
        if (check_orientation) {
            const int b = rotation_bin(angle_q[i], cur->keys_un[f].angle);
            if (b < 0) return fail(ORBX_ERR_INVALID_ARG, "keypoint angles out of range (the reference asserts)");
            rot[b].push_back(f);
        }
    }
    if (check_orientation) {
        int count[H], i1, i2, i3;
        for (int b = 0; b < H; ++b) count[b] = (int)rot[b].size();
        three_maxima(count, H, i1, i2, i3);
        for (int b = 0; b < H; ++b) {
            if (b == i1 || b == i2 || b == i3) continue;
            for (int f : rot[b]) { match_f[f] = -1; --nm; }
        }
    }
    *n_matches = nm;
    return ORBX_OK;
}

// Host body of orbx_fuse and orbx_fuse_sim3: the batched key frames, the pairs that pass the caller's pre-checks (valid) and
// KeyFrame::IsInImage, one pinned upload, the grids and the scan, one download.  gate = false is the Sim3 Fuse: no reprojection
// gate, so invz, inv_level_sigma2, bf and mvuRight are neither read nor uploaded.
int fuse_search(int device, ProjArena* arenas, const char* name, bool gate, int n_kf, const orbx_keyframe_view* kfs, const int32_t* kf_offsets,
                int n_desc, const uint8_t* point_desc, const int32_t* point, const uint8_t* valid, const float* u, const float* v,
                const float* invz, const int32_t* level, float th, int32_t* match, int* n_fused)
{
    int rc;
    if (n_kf < 0 || n_desc < 0 || !kf_offsets || (n_kf > 0 && (!kfs || !n_fused))) return fail(ORBX_ERR_INVALID_ARG, "%s: bad arguments", name);
    if (kf_offsets[0] != 0) return fail(ORBX_ERR_INVALID_ARG, "%s: kf_offsets[0] must be 0", name);
    for (int k = 0; k < n_kf; ++k)
        if (kf_offsets[k + 1] < kf_offsets[k]) return fail(ORBX_ERR_INVALID_ARG, "%s: kf_offsets not monotone at %d", name, k);
    const int nq = kf_offsets[n_kf];
    if (nq > 0 && (!point || !valid || !u || !v || (gate && !invz) || !level || !match))
        return fail(ORBX_ERR_INVALID_ARG, "%s: missing pair arrays", name);
    if (n_desc > 0 && !point_desc) return fail(ORBX_ERR_INVALID_ARG, "%s: point_desc missing", name);
    long long n_feat = 0;
    for (int k = 0; k < n_kf; ++k) {
        if ((rc = check_frame(&kfs[k].frame, true))) return rc;
        if (gate && !kfs[k].inv_level_sigma2) return fail(ORBX_ERR_INVALID_ARG, "%s: key frame %d: inv_level_sigma2 missing", name, k);
        n_feat += kfs[k].frame.n;
    }
    if (n_feat >= (1LL << 31) / 32) return fail(ORBX_ERR_UNSUPPORTED, "%s: too many key-frame features", name);
    // pre-checks of the caller (valid), then KeyFrame::IsInImage with strict upper bounds; the rest are compacted away
    std::vector<int> live;
    for (int k = 0; k < n_kf; ++k) {
        const orbx_frame_view& f = kfs[k].frame;
        for (int q = kf_offsets[k]; q < kf_offsets[k + 1]; ++q) {
            if (point[q] < 0 || point[q] >= n_desc) return fail(ORBX_ERR_INVALID_ARG, "%s: pair %d: point %d outside [0, %d)", name, q, point[q], n_desc);
            if (!valid[q]) continue;
            if (level[q] < 0 || level[q] >= f.n_levels) return fail(ORBX_ERR_INVALID_ARG, "%s: pair %d: level %d out of range", name, q, level[q]);
            if (!(u[q] >= f.min_x && u[q] < f.max_x && v[q] >= f.min_y && v[q] < f.max_y)) continue;
            if (f.n > 0) live.push_back(q);
        }
    }
    for (int q = 0; q < nq; ++q) match[q] = -1;
    for (int k = 0; k < n_kf; ++k) n_fused[k] = 0;
    if (live.empty()) return ORBX_OK;
    const int nv = (int)live.size();
    if ((rc = set_device(device))) return rc;
    Lease L(device, arenas);
    const size_t n_ur = gate ? (size_t)n_feat : 0;
    const size_t total = lease_pad((size_t)n_kf * sizeof(FuseKF)) + lease_pad((size_t)n_feat * 28) + lease_pad((size_t)n_feat * 32) + lease_pad(n_ur * 4) +
                         lease_pad((size_t)nv * sizeof(FuseQuery)) + lease_pad((size_t)n_desc * 32) + lease_pad((size_t)n_kf * (GRID_CELLS + 1) * 4) +
                         lease_pad((size_t)n_feat * 4) + lease_pad((size_t)n_feat * 2) + lease_pad((size_t)nv * 4);
    if ((rc = L.reserve(total))) return rc;
    // upload range
    const size_t o_kf = L.take<FuseKF>(n_kf), o_kp = L.take<orbx_keypoint>(n_feat), o_desc = L.take<uint8_t>((size_t)n_feat * 32),
                 o_ur = L.take<float>(n_ur), o_q = L.take<FuseQuery>(nv), o_pd = L.take<uint8_t>((size_t)n_desc * 32);
    L.upload_end = L.off;
    // device-only scratch / outputs
    const size_t o_cs = L.take<int>((size_t)n_kf * (GRID_CELLS + 1)), o_items = L.take<int>(n_feat), o_cellof = L.take<unsigned short>(n_feat),
                 o_match = L.take<int>(nv);
    FuseKF* K = L.host<FuseKF>(o_kf);
    size_t base = 0;
    for (int k = 0; k < n_kf; ++k) {
        const orbx_keyframe_view& kv = kfs[k];
        const orbx_frame_view& f = kv.frame;
        FuseKF e{};
        e.n = f.n;
        e.kp = L.dev<orbx_keypoint>(o_kp) + base; e.desc = L.dev<uint8_t>(o_desc) + base * 32;
        e.u_right = gate && f.u_right ? L.dev<float>(o_ur) + base : nullptr;
        e.min_x = f.min_x; e.min_y = f.min_y; e.grid_w_inv = f.grid_w_inv; e.grid_h_inv = f.grid_h_inv;
        e.cell_start = L.dev<int>(o_cs) + (size_t)k * (GRID_CELLS + 1);
        e.items = L.dev<int>(o_items) + base; e.cell_of = L.dev<unsigned short>(o_cellof) + base;
        if (gate)
            for (int l = 0; l < f.n_levels; ++l) e.inv_sigma2[l] = kv.inv_level_sigma2[l];
        K[k] = e;
        if (f.n) {
            memcpy(L.host<orbx_keypoint>(o_kp) + base, f.keys_un, (size_t)f.n * sizeof(orbx_keypoint));
            memcpy(L.host<uint8_t>(o_desc) + base * 32, f.descriptors, (size_t)f.n * 32);
            if (gate && f.u_right) memcpy(L.host<float>(o_ur) + base, f.u_right, (size_t)f.n * 4);
        }
        base += (size_t)f.n;
    }
    FuseQuery* Q = L.host<FuseQuery>(o_q);
    int k = 0;
    for (int i = 0; i < nv; ++i) {
        const int q = live[i];
        while (q >= kf_offsets[k + 1]) ++k;
        FuseQuery w{};
        w.u = u[q]; w.v = v[q];
        w.r = th * kfs[k].frame.scale_factors[level[q]];                     // src/ORBmatcher2.cc: radius = th * mvScaleFactors[nPredictedLevel]
        if (gate) w.ur = u[q] - kfs[k].bf * invz[q];                         // ur = uv(0) - bf * invz
        w.kf = k; w.point = point[q]; w.level = level[q];
        Q[i] = w;
    }
    if (n_desc) memcpy(L.host<uint8_t>(o_pd), point_desc, (size_t)n_desc * 32);
    FuseArgs A{};
    A.n_kf = n_kf; A.kfs = L.dev<FuseKF>(o_kf); A.nq = nv; A.q = L.dev<FuseQuery>(o_q); A.pdesc = L.dev<uint8_t>(o_pd);
    A.th_dist = 50;                                                          // TH_LOW, src/ORBmatcher1.cc:37
    A.match = L.dev<int>(o_match);
    cudaStream_t st = L.A.st;
    cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_fuse(A, gate, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(L.host<int>(o_match), A.match, (size_t)nv * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "%s: %s", name, cudaGetErrorString(e));
    const int* m = L.host<int>(o_match);
    k = 0;
    for (int i = 0; i < nv; ++i) {
        const int q = live[i];
        while (q >= kf_offsets[k + 1]) ++k;
        if (m[i] >= 0) { match[q] = m[i]; ++n_fused[k]; }
    }
    return ORBX_OK;
}

}  // namespace

}  // namespace orbx

using namespace orbx;

extern "C" {

int orbx_projection_rounds(void) { return t_rounds; }

int orbx_assign_features_to_grid(int device, const orbx_frame_view* frame, int32_t* cell_start, int32_t* items)
{
    int rc;
    if ((rc = check_frame(frame, false))) return rc;
    if (!cell_start || (frame->n > 0 && !items)) return fail(ORBX_ERR_INVALID_ARG, "null output");
    Session S(device);
    if ((rc = S.begin(device, frame, 0, false))) return rc;
    if ((rc = S.upload_and_grid())) return rc;
    cudaError_t e = cudaMemcpyAsync(cell_start, S.A.cell_start, (GRID_CELLS + 1) * 4, cudaMemcpyDeviceToHost, S.stream());
    if (e == cudaSuccess) e = cudaStreamSynchronize(S.stream());
    if (e == cudaSuccess && cell_start[GRID_CELLS] > 0)
        e = cudaMemcpy(items, S.A.items, (size_t)cell_start[GRID_CELLS] * 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "assign_features_to_grid: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

int orbx_get_features_in_area(int device, const orbx_frame_view* frame, float x, float y, float r, int min_level, int max_level,
                              int32_t* out, int capacity, int* n_out)
{
    int rc;
    if ((rc = check_frame(frame, false))) return rc;
    if (!n_out || capacity < 0 || (capacity > 0 && !out)) return fail(ORBX_ERR_INVALID_ARG, "bad output arguments");
    Session S(device);
    if ((rc = S.begin(device, frame, 0, false, frame->n))) return rc;
    if ((rc = S.upload_and_grid())) return rc;
    int* d_n = S.L.dev<int>(S.o_area_n);
    unsigned long long* d_out = S.L.dev<unsigned long long>(S.o_area);
    cudaError_t e = launch_features_in_area(S.A, x, y, r, min_level, max_level, d_out, frame->n, d_n, S.stream());
    int cnt = 0;
    if (e == cudaSuccess) e = cudaMemcpyAsync(&cnt, d_n, 4, cudaMemcpyDeviceToHost, S.stream());
    if (e == cudaSuccess) e = cudaStreamSynchronize(S.stream());
    std::vector<unsigned long long> keys(cnt);
    if (e == cudaSuccess && cnt) e = cudaMemcpy(keys.data(), d_out, (size_t)cnt * 8, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "get_features_in_area: %s", cudaGetErrorString(e));
    *n_out = cnt;
    if (cnt > capacity) return fail(ORBX_ERR_CAPACITY, "get_features_in_area: %d candidates, capacity %d", cnt, capacity);
    std::sort(keys.begin(), keys.end());                      // (cell id, index) = the reference's visiting order
    for (int i = 0; i < cnt; ++i) out[i] = (int32_t)(uint32_t)keys[i];
    return ORBX_OK;
}

int orbx_search_by_projection_map(int device, const orbx_frame_view* frame, const orbx_track_points* p, float th, int far_points,
                                  float th_far_points, float nn_ratio, int32_t* match_f, int* n_matches)
{
    int rc;
    if ((rc = check_frame(frame, true))) return rc;
    if (!p || p->n < 0 || !n_matches || (frame->n > 0 && !match_f)) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (p->n > 0 && (!p->in_view || !p->bad || !p->proj_x || !p->proj_y || !p->proj_xr || !p->view_cos || !p->scale_level || !p->n_obs ||
                     !p->descriptors || (far_points && !p->track_depth)))
        return fail(ORBX_ERR_INVALID_ARG, "track points: missing arrays");
    *n_matches = 0;
    for (int i = 0; i < frame->n; ++i) match_f[i] = -1;
    if (frame->n == 0 || p->n == 0) { t_rounds = 0; return ORBX_OK; }
    Session S(device);
    if ((rc = S.begin(device, frame, p->n, true))) return rc;
    ProjQuery* q = S.queries();
    const bool bFactor = th != 1.0;
    for (int i = 0; i < p->n; ++i) {
        ProjQuery w{};
        bool ok = p->in_view[i] != 0;                                        // src/ORBmatcher1.cc:54-55 (mbTrackInViewR: two-fisheye only)
        if (ok && far_points && p->track_depth[i] > th_far_points) ok = false;   // :57-58
        if (ok && p->bad[i]) ok = false;                                     // :60-61
        if (ok) {
            const int lvl = p->scale_level[i];
            if (lvl < 0 || lvl >= frame->n_levels) return fail(ORBX_ERR_INVALID_ARG, "track point %d: scale level %d out of range", i, lvl);
            float r = radius_by_viewing_cos(p->view_cos[i]);                 // :68
            if (bFactor) r *= th;                                            // :70-71
            w.x = p->proj_x[i]; w.y = p->proj_y[i];
            w.r = r * frame->scale_factors[lvl];                             // :74
            w.ur = p->proj_xr[i];
            w.min_level = lvl - 1; w.max_level = lvl;
            w.flags = PROJ_Q_VALID | PROJ_Q_CHECK_RIGHT | (p->n_obs[i] > 0 ? PROJ_Q_TAKES : 0);
        }
        q[i] = w;
    }
    memcpy(S.qdesc(), p->descriptors, (size_t)p->n * 32);
    if ((rc = S.search(0, 100 /* TH_HIGH, src/ORBmatcher1.cc:37 */, nn_ratio))) return rc;
    int nm = 0;
    for (int i = 0; i < p->n; ++i)
        if (S.qmatch()[i] >= 0) { match_f[S.qmatch()[i]] = i; ++nm; }       // later map points overwrite earlier un-observed ones
    *n_matches = nm;
    return ORBX_OK;
}

int orbx_search_by_projection_last(int device, const orbx_frame_view* cur, float mbf, int n_last, const uint8_t* valid, const float* u,
                                   const float* v, const float* invz, const int32_t* octave, const float* angle, const int32_t* n_obs,
                                   const uint8_t* desc, float th, int forward, int backward, int check_orientation, int32_t* match_f,
                                   int* n_matches)
{
    int rc;
    if ((rc = check_frame(cur, true))) return rc;
    if (n_last < 0 || !n_matches || (cur->n > 0 && !match_f) ||
        (n_last > 0 && (!valid || !u || !v || !invz || !octave || !n_obs || !desc || (check_orientation && !angle))))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    *n_matches = 0;
    for (int i = 0; i < cur->n; ++i) match_f[i] = -1;
    if (cur->n == 0 || n_last == 0) { t_rounds = 0; return ORBX_OK; }
    Session S(device);
    if ((rc = S.begin(device, cur, n_last, true))) return rc;
    ProjQuery* q = S.queries();
    for (int i = 0; i < n_last; ++i) {
        ProjQuery w{};
        bool ok = valid[i] != 0;
        const float invzc = ok ? invz[i] : 0.0f;
        if (ok && invzc < 0) ok = false;                                                         // src/ORBmatcher3.cc:293-294
        if (ok && (u[i] < cur->min_x || u[i] > cur->max_x)) ok = false;                          // :298-299
        if (ok && (v[i] < cur->min_y || v[i] > cur->max_y)) ok = false;                          // :300-301
        if (ok) {
            const int oct = octave[i];
            if (oct < 0 || oct >= cur->n_levels) return fail(ORBX_ERR_INVALID_ARG, "last-frame feature %d: octave %d out of range", i, oct);
            w.x = u[i]; w.y = v[i];
            w.r = th * cur->scale_factors[oct];                                                  // :307
            if (forward) { w.min_level = oct; w.max_level = -1; }                                // :311-316
            else if (backward) { w.min_level = 0; w.max_level = oct; }
            else { w.min_level = oct - 1; w.max_level = oct + 1; }
            w.ur = u[i] - mbf * invzc;                                                           // :332
            w.flags = PROJ_Q_VALID | PROJ_Q_CHECK_RIGHT | (n_obs[i] > 0 ? PROJ_Q_TAKES : 0);
        }
        q[i] = w;
    }
    memcpy(S.qdesc(), desc, (size_t)n_last * 32);
    if ((rc = S.search(1, 100 /* TH_HIGH */, 0.0f))) return rc;
    return finish_1nn(S, cur, angle, check_orientation, match_f, n_matches);
}

int orbx_search_by_projection_kf(int device, const orbx_frame_view* cur, int n_kf, const uint8_t* valid, const float* u, const float* v,
                                 const float* dist3d, const float* min_dist, const float* max_dist, const int32_t* level,
                                 const float* angle, const uint8_t* desc, float th, int orb_dist, int check_orientation,
                                 int32_t* match_f, int* n_matches)
{
    int rc;
    if ((rc = check_frame(cur, true))) return rc;
    if (n_kf < 0 || !n_matches || (cur->n > 0 && !match_f) ||
        (n_kf > 0 && (!valid || !u || !v || !dist3d || !min_dist || !max_dist || !level || !desc || (check_orientation && !angle))))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    *n_matches = 0;
    for (int i = 0; i < cur->n; ++i) match_f[i] = -1;
    if (cur->n == 0 || n_kf == 0) { t_rounds = 0; return ORBX_OK; }
    Session S(device);
    if ((rc = S.begin(device, cur, n_kf, true))) return rc;
    ProjQuery* q = S.queries();
    for (int i = 0; i < n_kf; ++i) {
        ProjQuery w{};
        bool ok = valid[i] != 0;
        if (ok && (u[i] < cur->min_x || u[i] > cur->max_x)) ok = false;                          // src/ORBmatcher3.cc:498-499
        if (ok && (v[i] < cur->min_y || v[i] > cur->max_y)) ok = false;                          // :500-501
        if (ok && (dist3d[i] < min_dist[i] || dist3d[i] > max_dist[i])) ok = false;              // :511-512
        if (ok) {
            const int lvl = level[i];
            if (lvl < 0 || lvl >= cur->n_levels) return fail(ORBX_ERR_INVALID_ARG, "key-frame point %d: level %d out of range", i, lvl);
            w.x = u[i]; w.y = v[i];
            w.r = th * cur->scale_factors[lvl];                                                  // :517
            w.min_level = lvl - 1; w.max_level = lvl + 1;                                        // :519
            w.flags = PROJ_Q_VALID | PROJ_Q_TAKES;                                               // any map point occupies (:533)
        }
        q[i] = w;
    }
    memcpy(S.qdesc(), desc, (size_t)n_kf * 32);
    if ((rc = S.search(1, orb_dist, 0.0f))) return rc;
    return finish_1nn(S, cur, angle, check_orientation, match_f, n_matches);
}

int orbx_search_for_initialization(int device, const orbx_keypoint* kp1, const uint8_t* desc1, int n1, const orbx_frame_view* f2,
                                   float* prev_matched, int window_size, float nn_ratio, int check_orientation, int32_t* matches12,
                                   int* n_matches)
{
    int rc;
    if ((rc = check_frame(f2, false))) return rc;
    if (f2->n > 0 && !f2->descriptors) return fail(ORBX_ERR_INVALID_ARG, "frame view: descriptors missing");
    if (n1 < 0 || n1 >= (1 << 24) || !n_matches || (n1 > 0 && (!kp1 || !desc1 || !prev_matched || !matches12)))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    *n_matches = 0;
    for (int i = 0; i < n1; ++i) matches12[i] = -1;
    if (n1 == 0 || f2->n == 0) { t_rounds = 0; return ORBX_OK; }
    // neither mvuRight nor the map points of F2 take part in this search
    orbx_frame_view v = *f2;
    v.u_right = nullptr; v.occupied = nullptr;
    Session S(device);
    if ((rc = S.begin(device, &v, n1, true))) return rc;
    S.enable_chains();
    ProjQuery* q = S.queries();
    for (int i = 0; i < n1; ++i) {
        ProjQuery w{};
        const int level1 = kp1[i].octave;
        if (level1 <= 0) {                                                   // src/ORBmatcher1.cc:650-765: 'if(level1>0) continue;'
            w.x = prev_matched[2 * i]; w.y = prev_matched[2 * i + 1];
            w.r = (float)window_size;
            w.min_level = level1; w.max_level = level1;                       // GetFeaturesInArea(.., windowSize, level1, level1)
            w.flags = PROJ_Q_VALID;
        }
        q[i] = w;
    }
    memcpy(S.qdesc(), desc1, (size_t)n1 * 32);
    if ((rc = S.search(2, 50 /* TH_LOW, src/ORBmatcher1.cc:37 */, nn_ratio))) return rc;
    // Replay of the reference's bookkeeping in query order: qmatch holds every acceptance, including the ones a later query
    // took over (vnMatches21 / vMatchedDistance), and the rotation histogram counts those too.
    const int H = 30;
    std::vector<int> m12(n1, -1), m21(f2->n, -1);
    std::vector<int> rot[H];
    int nm = 0;
    for (int i = 0; i < n1; ++i) {
        const int f = S.qmatch()[i];
        if (f < 0) continue;
        if (m21[f] >= 0) { m12[m21[f]] = -1; --nm; }
        m12[i] = f; m21[f] = i; ++nm;
        if (check_orientation) {
            const int b = rotation_bin(kp1[i].angle, f2->keys_un[f].angle);
            if (b < 0) return fail(ORBX_ERR_INVALID_ARG, "keypoint angles out of range (the reference asserts)");
            rot[b].push_back(i);
        }
    }
    if (check_orientation) {
        int count[H], i1, i2, i3;
        for (int b = 0; b < H; ++b) count[b] = (int)rot[b].size();
        three_maxima(count, H, i1, i2, i3);
        for (int b = 0; b < H; ++b) {
            if (b == i1 || b == i2 || b == i3) continue;
            for (int i : rot[b])
                if (m12[i] >= 0) { m12[i] = -1; --nm; }
        }
    }
    for (int i = 0; i < n1; ++i) {
        matches12[i] = m12[i];
        if (m12[i] >= 0) { prev_matched[2 * i] = f2->keys_un[m12[i]].x; prev_matched[2 * i + 1] = f2->keys_un[m12[i]].y; }
    }
    *n_matches = nm;
    return ORBX_OK;
}

int orbx_search_by_projection_sim3(int device, const orbx_frame_view* kf, int n_points, const uint8_t* valid, const float* u,
                                   const float* v, const int32_t* level, const uint8_t* desc, float th, float ratio_hamming,
                                   int32_t* match_f, int* n_matches)
{
    int rc;
    if ((rc = check_frame(kf, true))) return rc;
    if (n_points < 0 || !n_matches || (kf->n > 0 && !match_f) || (n_points > 0 && (!valid || !u || !v || !level || !desc)))
        return fail(ORBX_ERR_INVALID_ARG, "search_by_projection_sim3: bad arguments");
    // 'bestDist <= TH_LOW * ratioHamming': int times float, compared in float.  bestDist is at most 256 and starts there, so the
    // threshold is the largest integer d with (float)d <= the product; at 256 or more the reference writes vpMatched[-1].
    const float lim = 50.0f * ratio_hamming;
    if (!(lim < 256.0f)) return fail(ORBX_ERR_INVALID_ARG, "search_by_projection_sim3: TH_LOW * ratio_hamming = %g must be below 256", (double)lim);
    const int th_dist = lim < 0.0f ? -1 : (int)lim;
    for (int i = 0; i < n_points; ++i)
        if (valid[i] && (level[i] < 0 || level[i] >= kf->n_levels))
            return fail(ORBX_ERR_INVALID_ARG, "search_by_projection_sim3: point %d: level %d out of range", i, level[i]);
    *n_matches = 0;
    for (int i = 0; i < kf->n; ++i) match_f[i] = -1;
    if (kf->n == 0 || n_points == 0) { t_rounds = 0; return ORBX_OK; }
    orbx_frame_view fv = *kf;
    fv.u_right = nullptr;                                                    // no mvuRight gate in this search
    Session S(device, g_loop_arena);
    if ((rc = S.begin(device, &fv, n_points, true))) return rc;
    ProjQuery* q = S.queries();
    for (int i = 0; i < n_points; ++i) {
        ProjQuery w{};
        // KeyFrame::IsInImage: x >= mnMinX && x < mnMaxX && y >= mnMinY && y < mnMaxY
        if (valid[i] && u[i] >= kf->min_x && u[i] < kf->max_x && v[i] >= kf->min_y && v[i] < kf->max_y) {
            const int lvl = level[i];
            w.x = u[i]; w.y = v[i];
            w.r = th * kf->scale_factors[lvl];                               // radius = th * mvScaleFactors[nPredictedLevel]
            w.min_level = lvl - 1; w.max_level = lvl;                        // kpLevel < nPredictedLevel - 1 || kpLevel > nPredictedLevel
            w.flags = PROJ_Q_VALID | PROJ_Q_TAKES;                           // vpMatched[bestIdx] = pMP: later points skip it
        }
        q[i] = w;
    }
    memcpy(S.qdesc(), desc, (size_t)n_points * 32);
    if ((rc = S.search(1, th_dist, 0.0f))) return rc;
    int nm = 0;
    for (int i = 0; i < n_points; ++i)
        if (S.qmatch()[i] >= 0) { match_f[S.qmatch()[i]] = i; ++nm; }
    *n_matches = nm;
    return ORBX_OK;
}

int orbx_fuse(int device, int n_kf, const orbx_keyframe_view* kfs, const int32_t* kf_offsets, int n_desc, const uint8_t* point_desc,
              const int32_t* point, const uint8_t* valid, const float* u, const float* v, const float* invz, const int32_t* level,
              float th, int32_t* match, int* n_fused)
{
    return fuse_search(device, g_fuse_arena, "fuse", true, n_kf, kfs, kf_offsets, n_desc, point_desc, point, valid, u, v, invz, level, th, match,
                       n_fused);
}

int orbx_fuse_sim3(int device, int n_kf, const orbx_keyframe_view* kfs, const int32_t* kf_offsets, int n_desc, const uint8_t* point_desc,
                   const int32_t* point, const uint8_t* valid, const float* u, const float* v, const int32_t* level, float th,
                   int32_t* match, int* n_fused)
{
    return fuse_search(device, g_loop_arena, "fuse_sim3", false, n_kf, kfs, kf_offsets, n_desc, point_desc, point, valid, u, v, nullptr, level,
                       th, match, n_fused);
}

}  // extern "C"
