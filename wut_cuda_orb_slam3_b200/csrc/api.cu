// api.cu — host side of liborbx.so: the C ABI of include/orbx.h over the sm_100a kernels.
//
// One orbx_extractor == one ORB_SLAM3::ORBextractor instance (reference include/ORBextractor.h:52-120): parameters,
// scale tables, a private CUDA stream and a device workspace sized for the current image shape.  There is no CPU
// fallback anywhere in this file: without a CUDA device every compute entry point returns ORBX_ERR_NO_DEVICE.
#include <algorithm>
#include <atomic>
#include <climits>
#include <cfloat>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>

#include "orbx_internal.cuh"
#include "introsort_replay.h"
#include "synth.h"

namespace orbx {

static thread_local std::string t_err;
static std::atomic<long long> g_launches{0};

void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    t_err = buf;
    return code;
}

#define CU(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e__ = (call);                                                                        \
        if (e__ != cudaSuccess)                                                                          \
            return fail(e__ == cudaErrorMemoryAllocation ? ORBX_ERR_OOM : ORBX_ERR_CUDA, "%s failed: %s", #call, \
                        cudaGetErrorString(e__));                                                        \
    } while (0)

static inline int cvRoundF(float v) { return (int)lrintf(v); }
static inline int cvRoundD(double v) { return (int)lrint(v); }
static inline int cvFloorF(float v) { int i = (int)v; return i - (i > v); }
static inline int reflect101(int i, int n)
{
    if (n == 1) return 0;
    while (i < 0 || i >= n) i = i < 0 ? -i : 2 * (n - 1) - i;
    return i;
}
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct Tables {
    std::vector<float> scale, inv, sigma2, invsigma2;
    std::vector<int> nfeat;
};

// ORBextractor::ORBextractor — reference src/ORBextractor.cc:410-447 (scaleFactor is stored as double, include/ORBextractor.h:105).
static void make_tables(Tables& t, int nfeatures, float scaleFactorF, int nlevels)
{
    const double scaleFactor = scaleFactorF;
    t.scale.assign(nlevels, 1.f); t.sigma2.assign(nlevels, 1.f);
    for (int i = 1; i < nlevels; ++i) {
        t.scale[i] = (float)(t.scale[i - 1] * scaleFactor);
        t.sigma2[i] = t.scale[i] * t.scale[i];
    }
    t.inv.resize(nlevels); t.invsigma2.resize(nlevels);
    for (int i = 0; i < nlevels; ++i) { t.inv[i] = 1.0f / t.scale[i]; t.invsigma2[i] = 1.0f / t.sigma2[i]; }
    t.nfeat.assign(nlevels, 0);
    const float factor = (float)(1.0f / scaleFactor);
    float nDesired = nfeatures * (1 - factor) / (1 - (float)pow((double)factor, (double)nlevels));
    int sum = 0;
    for (int level = 0; level < nlevels - 1; ++level) {
        t.nfeat[level] = cvRoundF(nDesired);
        sum += t.nfeat[level];
        nDesired *= factor;
    }
    t.nfeat[nlevels - 1] = std::max(nfeatures - sum, 0);
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_tiled()
{
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            p = nullptr;
        }
        return (EncodeTiledFn)p;
    }();
    return fn;
}

struct Slot {
    Workspace ws{};
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_in = nullptr, ev_done = nullptr, ev_out = nullptr;   // H2D complete / compute complete / D2H complete (serial-compute pipeline)
    cudaEvent_t ev_cnt = nullptr;                                       // the chunk's per-frame counts have reached the host
    int cap_frames = 0;
    // staging for the host-buffer API
    uint8_t* d_in = nullptr; size_t d_in_bytes = 0;
    uint8_t* d_color = nullptr; size_t d_color_bytes = 0;      // colour input of orbx_extract_color
    orbx_keypoint* d_kps = nullptr; uint8_t* d_desc = nullptr; int* d_n = nullptr; int* d_nm = nullptr;
    size_t out_cap = 0;            // keypoint rows the output staging holds
    int out_frames = 0;            // frames the per-frame counters hold
    // stereo batches: mvuRight / mvDepth staging of the host-buffer call and the matcher's SAD scratch, [pairs][capacity]
    float* d_su = nullptr; float* d_sd = nullptr; int* d_sad = nullptr;
    int* d_snm = nullptr;          // [2 * pairs] monoIndex scratch of the device call (stereo outputs have no n_mono)
    size_t stereo_rows = 0; int stereo_pairs = 0;
    std::vector<void*> allocs;
};

int rotation_bin(float angle_a, float angle_b)
{
    const int HISTO_LENGTH = 30;
    const float factor = 1.0f / HISTO_LENGTH;                 // src/ORBmatcher1.cc:238 (sic: bins are 30 degrees wide)
    float rot = angle_a - angle_b;
    if (rot < 0.0) rot += 360.0f;
    int b = (int)round(rot * factor);
    if (b == HISTO_LENGTH) b = 0;
    return (b < 0 || b >= HISTO_LENGTH) ? -1 : b;
}

void three_maxima(const int* count, int L, int& ind1, int& ind2, int& ind3)
{
    int max1 = 0, max2 = 0, max3 = 0;
    ind1 = ind2 = ind3 = -1;
    for (int i = 0; i < L; i++) {
        const int s = count[i];
        if (s > max1) { max3 = max2; max2 = max1; max1 = s; ind3 = ind2; ind2 = ind1; ind1 = i; }
        else if (s > max2) { max3 = max2; max2 = s; ind3 = ind2; ind2 = i; }
        else if (s > max3) { max3 = s; ind3 = i; }
    }
    if (max2 < 0.1f * (float)max1) { ind2 = -1; ind3 = -1; }
    else if (max3 < 0.1f * (float)max1) { ind3 = -1; }
}


}  // namespace orbx

using namespace orbx;

struct orbx_extractor {
    int nfeatures, nlevels, iniTh, minTh, device;
    float scaleFactorF;
    Tables tab;
    FrameGeom fg{};
    bool geom_valid = false;
    uint2* d_tables = nullptr;     // resize tables
    size_t per_frame_pyr = 0, per_frame_blur = 0;
    int max_batch = 0;
    static const int kSlots = 6;
    Slot slots[kSlots];
    cudaStream_t compute = nullptr, copy_in = nullptr, copy_out = nullptr;   // serial-compute pipeline of orbx_extract_batch (3 streams)
    int last_frames = 0;           // frames of the last call that are probe-able (slot 0)
    // orbx_extract_batch_device on a caller's stream: an event recorded behind its last launch.  orbx_sync, the probes,
    // stereo matching, re-configuration and the next extraction on the extractor's own streams wait for it.
    cudaEvent_t ev_user = nullptr;
    bool user_pending = false;
    int max_kp = 0;
    // single-frame calls replay a captured CUDA graph of the 15 kernel launches (orbx_extract is the tracking thread's per-frame call:
    // launch gaps, not kernels, dominate it).  The graph is keyed by everything the captured launches bake in.
    struct GraphKey {
        int rows = 0, cols = 0, lap0 = 0, lap1 = 0, capacity = 0, cap_frames = 0;
        const void* pyr = nullptr; const void* d_in = nullptr; const void* d_kps = nullptr; const void* cand = nullptr;
        const void* d_n = nullptr; const void* tables = nullptr; const void* mirror = nullptr;
        bool operator==(const GraphKey& o) const
        {
            return mirror == o.mirror && rows == o.rows && cols == o.cols && lap0 == o.lap0 && lap1 == o.lap1 && capacity == o.capacity && cap_frames == o.cap_frames &&
                   pyr == o.pyr && d_in == o.d_in && d_kps == o.d_kps && cand == o.cand && d_n == o.d_n && tables == o.tables;
        }
    } graph_key;
    cudaGraphExec_t graph_exec = nullptr;
    int single_calls = 0;          // the first single-frame call runs un-captured (lazy one-time initialisation inside the launchers)
    int graph_launches = 0;        // kernel launches one replay of the captured graph stands for
    // host mirror of the bordered pyramid (std::vector<cv::Mat> mvImagePyramid of the reference, read on the host by
    // Frame::ComputeStereoMatches): pinned storage, filled level by level on a copy branch while FAST / octree run
    bool mirror = false;
    bool mirror_valid = false;     // the mirror holds the pyramid of the LAST call (single-frame calls fill it, batch calls do not)
    uint8_t* h_mirror = nullptr; size_t h_mirror_bytes = 0;
    size_t mirror_off[ORBX_MAX_LEVELS] = {0};
    cudaStream_t mirror_stream = nullptr;
    cudaEvent_t ev_mirror = nullptr;
    bool force_eager = false;      // debug hooks that patch the workspace (orbx_debug_octree_timing) must not replay a captured graph
    // fork / join of the single-frame pipeline: FAST + octree of level l run on side[l] as soon as level l of the pyramid exists
    cudaStream_t side[ORBX_MAX_LEVELS] = {nullptr};
    cudaEvent_t ev_lvl[ORBX_MAX_LEVELS] = {nullptr}, ev_side[ORBX_MAX_LEVELS] = {nullptr};
    // per-stage CUDA-event timing (orbx_profile_begin / orbx_profile_end)
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;   // kStages+1 events per profiled chunk
    size_t ev_used = 0;
};

namespace orbx {

// Block the host until the last orbx_extract_batch_device call on a caller-supplied stream has finished with the workspace.
static void wait_user_work(orbx_extractor* ex)
{
    if (ex->user_pending && ex->ev_user) cudaEventSynchronize(ex->ev_user);
    ex->user_pending = false;
}

int set_device(int device)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
        cudaGetLastError();
        return fail(ORBX_ERR_NO_DEVICE, "no CUDA device visible: liborbx has no CPU fallback");
    }
    if (device < 0 || device >= n) return fail(ORBX_ERR_INVALID_ARG, "device %d out of range (%d visible)", device, n);
    CU(cudaSetDevice(device));
    // stream-ordered scratch (cudaMallocAsync in the matcher entry points) should stay in the pool between calls
    static std::atomic<unsigned long long> pool_ready{0};
    if (device < 64 && !(pool_ready.load(std::memory_order_relaxed) & (1ull << device))) {
        cudaMemPool_t pool = nullptr;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
        pool_ready.fetch_or(1ull << device, std::memory_order_relaxed);
    }
    return ORBX_OK;
}

static void free_slot(Slot& s)
{
    for (void* p : s.allocs) cudaFree(p);
    s.allocs.clear();
    s.ws = Workspace{};
    s.cap_frames = 0;
    s.d_in = nullptr; s.d_in_bytes = 0; s.d_color = nullptr; s.d_color_bytes = 0; s.d_kps = nullptr; s.d_desc = nullptr; s.d_n = nullptr; s.d_nm = nullptr;
    s.out_cap = 0; s.out_frames = 0;
    s.d_su = nullptr; s.d_sd = nullptr; s.d_sad = nullptr; s.d_snm = nullptr; s.stereo_rows = 0; s.stereo_pairs = 0;
}

// release one buffer of a slot early (a staging buffer that is being replaced by a larger one)
template <typename T>
static void dev_release(Slot& s, T*& p)
{
    if (!p) return;
    for (size_t i = 0; i < s.allocs.size(); ++i)
        if (s.allocs[i] == (void*)p) { s.allocs[i] = s.allocs.back(); s.allocs.pop_back(); break; }
    cudaFree((void*)p);
    p = nullptr;
}

template <typename T>
static int dev_alloc(Slot& s, T** out, size_t count)
{
    void* p = nullptr;
    CU(cudaMalloc(&p, std::max<size_t>(count * sizeof(T), 16)));
    s.allocs.push_back(p);
    *out = (T*)p;
    return ORBX_OK;
}

// Geometry for an image of rows x cols: level sizes (src/ORBextractor.cc:1312-1313), buffer layout, FAST cell grid
// (873-886), octree parameters (589-591), resize coefficient tables (OpenCV resizeLinear, 8U fixed point).
static int configure(orbx_extractor* ex, int rows, int cols)
{
    if (ex->geom_valid && ex->fg.rows == rows && ex->fg.cols == cols) return ORBX_OK;
    if (cols > kMaxDim || rows > kMaxDim) return fail(ORBX_ERR_UNSUPPORTED, "image %dx%d exceeds %d px per side", cols, rows, kMaxDim);
    // From here on the old geometry is gone: a failure below must leave the handle "unconfigured" (every entry point calls
    // configure() first and probes / stereo matching check geom_valid), never half-built with the previous shape's flag set.
    ex->geom_valid = false;
    ex->last_frames = 0;
    ex->mirror_valid = false;
    wait_user_work(ex);
    if (ex->graph_exec) { cudaGraphExecDestroy(ex->graph_exec); ex->graph_exec = nullptr; }
    for (int i = 0; i < orbx_extractor::kSlots; ++i) {
        if (ex->slots[i].stream) cudaStreamSynchronize(ex->slots[i].stream);
        cudaStream_t st = ex->slots[i].stream;
        free_slot(ex->slots[i]);
        ex->slots[i].stream = st;
    }
    if (ex->d_tables) { cudaFree(ex->d_tables); ex->d_tables = nullptr; }
    FrameGeom& fg = ex->fg;
    memset(&fg, 0, sizeof fg);
    fg.nlevels = ex->nlevels; fg.rows = rows; fg.cols = cols; fg.iniTh = ex->iniTh; fg.minTh = ex->minTh;
    size_t pyr_off = 0, blur_off = 0;
    unsigned long long cand_off = 0, oct_off = 0;
    int cell_base = 0, kp_base = 0;
    std::vector<uint2> tables;
    std::vector<size_t> xtab_off(ex->nlevels, 0), ytab_off(ex->nlevels, 0);
    for (int l = 0; l < ex->nlevels; ++l) {
        LevelGeom& g = fg.L[l];
        const float scale = ex->tab.inv[l];
        g.w = cvRoundF((float)cols * scale);
        g.h = cvRoundF((float)rows * scale);
        if (g.w <= 0 || g.h <= 0) return fail(ORBX_ERR_UNSUPPORTED, "level %d of a %dx%d image is empty", l, cols, rows);
        g.pitch = (int)align_up((size_t)kXPad + g.w + kEdge, 16);
        g.rows_alloc = g.h + 2 * kEdge;
        g.pyr_off = pyr_off;
        g.pyr_frame_stride = align_up((size_t)g.pitch * g.rows_alloc, 256);
        pyr_off += 0;   // level slabs are laid out after the batch size is known (see ensure_slot)
        g.bpitch = (int)align_up((size_t)g.w, 16);
        g.blur_off = blur_off;
        g.blur_frame_stride = align_up((size_t)g.bpitch * g.h, 256);
        g.scale = ex->tab.scale[l];
        g.inv_scale = ex->tab.inv[l];
        g.kp_size = (float)(int)(31 * ex->tab.scale[l]);           // PATCH_SIZE * mvScaleFactor[level] (src 1017)
        // FAST grid
        const int maxBX = g.w - kEdge + 3, maxBY = g.h - kEdge + 3;
        const float width = (float)(maxBX - kWinBorder), height = (float)(maxBY - kWinBorder);
        const float W = 35;
        g.nCols = width > 0 ? (int)(width / W) : 0;
        g.nRows = height > 0 ? (int)(height / W) : 0;
        if (g.nCols > 0 && g.nRows > 0) {
            g.wCell = (int)ceil(width / g.nCols);
            g.hCell = (int)ceil(height / g.nRows);
        } else {
            g.nCols = g.nRows = 0; g.wCell = g.hCell = 1;       // reference divides by zero here; we return no keypoints
        }
        if (g.wCell > kMaxCellDim || g.hCell > kMaxCellDim) return fail(ORBX_ERR_UNSUPPORTED, "cell %dx%d too large", g.wCell, g.hCell);
        g.cell_base = cell_base;
        cell_base += g.nCols * g.nRows;
        g.cell_cap = ((g.wCell + 1) / 2) * ((g.hCell + 1) / 2);
        g.cand_off = cand_off;
        g.cand_max = g.nCols * g.nRows * g.cell_cap;
        if ((long long)g.nCols * g.nRows * g.cell_cap >= (1 << 24)) return fail(ORBX_ERR_UNSUPPORTED, "level %d has too many candidate slots", l);
        cand_off += (unsigned long long)g.cand_max;
        g.oct_off = oct_off;
        oct_off += 5ull * g.cand_max + (unsigned long long)(g.nCols * g.nRows) + 16;
        // octree
        g.nfeat = ex->tab.nfeat[l];
        g.nIni = (width > 0 && height > 0) ? (int)round(width / height) : 0;   // src 589
        if (g.nIni > 64) return fail(ORBX_ERR_UNSUPPORTED, "aspect ratio %d:1 not supported", g.nIni);
        g.hX = g.nIni > 0 ? width / g.nIni : 1.f;                               // src 591
        {
            int maxRootW = 1;
            for (int i = 0; i < g.nIni; ++i) {
                const int ulx = (int)(g.hX * (float)i), urx = (int)(g.hX * (float)(i + 1));
                maxRootW = std::max(maxRootW, urx - ulx);
            }
            auto clog2 = [](int v) { int b = 0; while ((1 << b) < v) ++b; return b; };
            g.depth = std::max(clog2(maxRootW) + 1, clog2(std::max((int)height, 1))) + 1;
            g.root_bits = clog2(std::max(g.nIni, 1));
            if (2 * g.depth + g.root_bits > 32) return fail(ORBX_ERR_UNSUPPORTED, "quadtree path code needs %d bits", 2 * g.depth + g.root_bits);
        }
        g.kp_base = kp_base;
        g.kp_cap = std::max(g.nfeat + 4, 4 * g.nIni + 1);
        kp_base += g.kp_cap;
        // resize tables, indexed by bordered coordinates
        if (l > 0) {
            const LevelGeom& p = fg.L[l - 1];
            const double scale_x = 1. / ((double)g.w / p.w), scale_y = 1. / ((double)g.h / p.h);
            const int iscale_x = cvRoundD(scale_x), iscale_y = cvRoundD(scale_y);
            const bool area_fast = std::abs(scale_x - iscale_x) < DBL_EPSILON && std::abs(scale_y - iscale_y) < DBL_EPSILON;
            g.area2x = (area_fast && iscale_x == 2 && iscale_y == 2) ? 1 : 0;
            auto entry = [&](int d, double sc, int n) -> uint2 {
                if (g.area2x) return make_uint2((uint32_t)(2 * d) | ((uint32_t)(2 * d + 1) << 16), 1u | (1u << 16));
                float f = (float)((d + 0.5) * sc - 0.5);
                int s = cvFloorF(f);
                f -= s;
                if (s < 0) { s = 0; f = 0.f; }
                if (s >= n - 1) { s = n - 1; f = 0.f; }
                const int c0 = (short)cvRoundF((1.f - f) * 2048.f), c1 = (short)cvRoundF(f * 2048.f);
                const int s1 = std::min(s + 1, n - 1);
                return make_uint2((uint32_t)s | ((uint32_t)s1 << 16), (uint32_t)c0 | ((uint32_t)c1 << 16));
            };
            xtab_off[l] = tables.size();
            for (int bc = 0; bc < g.w + 2 * kEdge; ++bc) tables.push_back(entry(reflect101(bc - kEdge, g.w), scale_x, p.w));
            ytab_off[l] = tables.size();
            for (int br = 0; br < g.h + 2 * kEdge; ++br) tables.push_back(entry(reflect101(br - kEdge, g.h), scale_y, p.h));
        }
    }
    // TMA box of level l when it is the SOURCE of level l+1 (128x32 output tiles): the largest source window any tile needs
    std::vector<uint2> rp_tables;
    std::vector<size_t> rp_x_off(ex->nlevels + 1, 0), rp_y_off(ex->nlevels + 1, 0);
    for (int l = 0; l + 1 < ex->nlevels; ++l) {
        const LevelGeom& d = fg.L[l + 1];
        const uint2* xt = tables.data() + xtab_off[l + 1];
        const uint2* yt = tables.data() + ytab_off[l + 1];
        int bw = 0, bh = 0;
        for (int x0 = 0; x0 < d.w; x0 += 128) {
            const int x1 = std::min(x0 + 128, d.w) - 1;
            bw = std::max(bw, (int)(xt[kEdge + x1].x >> 16) - ((int)(xt[kEdge + x0].x & 0xffff) & ~15) + 1);   // box starts 16-byte aligned
        }
        for (int y0 = 0; y0 < d.h; y0 += 32) {
            const int y1 = std::min(y0 + 32, d.h) - 1;
            bh = std::max(bh, (int)(yt[kEdge + y1].x >> 16) - (int)(yt[kEdge + y0].x & 0xffff) + 1);
        }
        fg.L[l].tma_box_w = (int)align_up((size_t)bw, 16);
        fg.L[l].tma_box_h = bh;
        // the warp-streaming kernel (kernels_pyramid.cu: pyr_resize_pipe_kernel) works on the BORDERED level: items of 128 buffer
        // columns (from column kXPad - kEdge - 1, word aligned) x 16 bordered rows; a border pixel takes the taps of its mirror
        // image, so the window of an item at the rim is a little larger than 16 * scale rows.  Everything an item needs is
        // tabulated here: per (column tile, lane) the four coefficient words, the two 8-byte windows of the lane and the byte
        // selectors; per row strip the source rows in ascending order with the output row(s) each pair of rows produces (two at
        // the rim: a border row and its mirror image are the same bytes).
        fg.L[l].rp_box_w = fg.L[l].rp_box_h = 0;
        rp_x_off[l + 1] = rp_y_off[l + 1] = 0;
        if (d.area2x) continue;
        const int wb = d.w + 2 * kEdge, hb = d.h + 2 * kEdge;
        const int ntx = (wb + 1 + 127) / 128, nstrips = (hb + 15) / 16;
        int rw = 0, rh = 0;
        bool ok = true;
        std::vector<uint2> xl, ys;
        for (int ct = 0; ct < ntx; ++ct) {
            auto col = [&](int c) { return xt[std::min(std::max(c, 0), wb - 1)]; };
            int lo = INT_MAX, hi = 0;
            for (int c = ct * 128 - 1; c < ct * 128 + 127; ++c) {
                const uint2 e = col(c);
                lo = std::min(lo, (int)(e.x & 0xffff)); hi = std::max(hi, (int)(e.x & 0xffff));
                if ((e.x >> 16) != (e.x & 0xffff) + 1 && (e.y >> 16) != 0) ok = false;     // second tap = first + 1 unless its weight is 0
            }
            const int cbase = lo & ~15;
            rw = std::max(rw, hi + 2 - cbase);
            for (int lane = 0; lane < 32; ++lane) {
                const int bc0 = ct * 128 + 4 * lane - 1;
                int c[4]; uint32_t a[4], keep = 0;
                for (int j = 0; j < 4; ++j) {
                    c[j] = (int)(col(bc0 + j).x & 0xffff) - cbase; a[j] = col(bc0 + j).y;
                    if (bc0 + j >= 0 && bc0 + j < wb) keep |= 0xffu << (8 * j);
                }
                const int qA = std::min(c[0], c[1]) & ~3, qB = std::min(c[2], c[3]) & ~3;
                const int i0 = c[0] - qA, i1 = c[1] - qA, i2 = c[2] - qB, i3 = c[3] - qB;
                if (std::max(std::max(i0, i1), std::max(i2, i3)) > 6) ok = false;
                const uint32_t selA = (uint32_t)(i0 | ((i0 + 1) << 4) | (i1 << 8) | ((i1 + 1) << 12));
                const uint32_t selB = (uint32_t)(i2 | ((i2 + 1) << 4) | (i3 << 8) | ((i3 + 1) << 12));
                xl.push_back(make_uint2(a[0], a[1])); xl.push_back(make_uint2(a[2], a[3]));
                xl.push_back(make_uint2(selA | (selB << 16), (uint32_t)qA | ((uint32_t)qB << 16))); xl.push_back(make_uint2(keep, (uint32_t)cbase));
            }
        }
        std::vector<std::vector<uint2>> strips(nstrips);
        for (int sidx = 0; sidx < nstrips; ++sidx) {
            const int r0 = sidx * 16, r1 = std::min(r0 + 16, hb);
            int lo = INT_MAX, hi = 0;
            for (int r = r0; r < r1; ++r) {
                lo = std::min(lo, (int)(yt[r].x & 0xffff)); hi = std::max(hi, (int)(yt[r].x & 0xffff));
                if ((yt[r].x >> 16) != (yt[r].x & 0xffff) + 1 && (yt[r].y >> 16) != 0) ok = false;
            }
            const int nbox = hi + 2 - lo;
            rh = std::max(rh, nbox);
            // entry k (two uint2) describes the pair of source rows (lo + k - 1, lo + k): {b0, b1}, {first output row | (second + 1) << 16, 0};
            // first = 0xffff: the pair produces nothing
            std::vector<uint2> e((size_t)nbox * 2, make_uint2(0u, 0u));
            for (int k = 0; k < nbox; ++k) e[2 * k + 1].x = 0xffffu;
            for (int r = r0; r < r1; ++r) {
                const int k = (int)(yt[r].x & 0xffff) - lo + 1;
                uint2& wgt = e[2 * k]; uint2& rows = e[2 * k + 1];
                const uint2 b = make_uint2(yt[r].y & 0xffffu, yt[r].y >> 16);
                if (rows.x == 0xffffu) { wgt = b; rows.x = (uint32_t)(r - r0); }
                else if ((rows.x >> 16) == 0 && wgt.x == b.x && wgt.y == b.y) rows.x |= (uint32_t)(r - r0 + 1) << 16;
                else ok = false;
            }
            strips[sidx].push_back(make_uint2((uint32_t)lo, (uint32_t)nbox));
            strips[sidx].push_back(make_uint2(0u, 0u));
            strips[sidx].insert(strips[sidx].end(), e.begin(), e.end());
        }
        if (!ok || rh > 31) continue;
        for (auto& sv : strips) { sv.resize(2 * ((size_t)rh + 1), make_uint2(0xffffu, 0u)); ys.insert(ys.end(), sv.begin(), sv.end()); }
        fg.L[l].rp_box_w = (int)align_up((size_t)rw, 16);
        fg.L[l].rp_box_h = rh;
        if (rp_tables.size() & 1) rp_tables.push_back(make_uint2(0, 0));            // 16-byte aligned lane records
        rp_x_off[l + 1] = rp_tables.size(); rp_tables.insert(rp_tables.end(), xl.begin(), xl.end());
        rp_y_off[l + 1] = rp_tables.size(); rp_tables.insert(rp_tables.end(), ys.begin(), ys.end());
    }
    if (tables.size() & 1) tables.push_back(make_uint2(0, 0));
    const size_t rp_base = tables.size();
    tables.insert(tables.end(), rp_tables.begin(), rp_tables.end());
    fg.total_cells = cell_base;
    fg.kp_slots = kp_base;
    for (int l = ex->nlevels; l < kMaxLevels; ++l) fg.L[l].kp_base = INT_MAX;      // slot -> level is a binary search over all kMaxLevels entries
    fg.cand_frame_stride = cand_off + 16;
    fg.oct_frame_stride = oct_off + 16;
    ex->max_kp = kp_base;
    // cell table (FAST kernel: global cell id -> level | cell row << 4 | cell column << 16), stored after the resize tables
    const size_t cell_tab_off = tables.size();
    {
        std::vector<uint32_t> flat;
        for (int l = 0; l < ex->nlevels; ++l)
            for (int i = 0; i < fg.L[l].nRows; ++i)
                for (int j = 0; j < fg.L[l].nCols; ++j) flat.push_back((uint32_t)l | ((uint32_t)i << 4) | ((uint32_t)j << 16));
        if (flat.size() & 1) flat.push_back(0);
        for (size_t k = 0; k < flat.size(); k += 2) tables.push_back(make_uint2(flat[k], flat[k + 1]));
    }
    if (!tables.empty()) {
        CU(cudaMalloc((void**)&ex->d_tables, tables.size() * sizeof(uint2)));
        CU(cudaMemcpy(ex->d_tables, tables.data(), tables.size() * sizeof(uint2), cudaMemcpyHostToDevice));
        for (int l = 1; l < ex->nlevels; ++l) {
            fg.L[l].xtab = ex->d_tables + xtab_off[l];
            fg.L[l].ytab = ex->d_tables + ytab_off[l];
            fg.L[l].rp_xlane = fg.L[l - 1].rp_box_w > 0 ? ex->d_tables + rp_base + rp_x_off[l] : nullptr;
            fg.L[l].rp_ysched = fg.L[l - 1].rp_box_w > 0 ? ex->d_tables + rp_base + rp_y_off[l] : nullptr;
        }
        fg.cell_tab = reinterpret_cast<const uint32_t*>(ex->d_tables + cell_tab_off);
    }
    const size_t smem = octree_smem_for(fg, 0, fg.nlevels);
    if (smem > 200 * 1024) return fail(ORBX_ERR_UNSUPPORTED, "nfeatures too large for the octree kernel (%zu B shared memory)", smem);
    CU(octree_prepare());
    ex->geom_valid = true;
    return ORBX_OK;
}

// (Re)allocate a slot's workspace for `frames` frames.  Level slabs are [level][frame].
static int ensure_slot(orbx_extractor* ex, Slot& s, int frames)
{
    if (!s.stream) CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    if (!s.ev_in) {
        CU(cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.ev_out, cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&s.ev_cnt, cudaEventDisableTiming));
    }
    if (s.cap_frames >= frames) return ORBX_OK;
    cudaStreamSynchronize(s.stream);
    free_slot(s);
    FrameGeom& fg = ex->fg;
    // offsets depend on the slot capacity; all slots of an extractor share one capacity so fg is consistent
    size_t pyr = 0, blur = 0;
    for (int l = 0; l < fg.nlevels; ++l) {
        fg.L[l].pyr_off = pyr; pyr += fg.L[l].pyr_frame_stride * (size_t)frames;
        fg.L[l].blur_off = blur; blur += fg.L[l].blur_frame_stride * (size_t)frames;
    }
    int rc;
    if ((rc = dev_alloc(s, &s.ws.pyr, pyr + 256))) return rc;
    if ((rc = dev_alloc(s, &s.ws.blur, blur + 256))) return rc;
    if ((rc = dev_alloc(s, &s.ws.cand, (size_t)fg.cand_frame_stride * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.cell_count, (size_t)std::max(fg.total_cells, 1) * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.oct, (size_t)fg.oct_frame_stride * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.lvl_kp, (size_t)fg.kp_slots * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.lvl_n, (size_t)fg.nlevels * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.lvl_ncand, (size_t)fg.nlevels * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.lvl_angle, (size_t)fg.kp_slots * frames))) return rc;
    if ((rc = dev_alloc(s, &s.ws.lvl_desc, (size_t)fg.kp_slots * frames * 32))) return rc;
    // TMA descriptors of the bordered pyramid levels (3-D: byte column, row, frame)
    s.ws.tmap_resize = nullptr; s.ws.tmap_blur = nullptr; s.ws.tmap_rpipe = nullptr; s.ws.tmap_desc = nullptr;
    if (EncodeTiledFn enc = get_encode_tiled()) {
        std::vector<CUtensorMap> maps(4 * kMaxLevels);
        bool ok_resize = true, ok_blur = true, ok_rpipe = true, ok_desc = true;
        for (int l = 0; l < fg.nlevels; ++l) {
            const LevelGeom& g = fg.L[l];
            const cuuint64_t dims[3] = {(cuuint64_t)g.pitch, (cuuint64_t)g.rows_alloc, (cuuint64_t)frames};
            const cuuint64_t strides[2] = {(cuuint64_t)g.pitch, (cuuint64_t)g.pyr_frame_stride};
            const cuuint32_t estr[3] = {1, 1, 1};
            void* base = s.ws.pyr + g.pyr_off;
            if (l + 1 < fg.nlevels) {
                const bool fits = g.tma_box_w > 0 && g.tma_box_w <= 224 && g.tma_box_h > 0 && g.tma_box_h <= 52;
                const cuuint32_t box[3] = {(cuuint32_t)std::max(g.tma_box_w, 16), (cuuint32_t)std::max(g.tma_box_h, 1), 1};
                if (!fits || enc(&maps[l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                 CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                    ok_resize = false;
            }
            if (l + 1 < fg.nlevels) {
                const bool fits = g.rp_box_w >= 16 && g.rp_box_w <= 256 && g.rp_box_h > 0 && g.rp_box_h <= 256;
                const cuuint32_t box[3] = {(cuuint32_t)std::max(g.rp_box_w, 16), (cuuint32_t)std::max(g.rp_box_h, 1), 1};
                if (!fits || enc(&maps[2 * kMaxLevels + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                 CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                    ok_rpipe = false;
            }
            {   // blurred level (no border): the window around a keypoint's descriptor patch
                const cuuint64_t bdims[3] = {(cuuint64_t)g.bpitch, (cuuint64_t)g.h, (cuuint64_t)frames};
                const cuuint64_t bstrides[2] = {(cuuint64_t)g.bpitch, (cuuint64_t)g.blur_frame_stride};
                const cuuint32_t dbox[3] = {kDescBoxW, kDescBoxH, 1};
                if (enc(&maps[3 * kMaxLevels + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, s.ws.blur + g.blur_off, bdims, bstrides, dbox, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                    ok_desc = false;
            }
            const cuuint32_t bbox[3] = {160, 38, 1};
            if (enc(&maps[kMaxLevels + l], CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, base, dims, strides, bbox, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
                ok_blur = false;
        }
        CUtensorMap* d_maps = nullptr;
        if ((rc = dev_alloc(s, &d_maps, maps.size()))) return rc;
        CU(cudaMemcpy(d_maps, maps.data(), maps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
        // ORBX_NO_TMA: a test hook, the only way the suite reaches the kernels taken when no tensor maps can be built
        static const bool no_tma = getenv("ORBX_NO_TMA") != nullptr;
        if (ok_resize && !no_tma) s.ws.tmap_resize = d_maps;
        if (ok_blur && !no_tma) s.ws.tmap_blur = d_maps + kMaxLevels;
        if (ok_rpipe && !no_tma) s.ws.tmap_rpipe = d_maps + 2 * kMaxLevels;
        if (ok_desc && !no_tma) s.ws.tmap_desc = d_maps + 3 * kMaxLevels;
    }
    CU(cudaMemsetAsync(s.ws.pyr, 0, pyr + 256, s.stream));
    CU(cudaMemsetAsync(s.ws.lvl_n, 0, sizeof(int) * (size_t)fg.nlevels * frames, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    s.cap_frames = frames;
    return ORBX_OK;
}

// All slots must share one capacity because level offsets live in the (shared) FrameGeom.
static int ensure_capacity(orbx_extractor* ex, int frames, int nslots)
{
    int cap = ex->slots[0].cap_frames;
    bool grow = frames > cap;
    if (grow) {
        wait_user_work(ex);
        if (ex->graph_exec) { cudaGraphExecDestroy(ex->graph_exec); ex->graph_exec = nullptr; }
        for (int i = 0; i < orbx_extractor::kSlots; ++i) {
            cudaStream_t st = ex->slots[i].stream;
            if (st) cudaStreamSynchronize(st);
            free_slot(ex->slots[i]);
            ex->slots[i].stream = st;
        }
        cap = frames;
    }
    for (int i = 0; i < nslots; ++i) {
        int rc = ensure_slot(ex, ex->slots[i], cap);
        if (rc) return rc;
    }
    return ORBX_OK;
}

// Staging of the host-buffer API.  The caller has made sure no work is in flight on the slot when a buffer is replaced.
static int ensure_host_staging(Slot& s, size_t in_bytes, int frames, int capacity)
{
    int rc;
    if (s.d_in_bytes < in_bytes) {
        dev_release(s, s.d_in);
        s.d_in_bytes = 0;
        if ((rc = dev_alloc(s, &s.d_in, in_bytes))) return rc;
        s.d_in_bytes = in_bytes;
    }
    const size_t rows = (size_t)frames * capacity;
    if (s.out_cap < rows || !s.d_kps) {
        dev_release(s, s.d_kps); dev_release(s, s.d_desc);
        s.out_cap = 0;
        if ((rc = dev_alloc(s, &s.d_kps, rows))) return rc;
        if ((rc = dev_alloc(s, &s.d_desc, rows * 32))) return rc;
        s.out_cap = rows;
    }
    if (s.out_frames < frames || !s.d_n) {          // the per-frame counters follow the FRAME count, not rows
        dev_release(s, s.d_n); dev_release(s, s.d_nm);
        s.out_frames = 0;
        if ((rc = dev_alloc(s, &s.d_n, (size_t)frames))) return rc;
        if ((rc = dev_alloc(s, &s.d_nm, (size_t)frames))) return rc;
        s.out_frames = frames;
    }
    return ORBX_OK;
}

// Matcher staging of a stereo chunk of `pairs` pairs.  As above: nothing may be in flight on the slot.
static bool stereo_staging_fits(const Slot& s, int pairs, int capacity)
{
    return s.stereo_pairs >= pairs && s.stereo_rows >= (size_t)pairs * capacity;
}
static int ensure_stereo_staging(Slot& s, int pairs, int capacity)
{
    if (stereo_staging_fits(s, pairs, capacity)) return ORBX_OK;
    dev_release(s, s.d_su); dev_release(s, s.d_sd); dev_release(s, s.d_sad); dev_release(s, s.d_snm);
    s.stereo_rows = 0; s.stereo_pairs = 0;
    const size_t rows = (size_t)pairs * capacity;
    int rc;
    if ((rc = dev_alloc(s, &s.d_su, rows)) || (rc = dev_alloc(s, &s.d_sd, rows)) || (rc = dev_alloc(s, &s.d_sad, rows)) ||
        (rc = dev_alloc(s, &s.d_snm, 2 * (size_t)pairs)))
        return rc;
    s.stereo_rows = rows; s.stereo_pairs = pairs;
    return ORBX_OK;
}

// Chunk schedule of the host-buffer batches: the first host->device copy cannot overlap any compute, so the pipeline ramps
// up with a quarter and a half chunk before it settles on full chunks (shorter un-overlapped prologue) ...
static std::vector<std::pair<int, int>> chunk_schedule(int n, int chunk)
{
    std::vector<std::pair<int, int>> sched;          // (first item, items); no entry exceeds `chunk`
    int f0 = 0;
    const int ramp[2] = {std::max(chunk / 4, 1), std::max(chunk / 2, 1)};
    for (int r = 0; r < 2 && n - f0 > 2 * chunk; ++r) { sched.emplace_back(f0, ramp[r]); f0 += ramp[r]; }
    // ... and ramps down the same way: the compute of a chunk trails its upload, so what is left after the LAST upload
    // is one chunk of compute + its download — a quarter chunk instead of a full one (trace of a 4096-frame call:
    // 2.8 ms of tail behind 27.3 ms of back-to-back uploads)
    const int tail = n - f0 > 3 * chunk ? ramp[0] + ramp[1] : 0;
    while (f0 < n - tail) { const int nf = std::min(chunk, n - tail - f0); sched.emplace_back(f0, nf); f0 += nf; }
    if (tail) { sched.emplace_back(f0, ramp[1]); f0 += ramp[1]; sched.emplace_back(f0, ramp[0]); f0 += ramp[0]; }
    return sched;
}

// The whole per-chunk pipeline on one stream.
static const int kStages = 6;   // pyramid, fast, blur, octree, orient+describe, pack

static int prof_mark(orbx_extractor* ex, cudaStream_t st)
{
    if (!ex->profiling) return ORBX_OK;
    if (ex->ev_used == ex->ev_pool.size()) {
        cudaEvent_t e;
        CU(cudaEventCreate(&e));
        ex->ev_pool.push_back(e);
    }
    CU(cudaEventRecord(ex->ev_pool[ex->ev_used++], st));
    return ORBX_OK;
}

static int run_chunk(orbx_extractor* ex, Slot& s, const ChunkIO& io, int frames, int lap0, int lap1, cudaStream_t st)
{
    const FrameGeom& fg = ex->fg;
    int rc;
    ex->mirror_valid = false;          // only the forked single-frame pipeline sends the levels home
    if ((rc = prof_mark(ex, st))) return rc;
    CU(launch_pyramid(fg, s.ws, io, frames, st));
    if ((rc = prof_mark(ex, st))) return rc;
    // The blur depends on the pyramid only: for batches it runs on a side stream beside FAST and the octree.  While a FAST launch
    // is at full occupancy there is no room for a blur CTA (shared memory and registers are taken), but each of FAST's three
    // launches ends with a tail of half-empty SMs, and the blur's persistent CTAs fill those: 3.163 -> 3.088 ms per 512 frames.
    // (The blur beside the octree instead: no gain — the octree's four CTAs hold the whole register file of an SM.  FAST's three
    // launches alternating between two streams: 3.17 ms.  The octree of the first FAST group's levels beside the later FAST launches: 3.13 ms.)  Not while
    // profiling (the per-stage events assume one stream), not for a few frames (run_single_forked forks per level).
    const bool fork = !ex->profiling && frames >= 8;
    if (fork) {
        if (!ex->side[0]) CU(cudaStreamCreateWithFlags(&ex->side[0], cudaStreamNonBlocking));
        if (!ex->ev_lvl[0]) CU(cudaEventCreateWithFlags(&ex->ev_lvl[0], cudaEventDisableTiming));
        if (!ex->ev_side[0]) CU(cudaEventCreateWithFlags(&ex->ev_side[0], cudaEventDisableTiming));
        CU(cudaEventRecord(ex->ev_lvl[0], st));
        CU(cudaStreamWaitEvent(ex->side[0], ex->ev_lvl[0], 0));
        CU(launch_fast(fg, s.ws, frames, st));
        CU(launch_blur(fg, s.ws, frames, ex->side[0]));
        CU(cudaEventRecord(ex->ev_side[0], ex->side[0]));
        CU(launch_octree(fg, s.ws, frames, st));
        CU(cudaStreamWaitEvent(st, ex->ev_side[0], 0));
    } else {
        CU(launch_fast(fg, s.ws, frames, st));
        if ((rc = prof_mark(ex, st))) return rc;
        CU(launch_blur(fg, s.ws, frames, st));
        if ((rc = prof_mark(ex, st))) return rc;
        CU(launch_octree(fg, s.ws, frames, st));
    }
    if ((rc = prof_mark(ex, st))) return rc;
    bool fused = false;
    CU(launch_orient_describe(fg, s.ws, frames, st, lap0, lap1, io, &fused));
    if ((rc = prof_mark(ex, st))) return rc;
    if (!fused) CU(launch_pack(fg, s.ws, frames, lap0, lap1, io, st));
    if ((rc = prof_mark(ex, st))) return rc;
    return ORBX_OK;
}

// The single-frame pipeline (orbx_extract: what Frame::ExtractORB calls once per image, src/Frame.cc:420-455).  One frame
// cannot fill the GPU, so the stages are forked per pyramid level: as soon as level l exists, FAST and the quadtree of that
// level run on their own branch while the resize chain continues; the blur follows the chain; orientation + descriptors and
// the packing join everything.  The critical path is level 0 (pyramid copy -> FAST -> octree), not the sum of all stages.
// Works eagerly and under stream capture (the events become graph edges).
static int run_single_forked(orbx_extractor* ex, Slot& s, const uint8_t* d_image, size_t pitch, int lap0, int lap1,
                             orbx_keypoint* d_kps, uint8_t* d_desc, int capacity, int* d_n, int* d_nm, cudaStream_t st)
{
    const FrameGeom& fg = ex->fg;
    const ChunkIO io = one_set_io(d_image, pitch * fg.rows, pitch, d_kps, d_desc, capacity, d_n, d_nm);
    for (int l = 0; l < fg.nlevels; ++l) {
        if (!ex->side[l]) CU(cudaStreamCreateWithFlags(&ex->side[l], cudaStreamNonBlocking));
        if (!ex->ev_lvl[l]) CU(cudaEventCreateWithFlags(&ex->ev_lvl[l], cudaEventDisableTiming));
        if (!ex->ev_side[l]) CU(cudaEventCreateWithFlags(&ex->ev_side[l], cudaEventDisableTiming));
    }
    for (int l = 0; l < fg.nlevels; ++l) {
        CU(launch_pyramid(fg, s.ws, io, 1, st, l, l + 1));
        CU(cudaEventRecord(ex->ev_lvl[l], st));
        if (ex->mirror) {           // the level goes home while the later stages run
            const LevelGeom& g = fg.L[l];
            const size_t bw = (size_t)g.w + 2 * kEdge;
            CU(cudaStreamWaitEvent(ex->mirror_stream, ex->ev_lvl[l], 0));
            CU(cudaMemcpy2DAsync(ex->h_mirror + ex->mirror_off[l], bw, s.ws.pyr + g.pyr_off + (kXPad - kEdge), g.pitch, bw, (size_t)g.rows_alloc,
                                 cudaMemcpyDeviceToHost, ex->mirror_stream));
        }
        CU(cudaStreamWaitEvent(ex->side[l], ex->ev_lvl[l], 0));
        CU(launch_fast(fg, s.ws, 1, ex->side[l], l, l + 1));
        CU(launch_octree(fg, s.ws, 1, ex->side[l], l, l + 1));
        CU(cudaEventRecord(ex->ev_side[l], ex->side[l]));
    }
    CU(launch_blur(fg, s.ws, 1, st));
    for (int l = 0; l < fg.nlevels; ++l) CU(cudaStreamWaitEvent(st, ex->ev_side[l], 0));
    bool fused = false;
    CU(launch_orient_describe(fg, s.ws, 1, st, lap0, lap1, io, &fused));
    if (!fused) CU(launch_pack(fg, s.ws, 1, lap0, lap1, io, st));
    if (ex->mirror) { CU(cudaEventRecord(ex->ev_mirror, ex->mirror_stream)); CU(cudaStreamWaitEvent(st, ex->ev_mirror, 0)); }
    ex->mirror_valid = ex->mirror;
    return ORBX_OK;
}

// Pinned host storage + copy stream of the mvImagePyramid mirror for the current geometry (no-op when the mirror is off).
static int ensure_mirror(orbx_extractor* ex, cudaStream_t st)
{
    if (ex->mirror) {
        if (!ex->mirror_stream) CU(cudaStreamCreateWithFlags(&ex->mirror_stream, cudaStreamNonBlocking));
        if (!ex->ev_mirror) CU(cudaEventCreateWithFlags(&ex->ev_mirror, cudaEventDisableTiming));
        size_t need = 0;
        for (int l = 0; l < ex->fg.nlevels; ++l) {
            ex->mirror_off[l] = need;
            need += align_up(((size_t)ex->fg.L[l].w + 2 * kEdge) * (size_t)ex->fg.L[l].rows_alloc, 256);
        }
        if (ex->h_mirror_bytes < need) {
            CU(cudaStreamSynchronize(st));
            if (ex->h_mirror) cudaFreeHost(ex->h_mirror);
            ex->h_mirror = nullptr; ex->h_mirror_bytes = 0;
            CU(cudaMallocHost((void**)&ex->h_mirror, need));
            ex->h_mirror_bytes = need;
        }
    }
    return ORBX_OK;
}

// Upload one host image into slot 0 and queue its extraction on the slot's stream (captured graph after the first call).
// Results stay on the device (s.d_kps / s.d_desc / s.d_n / s.d_nm); nothing is copied back and nothing is waited for.
static int enqueue_single(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int lap0, int lap1, int capacity)
{
    int rc = set_device(ex->device);
    if (rc) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    wait_user_work(ex);
    if ((rc = ensure_capacity(ex, 1, 1))) return rc;
    Slot& s = ex->slots[0];
    const size_t dpitch = (size_t)cols, dframe = dpitch * rows;
    if (s.d_in_bytes < dframe || s.out_cap < (size_t)capacity || s.out_frames < 1) CU(cudaStreamSynchronize(s.stream));
    if ((rc = ensure_host_staging(s, dframe, 1, capacity))) return rc;
    cudaStream_t st = s.stream;
    if ((rc = ensure_mirror(ex, st))) return rc;
    if (step == (size_t)cols) CU(cudaMemcpyAsync(s.d_in, image, dframe, cudaMemcpyHostToDevice, st));
    else CU(cudaMemcpy2DAsync(s.d_in, dpitch, image, step, cols, rows, cudaMemcpyHostToDevice, st));
    auto body = [&](cudaStream_t cs) -> int {
        if (!ex->profiling || ex->mirror) return run_single_forked(ex, s, s.d_in, dpitch, lap0, lap1, s.d_kps, s.d_desc, capacity, s.d_n, s.d_nm, cs);
        return run_chunk(ex, s, one_set_io(s.d_in, dframe, dpitch, s.d_kps, s.d_desc, capacity, s.d_n, s.d_nm), 1, lap0, lap1, cs);
    };
    if (!ex->profiling && !ex->force_eager && ex->single_calls++ > 0) {
        orbx_extractor::GraphKey key;
        key.rows = rows; key.cols = cols; key.lap0 = lap0; key.lap1 = lap1; key.capacity = capacity;
        key.pyr = s.ws.pyr; key.d_in = s.d_in; key.d_kps = s.d_kps; key.cand = s.ws.cand;
        key.cap_frames = s.cap_frames; key.d_n = s.d_n; key.tables = ex->d_tables; key.mirror = ex->mirror ? ex->h_mirror : nullptr;
        if (!ex->graph_exec || !(key == ex->graph_key)) {
            if (ex->graph_exec) { cudaGraphExecDestroy(ex->graph_exec); ex->graph_exec = nullptr; }
            cudaGraph_t g = nullptr;
            const long long l0 = g_launches.load();
            CU(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
            rc = body(st);
            cudaError_t ce = cudaStreamEndCapture(st, &g);
            ex->graph_launches = (int)(g_launches.load() - l0);
            count_launch(-ex->graph_launches);              // captured, not launched: the replay below counts them
            if (rc) { if (g) cudaGraphDestroy(g); cudaGetLastError(); return rc; }
            if (ce != cudaSuccess) return fail(ORBX_ERR_CUDA, "graph capture: %s", cudaGetErrorString(ce));
            ce = cudaGraphInstantiate(&ex->graph_exec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { ex->graph_exec = nullptr; return fail(ORBX_ERR_CUDA, "graph instantiate: %s", cudaGetErrorString(ce)); }
            ex->graph_key = key;
        }
        CU(cudaGraphLaunch(ex->graph_exec, st));
        count_launch(ex->graph_launches);
    } else if ((rc = body(st))) return rc;
    ex->last_frames = 1;
    ex->mirror_valid = ex->mirror;     // (a graph replay does not pass through run_single_forked)
    return ORBX_OK;
}

// Grow-only device scratch per device for the matcher entry points that take host buffers (orbx_knn2, orbx_stereo_match): a
// cudaMalloc/cudaFree pair per call costs more than the kernels on frame-sized inputs.  One call at a time per device holds it.
struct ScratchArena {
    std::mutex mu;
    unsigned char* base = nullptr;
    size_t bytes = 0;
};
static ScratchArena g_scratch[64];

struct ScratchLease {
    ScratchArena& a;
    std::unique_lock<std::mutex> lock;
    size_t off = 0;
    explicit ScratchLease(int device) : a(g_scratch[device & 63]), lock(a.mu) {}
    int reserve(size_t total)
    {
        total += 4096;
        if (a.bytes >= total) return ORBX_OK;
        if (a.base) cudaFree(a.base);
        a.base = nullptr; a.bytes = 0;
        cudaError_t e = cudaMalloc(&a.base, total);
        if (e != cudaSuccess) return fail(ORBX_ERR_OOM, "cudaMalloc(%zu): %s", total, cudaGetErrorString(e));
        a.bytes = total;
        return ORBX_OK;
    }
    template <typename T> T* take(size_t count)
    {
        off = (off + 255) & ~(size_t)255;
        T* p = reinterpret_cast<T*>(a.base + off);
        off += std::max<size_t>(count, 1) * sizeof(T);
        return p;
    }
};

}  // namespace orbx

// =====================================================================================================================
extern "C" {

const char* orbx_last_error(void) { return t_err.c_str(); }
int orbx_version(void) { return ORBX_VERSION; }

int orbx_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int64_t orbx_launch_count(void) { return g_launches.load(); }

int orbx_compute_tables(int nfeatures, float scaleFactor, int nlevels, float* scale, float* inv_scale, float* sigma2,
                        float* inv_sigma2, int* nfeatures_per_level)
{
    if (nlevels <= 0 || nlevels > ORBX_MAX_LEVELS || nfeatures < 0 || !(scaleFactor > 1.0f))
        return fail(ORBX_ERR_INVALID_ARG, "bad extractor parameters (nfeatures=%d scaleFactor=%g nlevels=%d)", nfeatures, scaleFactor, nlevels);
    Tables t;
    make_tables(t, nfeatures, scaleFactor, nlevels);
    for (int i = 0; i < nlevels; ++i) {
        if (scale) scale[i] = t.scale[i];
        if (inv_scale) inv_scale[i] = t.inv[i];
        if (sigma2) sigma2[i] = t.sigma2[i];
        if (inv_sigma2) inv_sigma2[i] = t.invsigma2[i];
        if (nfeatures_per_level) nfeatures_per_level[i] = t.nfeat[i];
    }
    return ORBX_OK;
}

int orbx_create(int nfeatures, float scaleFactor, int nlevels, int iniThFAST, int minThFAST, int device, int max_cols,
                int max_rows, int max_batch, orbx_extractor** out)
{
    if (!out) return fail(ORBX_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (nlevels <= 0 || nlevels > ORBX_MAX_LEVELS || nfeatures <= 0 || !(scaleFactor > 1.0f) || iniThFAST < 1 || minThFAST < 1 ||
        iniThFAST > 255 || minThFAST > iniThFAST)
        return fail(ORBX_ERR_INVALID_ARG, "bad extractor parameters (nfeatures=%d scaleFactor=%g nlevels=%d ini=%d min=%d)", nfeatures,
                    scaleFactor, nlevels, iniThFAST, minThFAST);
    int rc = set_device(device);
    if (rc) return rc;
    orbx_extractor* ex = new orbx_extractor();
    ex->nfeatures = nfeatures; ex->nlevels = nlevels; ex->iniTh = iniThFAST; ex->minTh = minThFAST; ex->device = device;
    ex->scaleFactorF = scaleFactor;
    ex->max_batch = max_batch > 0 ? max_batch : 0;
    make_tables(ex->tab, nfeatures, scaleFactor, nlevels);
    int kp = 0;
    for (int l = 0; l < nlevels; ++l) kp += ex->tab.nfeat[l] + 4;
    ex->max_kp = kp;
    if (max_cols > 0 && max_rows > 0) {
        rc = configure(ex, max_rows, max_cols);
        if (!rc) rc = ensure_capacity(ex, std::max(max_batch, 1), 1);
        if (rc) { orbx_destroy(ex); return rc; }
    }
    *out = ex;
    return ORBX_OK;
}

void orbx_destroy(orbx_extractor* ex)
{
    if (!ex) return;
    cudaSetDevice(ex->device);
    if (ex->compute) { cudaStreamSynchronize(ex->compute); cudaStreamDestroy(ex->compute); ex->compute = nullptr; }
    if (ex->copy_in) { cudaStreamSynchronize(ex->copy_in); cudaStreamDestroy(ex->copy_in); ex->copy_in = nullptr; }
    if (ex->copy_out) { cudaStreamSynchronize(ex->copy_out); cudaStreamDestroy(ex->copy_out); ex->copy_out = nullptr; }
    for (int i = 0; i < orbx_extractor::kSlots; ++i) {
        if (ex->slots[i].stream) cudaStreamSynchronize(ex->slots[i].stream);
        free_slot(ex->slots[i]);
        if (ex->slots[i].stream) cudaStreamDestroy(ex->slots[i].stream);
        if (ex->slots[i].ev_in) { cudaEventDestroy(ex->slots[i].ev_in); cudaEventDestroy(ex->slots[i].ev_done); cudaEventDestroy(ex->slots[i].ev_out); cudaEventDestroy(ex->slots[i].ev_cnt); }
    }
    if (ex->ev_user) { cudaEventSynchronize(ex->ev_user); cudaEventDestroy(ex->ev_user); }
    if (ex->mirror_stream) { cudaStreamSynchronize(ex->mirror_stream); cudaStreamDestroy(ex->mirror_stream); }
    if (ex->ev_mirror) cudaEventDestroy(ex->ev_mirror);
    if (ex->h_mirror) cudaFreeHost(ex->h_mirror);
    for (int l = 0; l < ORBX_MAX_LEVELS; ++l) {
        if (ex->side[l]) { cudaStreamSynchronize(ex->side[l]); cudaStreamDestroy(ex->side[l]); }
        if (ex->ev_lvl[l]) cudaEventDestroy(ex->ev_lvl[l]);
        if (ex->ev_side[l]) cudaEventDestroy(ex->ev_side[l]);
    }
    if (ex->graph_exec) cudaGraphExecDestroy(ex->graph_exec);
    if (ex->d_tables) cudaFree(ex->d_tables);
    for (cudaEvent_t e : ex->ev_pool) cudaEventDestroy(e);
    delete ex;
}

int orbx_get_levels(const orbx_extractor* ex) { return ex ? ex->nlevels : 0; }
float orbx_get_scale_factor(const orbx_extractor* ex) { return ex ? (float)(double)ex->scaleFactorF : 0.f; }

int orbx_get_tables(const orbx_extractor* ex, float* scale, float* inv_scale, float* sigma2, float* inv_sigma2,
                    int* nfeatures_per_level)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    for (int i = 0; i < ex->nlevels; ++i) {
        if (scale) scale[i] = ex->tab.scale[i];
        if (inv_scale) inv_scale[i] = ex->tab.inv[i];
        if (sigma2) sigma2[i] = ex->tab.sigma2[i];
        if (inv_sigma2) inv_sigma2[i] = ex->tab.invsigma2[i];
        if (nfeatures_per_level) nfeatures_per_level[i] = ex->tab.nfeat[i];
    }
    return ORBX_OK;
}

int orbx_level_size(const orbx_extractor* ex, int cols, int rows, int level, int* level_cols, int* level_rows)
{
    if (!ex || level < 0 || level >= ex->nlevels) return fail(ORBX_ERR_INVALID_ARG, "bad level");
    const float scale = ex->tab.inv[level];
    if (level_cols) *level_cols = cvRoundF((float)cols * scale);
    if (level_rows) *level_rows = cvRoundF((float)rows * scale);
    return ORBX_OK;
}

int orbx_max_keypoints(const orbx_extractor* ex) { return ex ? ex->max_kp : 0; }

// The first sweep of DistributeOctTree splits all nIni = round(width / height) root nodes before it looks at N (src
// 589-608, 635-698), so a level of a wide image can return up to 4 * nIni keypoints however small mnFeaturesPerLevel is.
// Same per-level bound as configure() (kp_cap), from the shape alone: no GPU work, no change of the handle.
int orbx_max_keypoints_for(const orbx_extractor* ex, int rows, int cols)
{
    if (!ex || rows <= 0 || cols <= 0) return 0;
    int kp = 0;
    for (int l = 0; l < ex->nlevels; ++l) {
        const int w = cvRoundF((float)cols * ex->tab.inv[l]), h = cvRoundF((float)rows * ex->tab.inv[l]);
        const float width = (float)(w - kEdge + 3 - kWinBorder), height = (float)(h - kEdge + 3 - kWinBorder);
        const int nIni = (width > 0 && height > 0) ? (int)round(width / height) : 0;
        kp += std::max(ex->tab.nfeat[l] + 4, 4 * nIni + 1);
    }
    return kp;
}

int orbx_sync(orbx_extractor* ex)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    CU(cudaSetDevice(ex->device));
    for (int i = 0; i < orbx_extractor::kSlots; ++i)
        if (ex->slots[i].stream) CU(cudaStreamSynchronize(ex->slots[i].stream));
    if (ex->user_pending && ex->ev_user) CU(cudaEventSynchronize(ex->ev_user));    // work queued on a caller's stream
    ex->user_pending = false;
    return ORBX_OK;
}

int orbx_extract_batch_device(orbx_extractor* ex, const uint8_t* d_images, size_t frame_stride, int n_frames, int rows,
                              int cols, size_t pitch, int lap0, int lap1, orbx_keypoint* d_keypoints,
                              uint8_t* d_descriptors, int capacity, int* d_n_out, int* d_n_mono, void* stream)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    if (!d_images || rows <= 0 || cols <= 0 || n_frames <= 0) return fail(ORBX_ERR_EMPTY_IMAGE, "empty image");
    if (!d_keypoints || !d_descriptors || !d_n_out || !d_n_mono || capacity <= 0 || pitch < (size_t)cols)
        return fail(ORBX_ERR_INVALID_ARG, "bad output buffers / pitch");
    int rc = set_device(ex->device);
    if (rc) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    const int chunk = ex->max_batch > 0 ? std::min(ex->max_batch, n_frames) : std::min(n_frames, 256);
    if ((rc = ensure_capacity(ex, chunk, 1))) return rc;
    Slot& s = ex->slots[0];
    cudaStream_t st = stream ? (cudaStream_t)stream : s.stream;
    if (!ex->ev_user) CU(cudaEventCreateWithFlags(&ex->ev_user, cudaEventDisableTiming));
    // the workspace is shared with whatever ran before: earlier work on another stream must be complete first
    if (ex->user_pending) CU(cudaStreamWaitEvent(st, ex->ev_user, 0));
    if (st != s.stream) { CU(cudaEventRecord(s.ev_done, s.stream)); CU(cudaStreamWaitEvent(st, s.ev_done, 0)); }
    for (int f0 = 0; f0 < n_frames; f0 += chunk) {
        const int nf = std::min(chunk, n_frames - f0);
        rc = run_chunk(ex, s, one_set_io(d_images + (size_t)f0 * frame_stride, frame_stride, pitch, d_keypoints + (size_t)f0 * capacity,
                                         d_descriptors + (size_t)f0 * capacity * 32, capacity, d_n_out + f0, d_n_mono + f0),
                       nf, lap0, lap1, st);
        if (rc) return rc;
        ex->last_frames = nf;
    }
    if (st != s.stream) { CU(cudaEventRecord(ex->ev_user, st)); ex->user_pending = true; }
    return ORBX_OK;
}

int orbx_extract_batch(orbx_extractor* ex, const uint8_t* const* images, int n_frames, int rows, int cols, size_t step,
                       int lap0, int lap1, orbx_keypoint* keypoints, uint8_t* descriptors, int capacity, int* n_out,
                       int* n_mono)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    if (!images || rows <= 0 || cols <= 0 || n_frames <= 0) return fail(ORBX_ERR_EMPTY_IMAGE, "empty image");
    for (int i = 0; i < n_frames; ++i)
        if (!images[i]) return fail(ORBX_ERR_EMPTY_IMAGE, "image %d is NULL", i);
    if (!keypoints || !descriptors || !n_out || !n_mono || capacity <= 0 || step < (size_t)cols)
        return fail(ORBX_ERR_INVALID_ARG, "bad output buffers / step");
    if (n_frames == 1) return orbx_extract(ex, images[0], rows, cols, step, lap0, lap1, keypoints, descriptors, capacity, n_out, n_mono);
    int rc = set_device(ex->device);
    if (rc) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    wait_user_work(ex);
    const int chunk = ex->max_batch > 0 ? std::min(ex->max_batch, n_frames) : std::min(n_frames, 64);
    const std::vector<std::pair<int, int>> sched = chunk_schedule(n_frames, chunk);   // (first frame, frames)
    const int nchunks = (int)sched.size();
    const int nslots = std::min(nchunks, (int)orbx_extractor::kSlots);
    if ((rc = ensure_capacity(ex, chunk, nslots))) return rc;
    const size_t dpitch = (size_t)cols;
    const size_t dframe = dpitch * rows;
    for (int i = 0; i < nslots; ++i)
        if ((rc = ensure_host_staging(ex->slots[i], dframe * chunk, chunk, capacity))) return rc;
    // ORBX_TRACE_BATCH=1: per-chunk timeline (H2D start/end, compute end, D2H end; ms since the first H2D) on stderr
    static const bool trace = getenv("ORBX_TRACE_BATCH") != nullptr;
    std::vector<cudaEvent_t> tev;                    // [chunk][4]: H2D start / end, compute end (= D2H may start), D2H end
    auto mark = [&](cudaStream_t st, int chunk, int k) {
        if (!trace) return;
        if (tev.empty()) tev.assign((size_t)4 * sched.size(), nullptr);
        cudaEvent_t e; cudaEventCreate(&e); cudaEventRecord(e, st); tev[(size_t)4 * chunk + k] = e;
    };
    // Two pipelines.  Small chunks (< 128 frames) run whole on their slot's stream, so that chunks overlap each other (a small
    // chunk under-fills the GPU: its octree is one partial wave).  Large chunks compute on ONE stream in order: interleaving the
    // kernels of two big chunks costs ~20 % (measured: 80 k vs 98 k frames/s at 256-frame chunks).  The serial pipeline uses
    // exactly three streams — H2D, compute, D2H — tied by per-slot events: with one copy stream per slot (seven streams) two of
    // them regularly landed on the same hardware connection (8 by default) and a chunk's D2H or the next H2D queued behind an
    // unrelated copy (90.5 k frames/s; 97.9 k with CUDA_DEVICE_MAX_CONNECTIONS=32; 98 k with three streams at any setting).
    const bool serial = chunk >= 128;
    if (serial && !ex->compute) {
        CU(cudaStreamCreateWithFlags(&ex->compute, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&ex->copy_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&ex->copy_out, cudaStreamNonBlocking));
    }
    if (serial)      // earlier work of this extractor on the slot streams (single-frame calls, small batches) must be complete
        for (int i = 0; i < nslots; ++i) CU(cudaStreamSynchronize(ex->slots[i].stream));
    // Results go home trimmed: a chunk's per-frame counts are copied first (a few hundred bytes), the host reads them and
    // then asks for the keypoint / descriptor rows every frame of the chunk actually has — one strided copy per array, row
    // count = the chunk's largest n_out — instead of `capacity` rows per frame.  The host looks at the counts of chunk c - 2
    // after it has queued chunk c, so two chunks of compute are always queued behind the one it waits for and the next
    // upload never starts late.
    auto finish = [&](int c) -> int {
        Slot& s = ex->slots[c % nslots];
        const int f0 = sched[c].first, nf = sched[c].second;
        cudaStream_t ost = serial ? ex->copy_out : s.stream;
        CU(cudaEventSynchronize(s.ev_cnt));
        int mx = 0;
        for (int f = 0; f < nf; ++f) mx = std::max(mx, n_out[f0 + f]);
        const int rows_out = std::min(mx, capacity);   // a frame over capacity wrote nothing: the call fails below
        if (rows_out > 0) {
            CU(cudaMemcpy2DAsync(keypoints + (size_t)f0 * capacity, sizeof(orbx_keypoint) * (size_t)capacity, s.d_kps,
                                 sizeof(orbx_keypoint) * (size_t)capacity, sizeof(orbx_keypoint) * (size_t)rows_out, nf, cudaMemcpyDeviceToHost, ost));
            CU(cudaMemcpy2DAsync(descriptors + (size_t)f0 * capacity * 32, (size_t)capacity * 32, s.d_desc, (size_t)capacity * 32,
                                 (size_t)rows_out * 32, nf, cudaMemcpyDeviceToHost, ost));
        }
        mark(ost, c, 3);
        if (serial) CU(cudaEventRecord(s.ev_out, ost));
        return ORBX_OK;
    };
    const int lag = 2;
    for (int c = 0; c < nchunks; ++c) {
        Slot& s = ex->slots[c % nslots];
        const int f0 = sched[c].first, nf = sched[c].second;
        cudaStream_t cst = serial ? ex->compute : s.stream;
        cudaStream_t ist = serial ? ex->copy_in : s.stream, ost = serial ? ex->copy_out : s.stream;
        // reuse of a slot: its input staging is free once the chunk that used it has been computed, its output staging once
        // that chunk's D2H has completed (one slot stream orders all of this by itself in the other pipeline).  The D2H of
        // chunk c - nslots was queued when chunk c - nslots + lag was (nslots > lag whenever a slot is reused).
        if (serial && c >= nslots) { CU(cudaStreamWaitEvent(ist, s.ev_done, 0)); CU(cudaStreamWaitEvent(cst, s.ev_out, 0)); }
        mark(ist, c, 0);
        bool contiguous = step == (size_t)cols;
        for (int f = 1; f < nf && contiguous; ++f) contiguous = images[f0 + f] == images[f0 + f - 1] + dframe;
        if (contiguous) {
            CU(cudaMemcpyAsync(s.d_in, images[f0], dframe * nf, cudaMemcpyHostToDevice, ist));
        } else {
            for (int f = 0; f < nf; ++f)
                CU(cudaMemcpy2DAsync(s.d_in + (size_t)f * dframe, dpitch, images[f0 + f], step, cols, rows, cudaMemcpyHostToDevice, ist));
        }
        mark(ist, c, 1);
        if (serial) { CU(cudaEventRecord(s.ev_in, ist)); CU(cudaStreamWaitEvent(cst, s.ev_in, 0)); }
        if ((rc = run_chunk(ex, s, one_set_io(s.d_in, dframe, dpitch, s.d_kps, s.d_desc, capacity, s.d_n, s.d_nm), nf, lap0, lap1, cst))) return rc;
        if (serial) { CU(cudaEventRecord(s.ev_done, cst)); CU(cudaStreamWaitEvent(ost, s.ev_done, 0)); }
        mark(ost, c, 2);
        CU(cudaMemcpyAsync(n_out + f0, s.d_n, sizeof(int) * nf, cudaMemcpyDeviceToHost, ost));
        CU(cudaMemcpyAsync(n_mono + f0, s.d_nm, sizeof(int) * nf, cudaMemcpyDeviceToHost, ost));
        CU(cudaEventRecord(s.ev_cnt, ost));
        if (c % nslots == 0) ex->last_frames = nf;
        if (c >= lag && (rc = finish(c - lag))) return rc;
    }
    for (int c = std::max(nchunks - lag, 0); c < nchunks; ++c)
        if ((rc = finish(c))) return rc;
    if (serial) { CU(cudaStreamSynchronize(ex->copy_out)); CU(cudaStreamSynchronize(ex->compute)); CU(cudaStreamSynchronize(ex->copy_in)); }
    for (int i = 0; i < nslots; ++i) CU(cudaStreamSynchronize(ex->slots[i].stream));
    if (trace) {
        for (int c = 0; c < nchunks; ++c) {
            float t[4];
            for (int k = 0; k < 4; ++k) cudaEventElapsedTime(&t[k], tev[0], tev[4 * c + k]);      // (all four marks of every chunk exist)
            fprintf(stderr, "[orbx] chunk %2d frames %3d: h2d %.3f-%.3f compute-end %.3f d2h-end %.3f ms\n", c, sched[c].second, t[0], t[1], t[2], t[3]);
        }
        for (cudaEvent_t e : tev) if (e) cudaEventDestroy(e);
    }
    for (int f = 0; f < n_frames; ++f)
        if (n_out[f] > capacity) return fail(ORBX_ERR_CAPACITY, "frame %d has %d keypoints, capacity %d", f, n_out[f], capacity);
    return ORBX_OK;
}

int orbx_extract(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int lap0, int lap1,
                 orbx_keypoint* keypoints, uint8_t* descriptors, int capacity, int* n_out, int* n_mono)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    if (!image || rows <= 0 || cols <= 0) return fail(ORBX_ERR_EMPTY_IMAGE, "empty image");
    if (!keypoints || !descriptors || !n_out || !n_mono || capacity <= 0 || step < (size_t)cols)
        return fail(ORBX_ERR_INVALID_ARG, "bad output buffers / step");
    int rc = enqueue_single(ex, image, rows, cols, step, lap0, lap1, capacity);
    if (rc) return rc;
    Slot& s = ex->slots[0];
    CU(cudaMemcpyAsync(keypoints, s.d_kps, sizeof(orbx_keypoint) * (size_t)capacity, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(descriptors, s.d_desc, (size_t)capacity * 32, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(n_out, s.d_n, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(n_mono, s.d_nm, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    if (*n_out > capacity) return fail(ORBX_ERR_CAPACITY, "frame has %d keypoints, capacity %d", *n_out, capacity);
    return ORBX_OK;
}

int orbx_set_pyramid_mirror(orbx_extractor* ex, int enable)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    ex->mirror = enable != 0;
    return ORBX_OK;
}

int orbx_get_pyramid_mirror(orbx_extractor* ex, int level, const uint8_t** bordered, size_t* step, int* level_cols, int* level_rows)
{
    if (!ex || !ex->geom_valid || !ex->mirror || !ex->h_mirror || !ex->mirror_valid)
        return fail(ORBX_ERR_INVALID_ARG, "no mirrored pyramid: enable orbx_set_pyramid_mirror before a single-frame orbx_extract");
    if (level < 0 || level >= ex->nlevels) return fail(ORBX_ERR_INVALID_ARG, "level out of range");
    const LevelGeom& g = ex->fg.L[level];
    if (bordered) *bordered = ex->h_mirror + ex->mirror_off[level];
    if (step) *step = (size_t)g.w + 2 * kEdge;
    if (level_cols) *level_cols = g.w;
    if (level_rows) *level_rows = g.h;
    return ORBX_OK;
}

int orbx_cvt_gray_device(int device, const uint8_t* d_src, size_t src_pitch, size_t src_frame_stride, int channels, int rgb,
                         int n_frames, int rows, int cols, uint8_t* d_dst, size_t dst_pitch, size_t dst_frame_stride, void* stream)
{
    if (!d_src || !d_dst || n_frames <= 0 || rows <= 0 || cols <= 0 || (channels != 3 && channels != 4) ||
        src_pitch < (size_t)cols * channels || dst_pitch < (size_t)cols)
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc = set_device(device);
    if (rc) return rc;
    CU(launch_cvt_gray(d_src, src_pitch, src_frame_stride, channels, rgb, n_frames, rows, cols, d_dst, dst_pitch, dst_frame_stride,
                       (cudaStream_t)stream));
    return ORBX_OK;
}

int orbx_extract_color(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int channels, int rgb, int lap0,
                       int lap1, orbx_keypoint* keypoints, uint8_t* descriptors, int capacity, int* n_out, int* n_mono)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    if (!image || rows <= 0 || cols <= 0) return fail(ORBX_ERR_EMPTY_IMAGE, "empty image");
    if (channels == 1) return orbx_extract(ex, image, rows, cols, step, lap0, lap1, keypoints, descriptors, capacity, n_out, n_mono);
    if ((channels != 3 && channels != 4) || step < (size_t)cols * channels) return fail(ORBX_ERR_INVALID_ARG, "channels must be 1, 3 or 4");
    if (!keypoints || !descriptors || !n_out || !n_mono || capacity <= 0) return fail(ORBX_ERR_INVALID_ARG, "bad output buffers");
    int rc = set_device(ex->device);
    if (rc) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    wait_user_work(ex);
    if ((rc = ensure_capacity(ex, 1, 1))) return rc;
    Slot& s = ex->slots[0];
    const size_t gpitch = (size_t)cols, cpitch = align_up((size_t)cols * channels, 16);
    if ((rc = ensure_host_staging(s, gpitch * rows, 1, capacity))) return rc;
    if (s.d_color_bytes < cpitch * rows) {
        if ((rc = dev_alloc(s, &s.d_color, cpitch * rows))) return rc;
        s.d_color_bytes = cpitch * rows;
    }
    CU(cudaMemcpy2DAsync(s.d_color, cpitch, image, step, (size_t)cols * channels, rows, cudaMemcpyHostToDevice, s.stream));
    CU(launch_cvt_gray(s.d_color, cpitch, 0, channels, rgb, 1, rows, cols, s.d_in, gpitch, 0, s.stream));
    // same per-level fork / join as orbx_extract (launched eagerly: the colour staging buffer is not part of the captured graph)
    if ((rc = ensure_mirror(ex, s.stream))) return rc;
    if (ex->profiling) rc = run_chunk(ex, s, one_set_io(s.d_in, gpitch * rows, gpitch, s.d_kps, s.d_desc, capacity, s.d_n, s.d_nm), 1, lap0, lap1, s.stream);
    else rc = run_single_forked(ex, s, s.d_in, gpitch, lap0, lap1, s.d_kps, s.d_desc, capacity, s.d_n, s.d_nm, s.stream);
    if (rc) return rc;
    CU(cudaMemcpyAsync(keypoints, s.d_kps, sizeof(orbx_keypoint) * (size_t)capacity, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(descriptors, s.d_desc, (size_t)capacity * 32, cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(n_out, s.d_n, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CU(cudaMemcpyAsync(n_mono, s.d_nm, sizeof(int), cudaMemcpyDeviceToHost, s.stream));
    CU(cudaStreamSynchronize(s.stream));
    ex->last_frames = 1;
    if (*n_out > capacity) return fail(ORBX_ERR_CAPACITY, "%d keypoints, capacity %d", *n_out, capacity);
    return ORBX_OK;
}

// ---- per-stage timing with CUDA events on the launching stream ---------------------------------------------------------
int orbx_profile_begin(orbx_extractor* ex)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    ex->profiling = true;
    ex->ev_used = 0;
    return ORBX_OK;
}

int orbx_profile_end(orbx_extractor* ex, float* stage_ms, int* n_chunks)
{
    if (!ex || !stage_ms) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    ex->profiling = false;
    for (int k = 0; k < kStages; ++k) stage_ms[k] = 0.f;
    const size_t per = kStages + 1, chunks = ex->ev_used / per;
    if (chunks > 0) CU(cudaEventSynchronize(ex->ev_pool[ex->ev_used - 1]));
    for (size_t c = 0; c < chunks; ++c)
        for (int k = 0; k < kStages; ++k) {
            float ms = 0.f;
            CU(cudaEventElapsedTime(&ms, ex->ev_pool[c * per + k], ex->ev_pool[c * per + k + 1]));
            stage_ms[k] += ms;
        }
    if (n_chunks) *n_chunks = (int)chunks;
    ex->ev_used = 0;
    return ORBX_OK;
}

// ---- probes ---------------------------------------------------------------------------------------------------------
static int probe_check(orbx_extractor* ex, int frame, int level)
{
    if (!ex || !ex->geom_valid) return fail(ORBX_ERR_INVALID_ARG, "no extraction has run on this handle");
    if (level < 0 || level >= ex->nlevels || frame < 0 || frame >= ex->last_frames)
        return fail(ORBX_ERR_INVALID_ARG, "frame/level out of range (the last call processed %d frame(s))", ex->last_frames);
    int rc = set_device(ex->device);
    if (rc) return rc;
    return orbx_sync(ex);
}

int orbx_get_pyramid_level(orbx_extractor* ex, int frame, int level, uint8_t* dst, size_t dst_step, int with_border)
{
    int rc = probe_check(ex, frame, level);
    if (rc) return rc;
    const LevelGeom& g = ex->fg.L[level];
    const uint8_t* base = ex->slots[0].ws.pyr + g.pyr_off + (size_t)frame * g.pyr_frame_stride;
    if (with_border)
        CU(cudaMemcpy2D(dst, dst_step, base + (kXPad - kEdge), g.pitch, g.w + 2 * kEdge, g.h + 2 * kEdge, cudaMemcpyDeviceToHost));
    else
        CU(cudaMemcpy2D(dst, dst_step, base + (size_t)kEdge * g.pitch + kXPad, g.pitch, g.w, g.h, cudaMemcpyDeviceToHost));
    return ORBX_OK;
}

int orbx_get_blurred_level(orbx_extractor* ex, int frame, int level, uint8_t* dst, size_t dst_step)
{
    int rc = probe_check(ex, frame, level);
    if (rc) return rc;
    const LevelGeom& g = ex->fg.L[level];
    CU(cudaMemcpy2D(dst, dst_step, ex->slots[0].ws.blur + g.blur_off + (size_t)frame * g.blur_frame_stride, g.bpitch, g.w, g.h,
                    cudaMemcpyDeviceToHost));
    return ORBX_OK;
}

int orbx_get_candidates(orbx_extractor* ex, int frame, int level, int* xs, int* ys, int* scores, int capacity)
{
    int rc = probe_check(ex, frame, level);
    if (rc) return rc;
    const FrameGeom& fg = ex->fg;
    const LevelGeom& g = fg.L[level];
    const int ncells = g.nCols * g.nRows;
    if (ncells == 0) return 0;
    std::vector<int> counts(ncells);
    CU(cudaMemcpy(counts.data(), ex->slots[0].ws.cell_count + (size_t)frame * fg.total_cells + g.cell_base, sizeof(int) * ncells,
                  cudaMemcpyDeviceToHost));
    std::vector<uint32_t> cand((size_t)g.cand_max);
    CU(cudaMemcpy(cand.data(), ex->slots[0].ws.cand + (size_t)frame * fg.cand_frame_stride + g.cand_off, sizeof(uint32_t) * cand.size(),
                  cudaMemcpyDeviceToHost));
    int n = 0;
    for (int c = 0; c < ncells; ++c)
        for (int i = 0; i < counts[c]; ++i, ++n)
            if (n < capacity) {
                const uint32_t k = cand[(size_t)c * g.cell_cap + i];
                xs[n] = (int)(k & 0xfff); ys[n] = (int)((k >> 12) & 0xfff); scores[n] = (int)(k >> 24);
            }
    return n;
}

int orbx_get_level_keypoints(orbx_extractor* ex, int frame, int level, orbx_keypoint* keypoints, uint8_t* descriptors, int capacity)
{
    int rc = probe_check(ex, frame, level);
    if (rc) return rc;
    const FrameGeom& fg = ex->fg;
    const LevelGeom& g = fg.L[level];
    const Workspace& ws = ex->slots[0].ws;
    int n = 0;
    CU(cudaMemcpy(&n, ws.lvl_n + (size_t)frame * fg.nlevels + level, sizeof(int), cudaMemcpyDeviceToHost));
    if (n <= 0) return 0;
    std::vector<uint32_t> keys(n);
    std::vector<float> ang(n);
    CU(cudaMemcpy(keys.data(), ws.lvl_kp + (size_t)frame * fg.kp_slots + g.kp_base, sizeof(uint32_t) * n, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(ang.data(), ws.lvl_angle + (size_t)frame * fg.kp_slots + g.kp_base, sizeof(float) * n, cudaMemcpyDeviceToHost));
    const int m = std::min(n, capacity);
    if (descriptors)
        CU(cudaMemcpy(descriptors, ws.lvl_desc + ((size_t)frame * fg.kp_slots + g.kp_base) * 32, (size_t)m * 32, cudaMemcpyDeviceToHost));
    for (int i = 0; i < m; ++i) {
        orbx_keypoint& k = keypoints[i];
        k.x = (float)((int)(keys[i] & 0xfff) + kWinBorder);
        k.y = (float)((int)((keys[i] >> 12) & 0xfff) + kWinBorder);
        k.size = g.kp_size; k.angle = ang[i]; k.response = (float)(keys[i] >> 24); k.octave = level; k.class_id = -1;
    }
    return n;
}

// ---- stand-alone octree (parity tests drive the kernel with hand-built candidate sets) --------------------------------
int orbx_distribute_octree(int device, const int* xs, const int* ys, const int* scores, int n, int minX, int maxX, int minY,
                           int maxY, int nFeatures, int* out_idx, int capacity, int* n_out)
{
    if (!n_out || n < 0 || (n > 0 && (!xs || !ys || !scores))) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc = set_device(device);
    if (rc) return rc;
    *n_out = 0;
    const int width = maxX - minX, height = maxY - minY;
    if (width <= 0 || height <= 0 || width > 4095 || height > 4095) return fail(ORBX_ERR_UNSUPPORTED, "window %dx%d", width, height);
    // Build a one-level geometry whose single "cell" holds all candidates in the given order.
    FrameGeom fg;
    memset(&fg, 0, sizeof fg);
    fg.nlevels = 1; fg.total_cells = 1;
    LevelGeom& g = fg.L[0];
    g.w = width + 2 * kWinBorder; g.h = height + 2 * kWinBorder;
    g.nCols = 1; g.nRows = 1; g.wCell = 1; g.hCell = 1; g.cell_base = 0; g.cell_cap = std::max(n, 1); g.cand_off = 0; g.cand_max = std::max(n, 1);
    g.oct_off = 0; g.nfeat = nFeatures;
    g.nIni = (int)round((float)width / (float)height);
    if (g.nIni > 64) return fail(ORBX_ERR_UNSUPPORTED, "aspect ratio");
    g.hX = g.nIni > 0 ? (float)width / g.nIni : 1.f;
    {
        int maxRootW = 1;
        for (int i = 0; i < g.nIni; ++i) maxRootW = std::max(maxRootW, (int)(g.hX * (float)(i + 1)) - (int)(g.hX * (float)i));
        auto clog2 = [](int v) { int b = 0; while ((1 << b) < v) ++b; return b; };
        g.depth = std::max(clog2(maxRootW) + 1, clog2(std::max(height, 1))) + 1;
        g.root_bits = clog2(std::max(g.nIni, 1));
        if (2 * g.depth + g.root_bits > 32) return fail(ORBX_ERR_UNSUPPORTED, "path code too long");
    }
    g.kp_base = 0; g.kp_cap = std::max(nFeatures + 4, 4 * g.nIni + 1);
    fg.kp_slots = g.kp_cap; fg.cand_frame_stride = g.cand_max; fg.oct_frame_stride = 5ull * g.cand_max + 32;
    if (g.cand_max >= (1 << 24)) return fail(ORBX_ERR_UNSUPPORTED, "too many candidates");
    if (octree_smem_for(fg, 0, 1) > 200 * 1024) return fail(ORBX_ERR_UNSUPPORTED, "nFeatures too large");
    CU(octree_prepare());
    std::vector<uint32_t> packed(std::max(n, 1));
    for (int i = 0; i < n; ++i) {
        if (xs[i] < 0 || xs[i] > 4095 || ys[i] < 0 || ys[i] > 4095 || scores[i] < 0 || scores[i] > 255)
            return fail(ORBX_ERR_INVALID_ARG, "candidate %d out of range", i);
        packed[i] = (uint32_t)xs[i] | ((uint32_t)ys[i] << 12) | ((uint32_t)scores[i] << 24);
    }
    {   // the quadtree separates distinct pixels only; the reference would loop on two candidates at one pixel until its
        // depth runs out, cv::FAST never produces them
        std::vector<uint32_t> seen(packed.begin(), packed.begin() + n);
        for (auto& v : seen) v &= 0xffffffu;
        std::sort(seen.begin(), seen.end());
        if (std::adjacent_find(seen.begin(), seen.end()) != seen.end()) return fail(ORBX_ERR_INVALID_ARG, "two candidates share a pixel");
    }
    Slot s;
    Workspace& ws = s.ws;
    int one = n;
    auto cleanup = [&] { free_slot(s); };
    if ((rc = dev_alloc(s, &ws.cand, packed.size())) || (rc = dev_alloc(s, &ws.cell_count, 1)) ||
        (rc = dev_alloc(s, &ws.oct, (size_t)fg.oct_frame_stride)) || (rc = dev_alloc(s, &ws.lvl_kp, (size_t)fg.kp_slots)) ||
        (rc = dev_alloc(s, &ws.lvl_n, 1)) || (rc = dev_alloc(s, &ws.lvl_ncand, 1))) { cleanup(); return rc; }
    cudaMemcpy(ws.cand, packed.data(), sizeof(uint32_t) * packed.size(), cudaMemcpyHostToDevice);
    cudaMemcpy(ws.cell_count, &one, sizeof(int), cudaMemcpyHostToDevice);
    cudaError_t e = launch_octree(fg, ws, 1, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { cleanup(); return fail(ORBX_ERR_CUDA, "octree kernel: %s", cudaGetErrorString(e)); }
    if (octree_take_error_flag()) { cleanup(); return fail(ORBX_ERR_INVALID_ARG, "quadtree depth exhausted (candidates not separable)"); }
    int m = 0;
    cudaMemcpy(&m, ws.lvl_n, sizeof(int), cudaMemcpyDeviceToHost);
    std::vector<uint32_t> keys(std::max(m, 1));
    cudaMemcpy(keys.data(), ws.lvl_kp, sizeof(uint32_t) * m, cudaMemcpyDeviceToHost);
    cleanup();
    *n_out = m;
    if (m > capacity) return fail(ORBX_ERR_CAPACITY, "need %d slots", m);
    // map retained keys back to input indices (pixel positions are unique)
    std::unordered_map<uint32_t, int> lut;
    lut.reserve((size_t)n * 2);
    for (int i = 0; i < n; ++i) lut[(uint32_t)ys[i] * 4096u + (uint32_t)xs[i]] = i;
    for (int i = 0; i < m; ++i) out_idx[i] = lut[((keys[i] >> 12) & 0xfff) * 4096u + (keys[i] & 0xfff)];
    return ORBX_OK;
}

// ---- matching ---------------------------------------------------------------------------------------------------------
int orbx_descriptor_distance(const uint8_t* a, const uint8_t* b)
{
    uint64_t x[4], y[4];
    memcpy(x, a, 32); memcpy(y, b, 32);
    return __builtin_popcountll(x[0] ^ y[0]) + __builtin_popcountll(x[1] ^ y[1]) + __builtin_popcountll(x[2] ^ y[2]) +
           __builtin_popcountll(x[3] ^ y[3]);
}

int orbx_knn2_device(int device, const uint8_t* d_queries, int nq, const uint8_t* d_database, int64_t ndb, int32_t index_base,
                     int32_t* d_idx, int32_t* d_dist, void* stream)
{
    if (nq < 0 || ndb < 0 || (nq > 0 && (!d_queries || !d_idx || !d_dist)) || (ndb > 0 && !d_database))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (ndb + (int64_t)index_base > 0x7fffffffLL) return fail(ORBX_ERR_UNSUPPORTED, "database rows must fit int32");
    int rc = set_device(device);
    if (rc) return rc;
    CU(launch_knn2(d_queries, nq, d_database, ndb, index_base, d_idx, d_dist, (cudaStream_t)stream));
    return ORBX_OK;
}

int orbx_knn2_merge_device(int device, const int32_t* d_idx_shards, const int32_t* d_dist_shards, int n_shards, int nq,
                           int32_t* d_idx, int32_t* d_dist, void* stream)
{
    if (n_shards <= 0 || nq < 0) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc = set_device(device);
    if (rc) return rc;
    CU(launch_knn2_merge(d_idx_shards, d_dist_shards, n_shards, nq, d_idx, d_dist, (cudaStream_t)stream));
    return ORBX_OK;
}

int orbx_knn2(int device, const uint8_t* queries, int nq, const uint8_t* database, int64_t ndb, int32_t* idx, int32_t* dist)
{
    if (nq < 0 || ndb < 0 || (nq > 0 && (!queries || !idx || !dist)) || (ndb > 0 && !database))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (nq == 0) return ORBX_OK;
    int rc = set_device(device);
    if (rc) return rc;
    ScratchLease L(device);
    const size_t ws_bytes = knn2_workspace_bytes(nq, ndb);
    if ((rc = L.reserve((size_t)nq * 32 + (size_t)std::max<int64_t>(ndb, 1) * 32 + (size_t)nq * 16 + ws_bytes + 5 * 256))) return rc;
    uint8_t* dq = L.take<uint8_t>((size_t)nq * 32);
    uint8_t* ddb = L.take<uint8_t>((size_t)std::max<int64_t>(ndb, 1) * 32);
    int32_t* di = L.take<int32_t>((size_t)nq * 2);
    int32_t* dd = L.take<int32_t>((size_t)nq * 2);
    void* dws = ws_bytes ? (void*)L.take<uint8_t>(ws_bytes) : nullptr;
    cudaError_t e = cudaMemcpy(dq, queries, (size_t)nq * 32, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && ndb > 0) e = cudaMemcpy(ddb, database, (size_t)ndb * 32, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = launch_knn2(dq, nq, ddb, ndb, 0, di, dd, 0, dws);
    if (e == cudaSuccess) e = cudaMemcpy(idx, di, (size_t)nq * 8, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaMemcpy(dist, dd, (size_t)nq * 8, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "knn2: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

int orbx_ratio_test(const int32_t* dist, int nq, float ratio, int th_low, int mode, uint8_t* accept)
{
    if (!dist || !accept || nq < 0) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    for (int i = 0; i < nq; ++i) {
        const int d1 = dist[2 * i], d2 = dist[2 * i + 1];
        bool ok;
        if (mode == 0) ok = d1 <= th_low && (float)d1 < ratio * (float)d2;          // src/ORBmatcher1.cc:329-333
        else if (mode == 1) ok = d1 < th_low && (float)d1 < ratio * (float)d2;      // src/ORBmatcher2.cc:120-125
        else ok = (float)d1 < (float)d2 * (double)ratio;                            // src/Frame.cc:1181
        accept[i] = ok ? 1 : 0;
    }
    return ORBX_OK;
}

int orbx_rotation_consistency(const float* angle_a, const float* angle_b, int n, uint8_t* keep)
{
    if (n < 0 || (n > 0 && (!angle_a || !angle_b || !keep))) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    const int HISTO_LENGTH = 30;
    std::vector<int> bin(n);
    int count[HISTO_LENGTH] = {0};
    for (int i = 0; i < n; ++i) {
        const int b = rotation_bin(angle_a[i], angle_b[i]);
        if (b < 0) return fail(ORBX_ERR_INVALID_ARG, "angle %d out of range (reference asserts)", i);
        bin[i] = b;
        count[b]++;
    }
    int ind1, ind2, ind3;
    three_maxima(count, HISTO_LENGTH, ind1, ind2, ind3);
    for (int i = 0; i < n; ++i) keep[i] = (bin[i] == ind1 || bin[i] == ind2 || bin[i] == ind3) ? 1 : 0;
    return ORBX_OK;
}

int orbx_distinctive_descriptor(const uint8_t* descriptors, int n, int* best_idx)
{
    if (n <= 0 || !descriptors || !best_idx) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    std::vector<int> dist((size_t)n * n, 0);
    for (int i = 0; i < n; ++i)
        for (int j = i + 1; j < n; ++j) {
            const int d = orbx_descriptor_distance(descriptors + (size_t)i * 32, descriptors + (size_t)j * 32);
            dist[(size_t)i * n + j] = d; dist[(size_t)j * n + i] = d;
        }
    int bestMedian = INT_MAX, bestIdx = 0;
    std::vector<int> row(n);
    for (int i = 0; i < n; ++i) {
        std::copy(dist.begin() + (size_t)i * n, dist.begin() + (size_t)(i + 1) * n, row.begin());
        std::sort(row.begin(), row.end());
        const int median = row[(size_t)(0.5 * (n - 1))];
        if (median < bestMedian) { bestMedian = median; bestIdx = i; }
    }
    *best_idx = bestIdx;
    return ORBX_OK;
}

// Checks shared by the stereo entry points; fills the pyramid part of the kernel arguments.
static int stereo_prepare(orbx_extractor* exL, int frameL, orbx_extractor* exR, int frameR, StereoArgs& A)
{
    if (!exL || !exR || !exL->geom_valid || !exR->geom_valid) return fail(ORBX_ERR_INVALID_ARG, "extractors have not run");
    if (exL->device != exR->device || exL->fg.rows != exR->fg.rows || exL->fg.cols != exR->fg.cols || exL->nlevels != exR->nlevels ||
        exL->scaleFactorF != exR->scaleFactorF)
        return fail(ORBX_ERR_INVALID_ARG, "left/right extractors must share device, image shape, levels and scale factor");
    if (frameL < 0 || frameL >= exL->last_frames || frameR < 0 || frameR >= exR->last_frames)
        return fail(ORBX_ERR_INVALID_ARG, "frame out of range");
    // Scale tables: the reference reads Frame::mvScaleFactors / mvInvScaleFactors — the LEFT extractor's — for both sides
    // (src/Frame.cc:112-118, 859, 933); the level sizes and pitches follow from the shape, which is shared.  What is NOT
    // shared is where each extractor put its level slabs (that depends on its own slot capacity).
    A.pyrL = exL->slots[0].ws.pyr; A.pyrR = exR->slots[0].ws.pyr; A.frameL = frameL; A.frameR = frameR; A.n_pairs = 1;
    for (int l = 0; l < exR->nlevels; ++l) A.offR[l] = exR->fg.L[l].pyr_off;
    return ORBX_OK;
}

int orbx_stereo_match(orbx_extractor* exL, int frameL, orbx_extractor* exR, int frameR, const orbx_keypoint* kpL,
                      const uint8_t* descL, int nL, const orbx_keypoint* kpR, const uint8_t* descR, int nR, float bf, float maxD,
                      float* uRight, float* depth)
{
    StereoArgs A{};
    int rc = stereo_prepare(exL, frameL, exR, frameR, A);
    if (rc) return rc;
    if (nL < 0 || nR < 0 || (nL > 0 && (!kpL || !descL || !uRight || !depth)) || (nR > 0 && (!kpR || !descR)))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (nR >= (1 << 20)) return fail(ORBX_ERR_UNSUPPORTED, "too many right keypoints");
    if (nL == 0) return ORBX_OK;
    if ((rc = set_device(exL->device))) return rc;
    if ((rc = orbx_sync(exL)) || (rc = orbx_sync(exR))) return rc;
    for (int i = 0; i < nL; ++i)
        if (kpL[i].octave < 0 || kpL[i].octave >= exL->nlevels) return fail(ORBX_ERR_INVALID_ARG, "left keypoint %d octave", i);
    for (int i = 0; i < nR; ++i)
        if (kpR[i].octave < 0 || kpR[i].octave >= exL->nlevels) return fail(ORBX_ERR_INVALID_ARG, "right keypoint %d octave", i);
    ScratchLease Ls(exL->device);
    const size_t nRa = (size_t)std::max(nR, 1);
    if ((rc = Ls.reserve(((size_t)nL + nRa) * (sizeof(orbx_keypoint) + 32) + (size_t)nL * 12 + 8 * 256))) return rc;
    orbx_keypoint* dkL = Ls.take<orbx_keypoint>((size_t)nL);
    uint8_t* ddL = Ls.take<uint8_t>((size_t)nL * 32);
    orbx_keypoint* dkR = Ls.take<orbx_keypoint>(nRa);
    uint8_t* ddR = Ls.take<uint8_t>(nRa * 32);
    A.uRight = Ls.take<float>((size_t)nL); A.depth = Ls.take<float>((size_t)nL); A.sad = Ls.take<int>((size_t)nL);
    cudaStream_t st = exL->slots[0].stream;          // idle: orbx_sync above
    cudaError_t e = cudaMemcpyAsync(dkL, kpL, sizeof(orbx_keypoint) * nL, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ddL, descL, (size_t)nL * 32, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && nR > 0) e = cudaMemcpyAsync(dkR, kpR, sizeof(orbx_keypoint) * nR, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess && nR > 0) e = cudaMemcpyAsync(ddR, descR, (size_t)nR * 32, cudaMemcpyHostToDevice, st);
    A.kpL = dkL; A.descL = ddL; A.nL = nL; A.kpR = dkR; A.descR = ddR; A.nR = nR; A.bf = bf; A.maxD = maxD;
    if (e == cudaSuccess) e = launch_stereo(exL->fg, A, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(uRight, A.uRight, sizeof(float) * nL, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(depth, A.depth, sizeof(float) * nL, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);          // the lease (scratch) is released on return
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "stereo: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

int orbx_stereo_match_device(orbx_extractor* exL, int frameL, orbx_extractor* exR, int frameR, const orbx_keypoint* d_kpL,
                             const uint8_t* d_descL, const int* d_nL, int capL, const orbx_keypoint* d_kpR, const uint8_t* d_descR,
                             const int* d_nR, int capR, float bf, float maxD, float* d_uRight, float* d_depth, void* stream)
{
    StereoArgs A{};
    int rc = stereo_prepare(exL, frameL, exR, frameR, A);
    if (rc) return rc;
    if (!d_kpL || !d_descL || !d_nL || !d_kpR || !d_descR || !d_nR || capL <= 0 || capR <= 0 || !d_uRight || !d_depth)
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (capR >= (1 << 20)) return fail(ORBX_ERR_UNSUPPORTED, "too many right keypoints");
    if ((rc = set_device(exL->device))) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    int* sad = nullptr;
    CU(cudaMallocAsync((void**)&sad, sizeof(int) * (size_t)capL, st));       // stream-ordered, private to the call
    A.kpL = d_kpL; A.descL = d_descL; A.nL = capL; A.d_nL = d_nL; A.kpR = d_kpR; A.descR = d_descR; A.nR = capR; A.d_nR = d_nR;
    A.bf = bf; A.maxD = maxD; A.uRight = d_uRight; A.depth = d_depth; A.sad = sad;
    cudaError_t e = launch_stereo(exL->fg, A, st);
    cudaError_t e2 = cudaFreeAsync(sad, st);
    if (e == cudaSuccess) e = e2;
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "stereo: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

// The stereo Frame constructor in one call (src/Frame.cc:124-143): both extractions run concurrently on their extractors'
// streams (as the reference's two std::threads do), ComputeStereoMatches follows on the device as soon as both are done —
// it reads the keypoints, descriptors and un-blurred pyramids where the extractors left them — and one wait at the end
// covers all copies back.  No intermediate host round trip, no second upload of the features.
int orbx_extract_stereo(orbx_extractor* exL, orbx_extractor* exR, const uint8_t* imageL, const uint8_t* imageR, int rows, int cols,
                        size_t step, orbx_keypoint* kpL, uint8_t* descL, int* nL, orbx_keypoint* kpR, uint8_t* descR, int* nR,
                        int capacity, float bf, float maxD, float* uRight, float* depth)
{
    if (!exL || !exR || exL == exR) return fail(ORBX_ERR_INVALID_ARG, "two distinct extractors are required");
    if (!imageL || !imageR || rows <= 0 || cols <= 0) return fail(ORBX_ERR_EMPTY_IMAGE, "empty image");
    if (!kpL || !descL || !nL || !kpR || !descR || !nR || !uRight || !depth || capacity <= 0 || step < (size_t)cols)
        return fail(ORBX_ERR_INVALID_ARG, "bad output buffers / step");
    if (exL->device != exR->device) return fail(ORBX_ERR_INVALID_ARG, "left/right extractors must share a device");
    // vLappingArea = {0, 0} for both cameras of a rectified pair (src/Frame.cc:124-125)
    int rc;
    if ((rc = enqueue_single(exL, imageL, rows, cols, step, 0, 0, capacity))) return rc;
    if ((rc = enqueue_single(exR, imageR, rows, cols, step, 0, 0, capacity))) return rc;
    Slot& sL = exL->slots[0];
    Slot& sR = exR->slots[0];
    // right side: its results go home on its own stream while the matcher runs
    CU(cudaEventRecord(sR.ev_done, sR.stream));
    CU(cudaMemcpyAsync(kpR, sR.d_kps, sizeof(orbx_keypoint) * (size_t)capacity, cudaMemcpyDeviceToHost, sR.stream));
    CU(cudaMemcpyAsync(descR, sR.d_desc, (size_t)capacity * 32, cudaMemcpyDeviceToHost, sR.stream));
    CU(cudaMemcpyAsync(nR, sR.d_n, sizeof(int), cudaMemcpyDeviceToHost, sR.stream));
    // left side: wait for the right extraction, match on the device, then copy everything back
    CU(cudaStreamWaitEvent(sL.stream, sR.ev_done, 0));
    ScratchLease Ls(exL->device);
    if ((rc = Ls.reserve((size_t)capacity * 12 + 4 * 256))) return rc;
    float* d_u = Ls.take<float>((size_t)capacity);
    float* d_d = Ls.take<float>((size_t)capacity);
    StereoArgs A{};
    if ((rc = stereo_prepare(exL, 0, exR, 0, A))) return rc;
    A.kpL = sL.d_kps; A.descL = sL.d_desc; A.nL = capacity; A.d_nL = sL.d_n;
    A.kpR = sR.d_kps; A.descR = sR.d_desc; A.nR = capacity; A.d_nR = sR.d_n;
    A.bf = bf; A.maxD = maxD; A.uRight = d_u; A.depth = d_d; A.sad = Ls.take<int>((size_t)capacity);
    if (capacity >= (1 << 20)) return fail(ORBX_ERR_UNSUPPORTED, "too many right keypoints");
    CU(launch_stereo(exL->fg, A, sL.stream));
    CU(cudaMemcpyAsync(kpL, sL.d_kps, sizeof(orbx_keypoint) * (size_t)capacity, cudaMemcpyDeviceToHost, sL.stream));
    CU(cudaMemcpyAsync(descL, sL.d_desc, (size_t)capacity * 32, cudaMemcpyDeviceToHost, sL.stream));
    CU(cudaMemcpyAsync(nL, sL.d_n, sizeof(int), cudaMemcpyDeviceToHost, sL.stream));
    CU(cudaMemcpyAsync(uRight, d_u, sizeof(float) * (size_t)capacity, cudaMemcpyDeviceToHost, sL.stream));
    CU(cudaMemcpyAsync(depth, d_d, sizeof(float) * (size_t)capacity, cudaMemcpyDeviceToHost, sL.stream));
    CU(cudaStreamSynchronize(sL.stream));
    CU(cudaStreamSynchronize(sR.stream));
    if (*nL > capacity || *nR > capacity) return fail(ORBX_ERR_CAPACITY, "%d / %d keypoints, capacity %d", *nL, *nR, capacity);
    return ORBX_OK;
}

// ---- stereo batches -----------------------------------------------------------------------------------------------------
// A chunk of P pairs is 2P frames of one slot: the pairs' left images, then their right images.  Both images of a pair are
// extracted in the same chunk and the pair is matched on the chunk's stream from that slot's pyramids, before the slot can be
// reused.  One handle serves both sides: results depend only on its parameters and the image, and the reference's matcher reads
// the left extractor's scale tables for both sides (src/Frame.cc:112-118).

static int stereo_batch_args(orbx_extractor* ex, int n_pairs, int rows, int cols, bool images_ok, bool outputs_ok, size_t step,
                             int capacity)
{
    if (!ex) return fail(ORBX_ERR_INVALID_ARG, "extractor is NULL");
    if (n_pairs < 0) return fail(ORBX_ERR_INVALID_ARG, "n_pairs %d < 0", n_pairs);
    if (n_pairs == 0) return ORBX_OK;
    if (!images_ok || rows <= 0 || cols <= 0) return fail(ORBX_ERR_EMPTY_IMAGE, "empty image");
    if (!outputs_ok || capacity <= 0 || step < (size_t)cols) return fail(ORBX_ERR_INVALID_ARG, "bad output buffers / step");
    if (capacity >= (1 << 20)) return fail(ORBX_ERR_UNSUPPORTED, "capacity %d: the stereo kernels index at most 2^20 - 1 rows", capacity);
    return ORBX_OK;
}

// Matcher arguments of pairs [p, p + np) whose 2 np frames the slot's pyramid holds (left frames 0.., right frames np..)
static StereoArgs stereo_chunk_args(const orbx_extractor* ex, const Slot& s, int np, const orbx_keypoint* kpL, const uint8_t* descL,
                                    const int* d_nL, const orbx_keypoint* kpR, const uint8_t* descR, const int* d_nR, int capacity,
                                    float bf, float maxD, float* uRight, float* depth)
{
    StereoArgs A{};
    A.pyrL = A.pyrR = s.ws.pyr;
    for (int l = 0; l < ex->nlevels; ++l) A.offR[l] = ex->fg.L[l].pyr_off;
    A.frameL = 0; A.frameR = np; A.n_pairs = np;
    A.kpL = kpL; A.descL = descL; A.nL = capacity; A.d_nL = d_nL;
    A.kpR = kpR; A.descR = descR; A.nR = capacity; A.d_nR = d_nR;
    A.bf = bf; A.maxD = maxD; A.uRight = uRight; A.depth = depth; A.sad = s.d_sad;
    return A;
}

int orbx_extract_stereo_batch(orbx_extractor* ex, const uint8_t* const* imagesL, const uint8_t* const* imagesR, int n_pairs, int rows,
                              int cols, size_t step, float bf, float maxD, orbx_keypoint* kpL, uint8_t* descL, int* nL,
                              orbx_keypoint* kpR, uint8_t* descR, int* nR, int capacity, float* uRight, float* depth)
{
    bool images_ok = imagesL && imagesR;
    for (int i = 0; images_ok && i < n_pairs; ++i) images_ok = imagesL[i] && imagesR[i];
    int rc = stereo_batch_args(ex, n_pairs, rows, cols, images_ok, kpL && descL && nL && kpR && descR && nR && uRight && depth, step,
                               capacity);
    if (rc || n_pairs == 0) return rc;
    if ((rc = set_device(ex->device))) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    wait_user_work(ex);
    ex->last_frames = 0;
    // orbx_extract_batch's chunking and ramp schedule, in whole pairs
    const int chunk_frames = ex->max_batch > 0 ? std::min(ex->max_batch, 2 * n_pairs) : std::min(2 * n_pairs, 64);
    const int chunk = std::max(chunk_frames / 2, 1);
    const std::vector<std::pair<int, int>> sched = chunk_schedule(n_pairs, chunk);   // (first pair, pairs)
    const int nchunks = (int)sched.size();
    const int nslots = std::min(nchunks, (int)orbx_extractor::kSlots);
    if ((rc = ensure_capacity(ex, 2 * chunk, nslots))) return rc;
    const size_t dpitch = (size_t)cols, dframe = dpitch * rows;
    for (int i = 0; i < nslots; ++i) {
        Slot& s = ex->slots[i];
        if (s.d_in_bytes < dframe * 2 * chunk || s.out_cap < (size_t)2 * chunk * capacity || s.out_frames < 2 * chunk ||
            !stereo_staging_fits(s, chunk, capacity))
            CU(cudaStreamSynchronize(s.stream));
        if ((rc = ensure_host_staging(s, dframe * 2 * chunk, 2 * chunk, capacity))) return rc;
        if ((rc = ensure_stereo_staging(s, chunk, capacity))) return rc;
    }
    // the two pipelines of orbx_extract_batch (there: why), chosen by the chunk's frame count
    const bool serial = 2 * chunk >= 128;
    if (serial && !ex->compute) {
        CU(cudaStreamCreateWithFlags(&ex->compute, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&ex->copy_in, cudaStreamNonBlocking));
        CU(cudaStreamCreateWithFlags(&ex->copy_out, cudaStreamNonBlocking));
    }
    if (serial)
        for (int i = 0; i < nslots; ++i) CU(cudaStreamSynchronize(ex->slots[i].stream));
    // trimmed downloads as in orbx_extract_batch: counts first, then the rows the chunk's pairs have
    auto finish = [&](int c) -> int {
        Slot& s = ex->slots[c % nslots];
        const int p0 = sched[c].first, np = sched[c].second;
        cudaStream_t ost = serial ? ex->copy_out : s.stream;
        CU(cudaEventSynchronize(s.ev_cnt));
        int mxL = 0, mxR = 0;
        for (int p = 0; p < np; ++p) { mxL = std::max(mxL, nL[p0 + p]); mxR = std::max(mxR, nR[p0 + p]); }
        const size_t kpitch = sizeof(orbx_keypoint) * (size_t)capacity, dpitch32 = (size_t)capacity * 32, fpitch = sizeof(float) * (size_t)capacity;
        const int rowsL = std::min(mxL, capacity), rowsR = std::min(mxR, capacity);   // a pair over capacity fails the call below
        if (rowsL > 0) {
            CU(cudaMemcpy2DAsync(kpL + (size_t)p0 * capacity, kpitch, s.d_kps, kpitch, sizeof(orbx_keypoint) * (size_t)rowsL, np, cudaMemcpyDeviceToHost, ost));
            CU(cudaMemcpy2DAsync(descL + (size_t)p0 * capacity * 32, dpitch32, s.d_desc, dpitch32, (size_t)rowsL * 32, np, cudaMemcpyDeviceToHost, ost));
            CU(cudaMemcpy2DAsync(uRight + (size_t)p0 * capacity, fpitch, s.d_su, fpitch, sizeof(float) * (size_t)rowsL, np, cudaMemcpyDeviceToHost, ost));
            CU(cudaMemcpy2DAsync(depth + (size_t)p0 * capacity, fpitch, s.d_sd, fpitch, sizeof(float) * (size_t)rowsL, np, cudaMemcpyDeviceToHost, ost));
        }
        if (rowsR > 0) {
            CU(cudaMemcpy2DAsync(kpR + (size_t)p0 * capacity, kpitch, s.d_kps + (size_t)np * capacity, kpitch, sizeof(orbx_keypoint) * (size_t)rowsR, np,
                                 cudaMemcpyDeviceToHost, ost));
            CU(cudaMemcpy2DAsync(descR + (size_t)p0 * capacity * 32, dpitch32, s.d_desc + (size_t)np * capacity * 32, dpitch32, (size_t)rowsR * 32, np,
                                 cudaMemcpyDeviceToHost, ost));
        }
        if (serial) CU(cudaEventRecord(s.ev_out, ost));
        return ORBX_OK;
    };
    auto upload = [&](const uint8_t* const* images, int p0, int np, uint8_t* dst, cudaStream_t ist) -> int {
        bool contiguous = step == (size_t)cols;
        for (int p = 1; p < np && contiguous; ++p) contiguous = images[p0 + p] == images[p0 + p - 1] + dframe;
        if (contiguous) {
            CU(cudaMemcpyAsync(dst, images[p0], dframe * np, cudaMemcpyHostToDevice, ist));
        } else {
            for (int p = 0; p < np; ++p)
                CU(cudaMemcpy2DAsync(dst + (size_t)p * dframe, dpitch, images[p0 + p], step, cols, rows, cudaMemcpyHostToDevice, ist));
        }
        return ORBX_OK;
    };
    const int lag = 2;
    for (int c = 0; c < nchunks; ++c) {
        Slot& s = ex->slots[c % nslots];
        const int p0 = sched[c].first, np = sched[c].second;
        cudaStream_t cst = serial ? ex->compute : s.stream;
        cudaStream_t ist = serial ? ex->copy_in : s.stream, ost = serial ? ex->copy_out : s.stream;
        if (serial && c >= nslots) { CU(cudaStreamWaitEvent(ist, s.ev_done, 0)); CU(cudaStreamWaitEvent(cst, s.ev_out, 0)); }
        if ((rc = upload(imagesL, p0, np, s.d_in, ist)) || (rc = upload(imagesR, p0, np, s.d_in + (size_t)np * dframe, ist))) return rc;
        if (serial) { CU(cudaEventRecord(s.ev_in, ist)); CU(cudaStreamWaitEvent(cst, s.ev_in, 0)); }
        // the staging holds both sides back to back: one set of 2 np frames (vLappingArea = {0, 0}, src/Frame.cc:124-125)
        if ((rc = run_chunk(ex, s, one_set_io(s.d_in, dframe, dpitch, s.d_kps, s.d_desc, capacity, s.d_n, s.d_nm), 2 * np, 0, 0, cst))) return rc;
        const size_t r = (size_t)np * capacity;
        const StereoArgs A = stereo_chunk_args(ex, s, np, s.d_kps, s.d_desc, s.d_n, s.d_kps + r, s.d_desc + r * 32, s.d_n + np, capacity, bf, maxD,
                                               s.d_su, s.d_sd);
        CU(launch_stereo(ex->fg, A, cst));
        if (serial) { CU(cudaEventRecord(s.ev_done, cst)); CU(cudaStreamWaitEvent(ost, s.ev_done, 0)); }
        CU(cudaMemcpyAsync(nL + p0, s.d_n, sizeof(int) * np, cudaMemcpyDeviceToHost, ost));
        CU(cudaMemcpyAsync(nR + p0, s.d_n + np, sizeof(int) * np, cudaMemcpyDeviceToHost, ost));
        CU(cudaEventRecord(s.ev_cnt, ost));
        if (c >= lag && (rc = finish(c - lag))) return rc;
    }
    for (int c = std::max(nchunks - lag, 0); c < nchunks; ++c)
        if ((rc = finish(c))) return rc;
    if (serial) { CU(cudaStreamSynchronize(ex->copy_out)); CU(cudaStreamSynchronize(ex->compute)); CU(cudaStreamSynchronize(ex->copy_in)); }
    for (int i = 0; i < nslots; ++i) CU(cudaStreamSynchronize(ex->slots[i].stream));
    for (int p = 0; p < n_pairs; ++p)
        if (nL[p] > capacity || nR[p] > capacity)
            return fail(ORBX_ERR_CAPACITY, "pair %d has %d / %d keypoints, capacity %d", p, nL[p], nR[p], capacity);
    return ORBX_OK;
}

int orbx_extract_stereo_batch_device(orbx_extractor* ex, const uint8_t* d_imagesL, const uint8_t* d_imagesR, size_t frame_stride,
                                     int n_pairs, int rows, int cols, size_t pitch, float bf, float maxD, orbx_keypoint* d_kpL,
                                     uint8_t* d_descL, int* d_nL, orbx_keypoint* d_kpR, uint8_t* d_descR, int* d_nR, int capacity,
                                     float* d_uRight, float* d_depth, void* stream)
{
    int rc = stereo_batch_args(ex, n_pairs, rows, cols, d_imagesL && d_imagesR,
                               d_kpL && d_descL && d_nL && d_kpR && d_descR && d_nR && d_uRight && d_depth, pitch, capacity);
    if (rc || n_pairs == 0) return rc;
    if ((rc = set_device(ex->device))) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    ex->last_frames = 0;
    const int chunk_frames = ex->max_batch > 0 ? std::min(ex->max_batch, 2 * n_pairs) : std::min(2 * n_pairs, 256);
    const int chunk = std::max(chunk_frames / 2, 1);
    if ((rc = ensure_capacity(ex, 2 * chunk, 1))) return rc;
    Slot& s = ex->slots[0];
    if (!stereo_staging_fits(s, chunk, capacity)) {          // replaced below: earlier work on any stream must be done with it
        wait_user_work(ex);
        CU(cudaStreamSynchronize(s.stream));
        if ((rc = ensure_stereo_staging(s, chunk, capacity))) return rc;
    }
    cudaStream_t st = stream ? (cudaStream_t)stream : s.stream;
    if (!ex->ev_user) CU(cudaEventCreateWithFlags(&ex->ev_user, cudaEventDisableTiming));
    if (ex->user_pending) CU(cudaStreamWaitEvent(st, ex->ev_user, 0));
    if (st != s.stream) { CU(cudaEventRecord(s.ev_done, s.stream)); CU(cudaStreamWaitEvent(st, s.ev_done, 0)); }
    for (int p0 = 0; p0 < n_pairs; p0 += chunk) {
        const int np = std::min(chunk, n_pairs - p0);
        const size_t r = (size_t)p0 * capacity;
        // level 0 reads the left images from one base and the right images from the other; the results go straight to the
        // caller's slabs
        ChunkIO io{};
        io.img0 = d_imagesL + (size_t)p0 * frame_stride; io.img1 = d_imagesR + (size_t)p0 * frame_stride;
        io.frame_stride = frame_stride; io.pitch = pitch;
        io.kps0 = d_kpL + r; io.kps1 = d_kpR + r; io.desc0 = d_descL + r * 32; io.desc1 = d_descR + r * 32;
        io.n_out0 = d_nL + p0; io.n_out1 = d_nR + p0; io.n_mono0 = s.d_snm; io.n_mono1 = s.d_snm + np;
        io.capacity = capacity; io.split = np;
        if ((rc = run_chunk(ex, s, io, 2 * np, 0, 0, st))) return rc;
        const StereoArgs A = stereo_chunk_args(ex, s, np, d_kpL + r, d_descL + r * 32, d_nL + p0, d_kpR + r, d_descR + r * 32, d_nR + p0,
                                               capacity, bf, maxD, d_uRight + r, d_depth + r);
        CU(launch_stereo(ex->fg, A, st));
    }
    if (st != s.stream) { CU(cudaEventRecord(ex->ev_user, st)); ex->user_pending = true; }
    return ORBX_OK;
}

// ---- measurement ------------------------------------------------------------------------------------------------------
int orbx_measure_popc_peak(int device, double* popc_per_second)
{
    if (!popc_per_second) return fail(ORBX_ERR_INVALID_ARG, "NULL output");
    int rc = set_device(device);
    if (rc) return rc;
    unsigned long long* sink = nullptr;
    CU(cudaMalloc(&sink, 8));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device);
    const int blocks = sms * 8, iters = 4096;
    launch_popc_bench(sink, 256, blocks, 0);   // warm-up
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        cudaEventRecord(e0, 0);
        launch_popc_bench(sink, iters, blocks, 0);
        cudaEventRecord(e1, 0);
        cudaEventSynchronize(e1);
        float ms = 0;
        cudaEventElapsedTime(&ms, e0, e1);
        const double ops = (double)blocks * 256.0 * iters * 8.0;
        if (ms > 0) best = std::max(best, ops / (ms * 1e-3));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(sink);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "popc bench: %s", cudaGetErrorString(e));
    *popc_per_second = best;
    return ORBX_OK;
}

// ---- synthetic inputs -----------------------------------------------------------------------------------------------------
void orbx_synth_image_host(uint32_t seed, int view, int cols, int rows, int max_disp, uint8_t* dst, size_t step)
{
    for (int y = 0; y < rows; ++y)
        for (int x = 0; x < cols; ++x) dst[(size_t)y * step + x] = orbx_synth::image_pixel(seed, view, x, y, max_disp);
}

int orbx_synth_images_device(int device, uint32_t seed0, int view, int n_frames, int cols, int rows, int max_disp, uint8_t* d_dst,
                             size_t pitch, size_t frame_stride, void* stream)
{
    int rc = set_device(device);
    if (rc) return rc;
    if (!d_dst || cols <= 0 || rows <= 0 || n_frames <= 0 || max_disp < 2) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    CU(launch_synth_images(seed0, view, n_frames, cols, rows, max_disp, d_dst, pitch, frame_stride, (cudaStream_t)stream));
    return ORBX_OK;
}

void orbx_synth_descriptors_host(uint32_t seed, int is_query, int64_t first_row, int64_t n_rows, int64_t ndb, int plant_every, uint8_t* dst)
{
    uint32_t* w = reinterpret_cast<uint32_t*>(dst);
    for (int64_t r = 0; r < n_rows; ++r)
        for (uint32_t k = 0; k < 8; ++k)
            w[r * 8 + k] = is_query ? orbx_synth::query_word(seed, (uint32_t)(first_row + r), k, (uint32_t)ndb, (uint32_t)plant_every)
                                    : orbx_synth::desc_word(seed, (uint32_t)(first_row + r), k);
}

int orbx_synth_descriptors_device(int device, uint32_t seed, int is_query, int64_t first_row, int64_t n_rows, int64_t ndb,
                                  int plant_every, uint8_t* d_dst, void* stream)
{
    int rc = set_device(device);
    if (rc) return rc;
    CU(launch_synth_desc(seed, is_query, first_row, n_rows, ndb, plant_every, d_dst, (cudaStream_t)stream));
    return ORBX_OK;
}

// Debug: per-phase clock64 cycles of the octree CTA of (frame 0, `level`) during one single-frame extraction of `image`.
// out[0..6] = codes + bin counts + scan, bin scatter, roots, phase-1 sweeps, introsort replay, phase-2 rest, retain; out[7] = sweeps,
// out[8] = phase-2 rounds, out[9] = candidates, out[10] = largest sorted vector.
int orbx_debug_octree_timing(orbx_extractor* ex, const uint8_t* image, int rows, int cols, size_t step, int level, long long* out16)
{
    if (!ex || !image || !out16) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc = set_device(ex->device);
    if (rc) return rc;
    if ((rc = configure(ex, rows, cols))) return rc;
    if ((rc = ensure_capacity(ex, std::max(ex->max_batch, 1), 1))) return rc;
    Slot& s = ex->slots[0];
    long long* d_dbg = nullptr;
    CU(cudaMalloc(&d_dbg, 16 * sizeof(long long)));
    CU(cudaMemset(d_dbg, 0, 16 * sizeof(long long)));
    const int cap = ex->max_kp;
    std::vector<orbx_keypoint> kps(cap);
    std::vector<uint8_t> desc((size_t)cap * 32);
    int n = 0, nm = 0;
    s.ws.dbg = d_dbg; s.ws.dbg_level = level;
    ex->force_eager = true;
    // ORBX_DBG_REPLICAS=R (<= 64): time the CTA of frame 0 while R copies of the frame are in flight (phase times under load)
    const int reps = getenv("ORBX_DBG_REPLICAS") ? std::min(std::max(atoi(getenv("ORBX_DBG_REPLICAS")), 1), 64) : 1;
    if (reps > 1) {
        std::vector<const uint8_t*> imgs(reps, image);
        std::vector<orbx_keypoint> kb((size_t)cap * reps);
        std::vector<uint8_t> db((size_t)cap * 32 * reps);
        std::vector<int> nb(reps), nmb(reps);
        if ((rc = ensure_capacity(ex, reps, 1))) return rc;
        ex->slots[0].ws.dbg = d_dbg; ex->slots[0].ws.dbg_level = level;
        rc = orbx_extract_batch(ex, imgs.data(), reps, rows, cols, step, 0, 0, kb.data(), db.data(), cap, nb.data(), nmb.data());
    } else
    rc = orbx_extract(ex, image, rows, cols, step, 0, 0, kps.data(), desc.data(), cap, &n, &nm);
    ex->slots[0].ws.dbg = nullptr;
    ex->force_eager = false;
    if (!rc) cudaMemcpy(out16, d_dbg, 16 * sizeof(long long), cudaMemcpyDeviceToHost);
    cudaFree(d_dbg);
    return rc;
}

// Test hook: the std::sort replay used by the octree kernel, on the host (tests/test_introsort.py).
void orbx_debug_sort_replay(unsigned long long* items, int n) { orbx_sort::sort_replay(items, n); }
void orbx_debug_sort_replay32(uint32_t* items, int n) { orbx_sort::sort_replay(items, n); }
// host simulation of the range-parallel schedule the octree kernel runs (n < 4352: at most 256 ranges longer than 16)
void orbx_debug_sort_replay_ranges(unsigned long long* items, int n)
{
    if (n <= 0 || n >= 4352) { orbx_sort::sort_replay(items, n); return; }
    std::vector<uint32_t> blk(n);
    std::vector<unsigned long long> tmp(n);
    orbx_sort::sort_replay_ranges_host(items, n, blk.data(), tmp.data());
}
void orbx_debug_sort_replay_ranges32(uint32_t* items, int n)
{
    if (n <= 0 || n >= 4352) { orbx_sort::sort_replay(items, n); return; }
    std::vector<uint32_t> blk(n), tmp(n);
    orbx_sort::sort_replay_ranges_host(items, n, blk.data(), tmp.data());
}

// the same schedule with the rank-arithmetic partition the octree kernel evaluates per warp
void orbx_debug_sort_replay_ranked(unsigned long long* items, int n)
{
    if (n <= 0 || n >= 4352) { orbx_sort::sort_replay(items, n); return; }
    std::vector<uint32_t> blk(n);
    std::vector<unsigned long long> tmp(n);
    orbx_sort::sort_replay_ranges_host(items, n, blk.data(), tmp.data(), true);
}
void orbx_debug_sort_replay_ranked32(uint32_t* items, int n)
{
    if (n <= 0 || n >= 4352) { orbx_sort::sort_replay(items, n); return; }
    std::vector<uint32_t> blk(n), tmp(n);
    orbx_sort::sort_replay_ranges_host(items, n, blk.data(), tmp.data(), true);
}

}  // extern "C"
