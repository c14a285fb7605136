// api_io.cu — the last two Hamming users / data formats of SURVEY.md §8(f)4:
//
//  * the on-disk form of descriptors and key points in the Atlas files: what serializeMatrix / serializeVectorKeyPoints
//    (reference include/SerializationUtils.h:76-153) hand to a boost archive for KeyFrame::mDescriptors, MapPoint::mDescriptor,
//    KeyFrame::mvKeys / mvKeysUn / mvKeysRight (include/KeyFrame.h:120-128, 180; include/MapPoint.h:92), in the two archive kinds
//    System::SaveAtlas / LoadAtlas use (src/System.cc:1339-1475: boost text_oarchive and binary_oarchive).  Only the primitive
//    stream of these two helpers is produced / parsed here — the archive header and the class-tracking records around it belong
//    to boost.  Encoding of the primitives: binary archive = native little-endian bytes (int 4, bool 1, float 4, arrays raw);
//    text archive = every primitive preceded by one space, integers in decimal (unsigned char as a number), floats with 9
//    significant digits in scientific notation.  boost is not in this image, so this restates boost's documented primitive
//    encoding; the round trip and hand-built streams are what tests/test_io_cpu.py checks ("parity unpinned against boost").
//  * MapPoint::ComputeDistinctiveDescriptors (src/MapPoint.cc:329-401) for MANY map points per call on the GPU: one warp per
//    map point (N x N Hamming distances, per-row median at index (int)(0.5 * (N - 1)) of the sorted row, first row with the
//    least median).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "orbx_internal.cuh"

using namespace orbx;

namespace {

struct Writer {
    uint8_t* dst; size_t cap; size_t n = 0; bool text;
    void raw(const void* p, size_t k) { if (dst && n + k <= cap) memcpy(dst + n, p, k); n += k; }
    void str(const char* s) { raw(s, strlen(s)); }
    void i32(int v) { if (text) { char b[16]; snprintf(b, sizeof b, " %d", v); str(b); } else raw(&v, 4); }
    void boolean(bool v) { if (text) str(v ? " 1" : " 0"); else { const uint8_t b = v; raw(&b, 1); } }
    void f32(float v) { if (text) { char b[32]; snprintf(b, sizeof b, " %.9e", (double)v); str(b); } else raw(&v, 4); }   // max_digits10 of float
    void bytes(const uint8_t* p, size_t k)
    {
        if (!text) { raw(p, k); return; }
        char b[8];
        for (size_t i = 0; i < k; ++i) { snprintf(b, sizeof b, " %u", (unsigned)p[i]); str(b); }
    }
};

struct Reader {
    const uint8_t* src; size_t len; size_t pos = 0; bool text; bool ok = true;
    bool raw(void* p, size_t k) { if (pos + k > len) return ok = false; memcpy(p, src + pos, k); pos += k; return true; }
    bool token(char* buf, size_t cap)
    {
        while (pos < len && (src[pos] == ' ' || src[pos] == '\n' || src[pos] == '\r' || src[pos] == '\t')) ++pos;
        size_t k = 0;
        while (pos < len && !(src[pos] == ' ' || src[pos] == '\n' || src[pos] == '\r' || src[pos] == '\t') && k + 1 < cap) buf[k++] = (char)src[pos++];
        buf[k] = 0;
        return k > 0 ? true : (ok = false);
    }
    int i32() { if (!text) { int v = 0; raw(&v, 4); return v; } char b[48]; if (!token(b, sizeof b)) return 0; return (int)strtol(b, nullptr, 10); }
    bool boolean() { if (!text) { uint8_t v = 0; raw(&v, 1); return v != 0; } return i32() != 0; }
    float f32() { if (!text) { float v = 0; raw(&v, 4); return v; } char b[64]; if (!token(b, sizeof b)) return 0.f; return strtof(b, nullptr); }
    void bytes(uint8_t* p, size_t k)
    {
        if (!text) { raw(p, k); return; }
        for (size_t i = 0; i < k && ok; ++i) p[i] = (uint8_t)i32();
    }
};

}  // namespace

extern "C" {

// serializeMatrix(ar, mat) for a CV_8U matrix (include/SerializationUtils.h:76-100): cols, rows, type, continuous, then the
// bytes (row by row if the matrix is not continuous; the stream is the same bytes either way).
int64_t orbx_serialize_matrix_u8(int text, const uint8_t* data, int rows, int cols, size_t step, uint8_t* dst, size_t dst_capacity)
{
    if (rows < 0 || cols < 0 || (rows > 0 && cols > 0 && !data) || (step != 0 && step < (size_t)cols)) return fail(ORBX_ERR_INVALID_ARG, "bad matrix");
    if (step == 0) step = (size_t)cols;
    Writer w{dst, dst_capacity, 0, text != 0};
    const bool continuous = step == (size_t)cols || rows <= 1;
    w.i32(cols); w.i32(rows); w.i32(0 /* CV_8UC1 */); w.boolean(continuous);
    for (int r = 0; r < rows; ++r) w.bytes(data + (size_t)r * step, (size_t)cols);
    if (dst && w.n > dst_capacity) return fail(ORBX_ERR_CAPACITY, "need %zu bytes", w.n);
    return (int64_t)w.n;
}

// The loading half: parses the header; with dst == NULL only reports the shape, otherwise fills rows x cols bytes (dst_step
// bytes per row).  Returns the number of stream bytes consumed, or a negative orbx_status.
int64_t orbx_deserialize_matrix_u8(int text, const uint8_t* src, size_t src_len, int* rows, int* cols, uint8_t* dst, size_t dst_step,
                                   size_t dst_capacity)
{
    if (!src) return fail(ORBX_ERR_INVALID_ARG, "src is NULL");
    Reader r{src, src_len, 0, text != 0};
    const int c = r.i32(), n = r.i32(), type = r.i32();
    r.boolean();
    if (!r.ok || c < 0 || n < 0) return fail(ORBX_ERR_INVALID_ARG, "truncated or malformed matrix header");
    if (type != 0) return fail(ORBX_ERR_UNSUPPORTED, "matrix type %d is not CV_8UC1", type);
    if (rows) *rows = n;
    if (cols) *cols = c;
    if (!dst) return 0;
    if (dst_step == 0) dst_step = (size_t)c;
    if (dst_step < (size_t)c || (n > 0 && dst_capacity < (size_t)(n - 1) * dst_step + (size_t)c)) return fail(ORBX_ERR_CAPACITY, "destination too small");
    for (int i = 0; i < n; ++i) r.bytes(dst + (size_t)i * dst_step, (size_t)c);
    if (!r.ok) return fail(ORBX_ERR_INVALID_ARG, "truncated matrix data");
    return (int64_t)r.pos;
}

// serializeVectorKeyPoints (include/SerializationUtils.h:118-153): NumEl, then per key point angle, response, size, pt.x,
// pt.y, class_id, octave — note the order differs from the in-memory layout.
int64_t orbx_serialize_keypoints(int text, const orbx_keypoint* kps, int n, uint8_t* dst, size_t dst_capacity)
{
    if (n < 0 || (n > 0 && !kps)) return fail(ORBX_ERR_INVALID_ARG, "bad key points");
    Writer w{dst, dst_capacity, 0, text != 0};
    w.i32(n);
    for (int i = 0; i < n; ++i) {
        w.f32(kps[i].angle); w.f32(kps[i].response); w.f32(kps[i].size); w.f32(kps[i].x); w.f32(kps[i].y);
        w.i32(kps[i].class_id); w.i32(kps[i].octave);
    }
    if (dst && w.n > dst_capacity) return fail(ORBX_ERR_CAPACITY, "need %zu bytes", w.n);
    return (int64_t)w.n;
}

int64_t orbx_deserialize_keypoints(int text, const uint8_t* src, size_t src_len, int* n_out, orbx_keypoint* kps, int capacity)
{
    if (!src || !n_out) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    Reader r{src, src_len, 0, text != 0};
    const int n = r.i32();
    if (!r.ok || n < 0) return fail(ORBX_ERR_INVALID_ARG, "truncated or malformed key point count");
    *n_out = n;
    if (!kps) return 0;
    if (capacity < n) return fail(ORBX_ERR_CAPACITY, "need room for %d key points", n);
    for (int i = 0; i < n; ++i) {
        orbx_keypoint k;
        k.angle = r.f32(); k.response = r.f32(); k.size = r.f32(); k.x = r.f32(); k.y = r.f32(); k.class_id = r.i32(); k.octave = r.i32();
        kps[i] = k;
    }
    if (!r.ok) return fail(ORBX_ERR_INVALID_ARG, "truncated key point data");
    return (int64_t)r.pos;
}

}  // extern "C"

// ---- batched ComputeDistinctiveDescriptors ---------------------------------------------------------------------------------
namespace orbx {

constexpr int kDdMaxN = 64;          // observations per map point handled by the warp kernel (more: host path)
constexpr int kDdWarps = 4;

// One warp per map point.  dist[i][j] in shared memory (u16), median of row i = the k-th smallest with k = (int)(0.5*(N-1))
// (std::sort + index, src/MapPoint.cc:388-390) by rank counting, result = the first row with the least median (strict '<',
// :392-396) = min over (median << 8 | row).
__global__ void __launch_bounds__(32 * kDdWarps) distinctive_kernel(const uint8_t* __restrict__ desc, const int* __restrict__ offsets,
                                                                    int n_points, int* __restrict__ best)
{
    __shared__ uint16_t sd[kDdWarps][kDdMaxN * kDdMaxN];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = blockIdx.x * kDdWarps + warp;
    if (p >= n_points) return;
    const int o = offsets[p], N = offsets[p + 1] - o;
    if (N <= 0 || N > kDdMaxN) { if (lane == 0) best[p] = N <= 0 ? -1 : -2; return; }      // -2: caller takes the host path
    const uint32_t* D = reinterpret_cast<const uint32_t*>(desc) + (size_t)o * 8;
    uint16_t* d = sd[warp];
    for (int e = lane; e < N * N; e += 32) {
        const int i = e / N, j = e - i * N;
        int acc = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) acc += __popc(__ldg(D + i * 8 + k) ^ __ldg(D + j * 8 + k));
        d[e] = (uint16_t)acc;
    }
    __syncwarp();
    const int kth = (int)(0.5 * (N - 1));
    uint32_t key = 0xffffffffu;
    for (int i = lane; i < N; i += 32) {
        const uint16_t* row = d + i * N;
        int median = 0;
        for (int j = 0; j < N; ++j) {
            const int v = row[j];
            int rank = 0;
            for (int t = 0; t < N; ++t) { const int u = row[t]; rank += (u < v) || (u == v && t < j); }
            if (rank == kth) median = v;
        }
        key = min(key, ((uint32_t)median << 8) | (uint32_t)i);
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) key = min(key, __shfl_xor_sync(0xffffffffu, key, s));
    if (lane == 0) best[p] = (int)(key & 0xffu);
}

}  // namespace orbx

extern "C" int orbx_distinctive_descriptors(int device, const uint8_t* descriptors, const int32_t* offsets, int n_points, int32_t* best_idx)
{
    if (n_points < 0 || (n_points > 0 && (!offsets || !best_idx))) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (n_points == 0) return ORBX_OK;
    for (int p = 0; p < n_points; ++p)
        if (offsets[p + 1] < offsets[p] || offsets[0] != 0) return fail(ORBX_ERR_INVALID_ARG, "offsets must start at 0 and not decrease");
    const int total = offsets[n_points];
    if (total > 0 && !descriptors) return fail(ORBX_ERR_INVALID_ARG, "descriptors is NULL");
    int rc = set_device(device);
    if (rc) return rc;
    Lease L(device, g_fuse_arena);          // MapPoint::ComputeDistinctiveDescriptors runs on the local-mapping thread
    const size_t n_off = (size_t)n_points + 1;
    if ((rc = L.reserve(lease_pad((size_t)total * 32) + lease_pad(n_off * 4) + lease_pad((size_t)n_points * 4)))) return rc;
    const size_t o_desc = L.take<uint8_t>((size_t)total * 32), o_off = L.take<int>(n_off);
    L.upload_end = L.off;
    const size_t o_best = L.take<int>(n_points);
    if (total > 0) memcpy(L.host<uint8_t>(o_desc), descriptors, (size_t)total * 32);
    memcpy(L.host<int>(o_off), offsets, n_off * 4);
    cudaStream_t st = L.A.st;
    cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) {
        distinctive_kernel<<<(n_points + kDdWarps - 1) / kDdWarps, 32 * kDdWarps, 0, st>>>(L.dev<uint8_t>(o_desc), L.dev<int>(o_off), n_points,
                                                                                         L.dev<int>(o_best));
        count_launch();
        e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(best_idx, L.dev<int>(o_best), sizeof(int) * (size_t)n_points, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "distinctive descriptors: %s", cudaGetErrorString(e));
    // map points with more than 64 observations: the single-point host entry (same arithmetic)
    for (int p = 0; p < n_points; ++p)
        if (best_idx[p] == -2) {
            int b = 0;
            if ((rc = orbx_distinctive_descriptor(descriptors + (size_t)offsets[p] * 32, offsets[p + 1] - offsets[p], &b))) return rc;
            best_idx[p] = b;
        }
    return ORBX_OK;
}
