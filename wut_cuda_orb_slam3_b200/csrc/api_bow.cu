// api_bow.cu — host side of the bag-of-words transform and the vocabulary-guided searches (C ABI of include/orbx.h).
//
// Reference interfaces replaced (paths relative to the reference root):
//   DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB>  Thirdparty/DBoW2/DBoW2/TemplatedVocabulary.h (transform :1126-1259,
//       loadFromTextFile :1337-1420), BowVector.cpp, FeatureVector.cpp, ScoringObject.cpp (L1 score :24-65)
//   Frame::ComputeBoW                                     src/Frame.cc:768-775
//   ORBmatcher::SearchByBoW (KF, Frame) / (KF, KF)        src/ORBmatcher1.cc:225-427, src/ORBmatcher2.cc:36-171
//   ORBmatcher::SearchForTriangulation                    src/ORBmatcher2.cc:173-471
// The Hamming work runs in kernels_bow.cu; the std::map bookkeeping (word weights, node -> feature lists, the 30-bin
// rotation histogram) is small ordered host logic and stays on the host, in the reference's own evaluation order so that
// the floating-point sums are bit-identical.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>
#include <string>
#include <type_traits>
#include <vector>

#include "orbx_internal.cuh"

struct orbx_vocabulary {
    int device = 0;
    int n_nodes = 0, n_words = 0, k = 0, L = 0, scoring = 0, weighting = 0;
    // device copy
    int *d_child_begin = nullptr, *d_child_count = nullptr, *d_child_id = nullptr, *d_word_of_node = nullptr;
    uint8_t* d_cdesc = nullptr;
    double* d_weight = nullptr;
    orbx::VocabDev dev{};
};

namespace orbx {

namespace {

int check_fv(const orbx_feature_vector* fv, int n_features, const char* name)
{
    if (!fv || fv->n_nodes < 0 || (fv->n_nodes > 0 && (!fv->node_ids || !fv->offsets))) return fail(ORBX_ERR_INVALID_ARG, "%s: bad feature vector", name);
    if (fv->n_nodes == 0) return ORBX_OK;
    if (fv->offsets[0] != 0) return fail(ORBX_ERR_INVALID_ARG, "%s: offsets[0] != 0", name);
    for (int i = 0; i < fv->n_nodes; ++i) {
        if (fv->offsets[i + 1] < fv->offsets[i]) return fail(ORBX_ERR_INVALID_ARG, "%s: offsets not monotone", name);
        if (i > 0 && fv->node_ids[i] <= fv->node_ids[i - 1]) return fail(ORBX_ERR_INVALID_ARG, "%s: node ids not ascending", name);
    }
    const int total = fv->offsets[fv->n_nodes];
    if (total > 0 && !fv->indices) return fail(ORBX_ERR_INVALID_ARG, "%s: indices missing", name);
    for (int i = 0; i < total; ++i)
        if ((int)fv->indices[i] < 0 || (int)fv->indices[i] >= n_features) return fail(ORBX_ERR_INVALID_ARG, "%s: feature index %d out of range", name, i);
    return ORBX_OK;
}

// SearchForTriangulation's rotation filter over vMatches12 (src/ORBmatcher2.cc:429-447); one histogram entry per match, so the
// filter depends on bin sizes only.  *nm is decremented per dropped match.
int tri_rotation_filter(const orbx_keypoint* kp_a, const orbx_keypoint* kp_b, int n_a, int32_t* mA, int* nm)
{
    const int H = 30;
    int count[H] = {0};
    std::vector<int> bin(n_a, -1);
    for (int i = 0; i < n_a; ++i) {
        if (mA[i] < 0) continue;
        const int b = rotation_bin(kp_a[i].angle, kp_b[mA[i]].angle);
        if (b < 0) return fail(ORBX_ERR_INVALID_ARG, "keypoint angles out of range (the reference asserts)");
        bin[i] = b; count[b]++;
    }
    int i1, i2, i3;
    three_maxima(count, H, i1, i2, i3);
    for (int i = 0; i < n_a; ++i)
        if (bin[i] >= 0 && bin[i] != i1 && bin[i] != i2 && bin[i] != i3) { mA[i] = -1; --*nm; }
    return ORBX_OK;
}

// SearchByBoW's rotation histogram + ComputeThreeMaxima over one key frame's row (src/ORBmatcher1.cc:344-356, 406-427;
// src/ORBmatcher2.cc:127-139, 152-169).  One histogram entry per accepted match; the filter depends on bin sizes only, so the
// entry order is irrelevant.  Mode 0: row[j] = A (key frame) index of the fixed Frame's feature j; mode 1: row[i] = B (key
// frame) index of the fixed KF1's feature i.  inv / inv_right (may be NULL) are the key frame's inverse maps, kept consistent.
// *nm is decremented per dropped match.
int bow_rotation_filter(int mode, int n, int32_t* row, const float* angle_fixed, const float* angle_kf, int32_t* inv, int32_t* inv_right,
                        int* nm)
{
    const int H = 30;
    int count[H] = {0};
    std::vector<int> bin(n, -1);
    for (int t = 0; t < n; ++t) {
        if (row[t] < 0) continue;
        const int b = mode == 0 ? rotation_bin(angle_kf[row[t]], angle_fixed[t]) : rotation_bin(angle_fixed[t], angle_kf[row[t]]);
        if (b < 0) return fail(ORBX_ERR_INVALID_ARG, "keypoint angles out of range (the reference asserts)");
        bin[t] = b; count[b]++;
    }
    int i1, i2, i3;
    three_maxima(count, H, i1, i2, i3);
    for (int t = 0; t < n; ++t) {
        if (bin[t] < 0 || bin[t] == i1 || bin[t] == i2 || bin[t] == i3) continue;
        const int o = row[t];
        row[t] = -1;
        if (mode == 0) { if (inv && inv[o] == t) inv[o] = -1; if (inv_right && inv_right[o] == t) inv_right[o] = -1; }
        else if (inv) inv[o] = -1;
        --*nm;
    }
    return ORBX_OK;
}

// orbx_search_by_bow_batch, plus the inverse maps the single call returns: inv / inv_right (may be NULL) are HOST arrays over
// the key frames' features, packed in order (sum of kfs[k].n): mode 0 match_a (inv_right: its right-camera twin), mode 1 match_b.
// They are written only when n > 0 (the caller initialises them to -1).
int search_by_bow_batch(int device, int mode, const uint8_t* desc, const float* angle, const uint8_t* valid, int n,
                        const orbx_feature_vector* fv, int nleft, int n_kf, const orbx_bow_view* kfs, float nn_ratio, int check_orientation,
                        int32_t* match, int* n_matches, int32_t* inv, int32_t* inv_right)
{
    if (n_kf < 0) return fail(ORBX_ERR_INVALID_ARG, "search_by_bow: n_kf < 0");
    if (n_kf == 0) return ORBX_OK;
    if (n_kf > 65535) return fail(ORBX_ERR_UNSUPPORTED, "search_by_bow: more than 65535 key frames");
    if ((mode != 0 && mode != 1) || !kfs || !n_matches || n < 0 || (n > 0 && (!desc || !match)) || (mode == 1 && n > 0 && !valid) ||
        (check_orientation && n > 0 && !angle))
        return fail(ORBX_ERR_INVALID_ARG, "search_by_bow: bad arguments");
    if (mode == 1 && nleft >= 0) return fail(ORBX_ERR_INVALID_ARG, "search_by_bow: nleft applies to mode 0 only");
    int rc;
    if ((rc = check_fv(fv, n, "fv"))) return rc;
    // the single call's checks, per key frame
    size_t n_feat = 0, n_nodes = 0, n_idx = 0;
    for (int k = 0; k < n_kf; ++k) {
        const orbx_bow_view& V = kfs[k];
        if (V.n < 0 || (V.n > 0 && (!V.desc || !V.valid)) || (check_orientation && V.n > 0 && !V.angle))
            return fail(ORBX_ERR_INVALID_ARG, "search_by_bow: kfs[%d]: bad arguments", k);
        char name[32];
        snprintf(name, sizeof name, "kfs[%d].fv", k);
        if ((rc = check_fv(&V.fv, V.n, name))) return rc;
        n_feat += (size_t)V.n; n_nodes += (size_t)V.fv.n_nodes; n_idx += V.fv.n_nodes ? (size_t)V.fv.offsets[V.fv.n_nodes] : 0;
    }
    const size_t rows = (size_t)n_kf * n;
    if (n > 0) {
        if ((rc = set_device(device))) return rc;
        const int f_nodes = fv->n_nodes, f_idx = f_nodes ? fv->offsets[f_nodes] : 0;
        const size_t vf = mode == 1 ? (size_t)n : 0;
        // KF -> Frame runs on the tracking thread, KF <-> KF on loop closing
        Lease L(device, mode == 0 ? g_arena : g_loop_arena);
        const size_t total = lease_pad((size_t)n_kf * sizeof(BowKF)) + lease_pad((size_t)n * 32) + lease_pad(vf) + lease_pad((size_t)f_nodes * 4) +
                             lease_pad((size_t)(f_nodes + 1) * 4) + lease_pad((size_t)f_idx * 4) + lease_pad(n_feat * 32) + lease_pad(n_feat) +
                             lease_pad(n_nodes * 4) + lease_pad((n_nodes + n_kf) * 4) + lease_pad(n_idx * 4) +
                             lease_pad((size_t)n_kf * f_nodes * 16) + lease_pad((size_t)n_kf * 4) + lease_pad(rows * 4) + 2 * lease_pad(n_feat * 4);
        if ((rc = L.reserve(total))) return rc;
        // upload range: the key-frame table, the fixed side once, then every key frame's arrays packed back to back
        const size_t o_kf = L.take<BowKF>(n_kf), o_d = L.take<uint8_t>((size_t)n * 32), o_v = L.take<uint8_t>(vf),
                     o_n = L.take<uint32_t>(f_nodes), o_o = L.take<int32_t>(f_nodes + 1), o_i = L.take<uint32_t>(f_idx),
                     o_dk = L.take<uint8_t>(n_feat * 32), o_vk = L.take<uint8_t>(n_feat), o_nk = L.take<uint32_t>(n_nodes),
                     o_ok = L.take<int32_t>(n_nodes + n_kf), o_ik = L.take<uint32_t>(n_idx);
        L.upload_end = L.off;
        // device-only scratch / outputs
        const size_t o_jobs = L.take<int4>((size_t)n_kf * f_nodes), o_cnt = L.take<int>(n_kf), o_row = L.take<int>(rows),
                     o_feat = L.take<int>(n_feat), o_right = L.take<int>(n_feat);
        memcpy(L.host<uint8_t>(o_d), desc, (size_t)n * 32);
        if (vf) memcpy(L.host<uint8_t>(o_v), valid, vf);
        if (f_nodes) {
            memcpy(L.host<uint32_t>(o_n), fv->node_ids, (size_t)f_nodes * 4);
            memcpy(L.host<int32_t>(o_o), fv->offsets, (size_t)(f_nodes + 1) * 4);
            if (f_idx) memcpy(L.host<uint32_t>(o_i), fv->indices, (size_t)f_idx * 4);
        }
        BowKF* T = L.host<BowKF>(o_kf);
        size_t f0 = 0, n0 = 0, i0 = 0, b0 = 0;                   // running bases: features, node ids, indices, offsets
        for (int k = 0; k < n_kf; ++k) {
            const orbx_bow_view& V = kfs[k];
            const int nn = V.fv.n_nodes, ni = nn ? V.fv.offsets[nn] : 0;
            BowKF e{};
            e.desc = L.dev<uint8_t>(o_dk) + f0 * 32; e.valid = L.dev<uint8_t>(o_vk) + f0;
            e.node_ids = L.dev<uint32_t>(o_nk) + n0; e.offsets = L.dev<int32_t>(o_ok) + b0; e.indices = L.dev<uint32_t>(o_ik) + i0;
            e.n = V.n; e.n_nodes = nn; e.base = f0;
            T[k] = e;
            if (V.n) {
                memcpy(L.host<uint8_t>(o_dk) + f0 * 32, V.desc, (size_t)V.n * 32);
                memcpy(L.host<uint8_t>(o_vk) + f0, V.valid, (size_t)V.n);
            }
            if (nn) {
                memcpy(L.host<uint32_t>(o_nk) + n0, V.fv.node_ids, (size_t)nn * 4);
                if (ni) memcpy(L.host<uint32_t>(o_ik) + i0, V.fv.indices, (size_t)ni * 4);
            }
            for (int p = 0; p <= nn; ++p) L.host<int32_t>(o_ok)[b0 + p] = nn ? V.fv.offsets[p] : 0;
            f0 += (size_t)V.n; n0 += (size_t)nn; i0 += (size_t)ni; b0 += (size_t)nn + 1;
        }
        BowBatchArgs A{};
        A.mode = mode; A.n_kf = n_kf; A.kfs = L.dev<BowKF>(o_kf);
        A.n = n; A.desc = L.dev<uint8_t>(o_d); A.valid = vf ? L.dev<uint8_t>(o_v) : nullptr;
        A.n_nodes = f_nodes; A.node_ids = L.dev<uint32_t>(o_n); A.offsets = L.dev<int32_t>(o_o); A.indices = L.dev<uint32_t>(o_i);
        A.nleft = nleft; A.nn_ratio = nn_ratio;
        A.jobs = L.dev<int4>(o_jobs); A.job_count = L.dev<int>(o_cnt); A.job_stride = f_nodes; A.row = L.dev<int>(o_row);
        A.feat = mode == 1 || inv ? L.dev<int>(o_feat) : nullptr;
        A.feat_right = mode == 0 && inv_right ? L.dev<int>(o_right) : nullptr;
        cudaStream_t st = L.A.st;
        cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_search_by_bow_batch(A, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(match, A.row, rows * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && inv && n_feat) e = cudaMemcpyAsync(inv, A.feat, n_feat * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess && A.feat_right && n_feat) e = cudaMemcpyAsync(inv_right, A.feat_right, n_feat * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "search_by_bow: %s", cudaGetErrorString(e));
    }
    // the return value and the rotation filter per key frame, on the host as in the reference
    size_t f0 = 0;
    for (int k = 0; k < n_kf; ++k) {
        int32_t* r = match + (size_t)k * n;
        int nm = 0;
        for (int t = 0; t < n; ++t) nm += r[t] >= 0;
        if (check_orientation &&
            (rc = bow_rotation_filter(mode, n, r, angle, kfs[k].angle, inv ? inv + f0 : nullptr, inv_right ? inv_right + f0 : nullptr, &nm)))
            return rc;
        n_matches[k] = nm;
        f0 += (size_t)kfs[k].n;
    }
    return ORBX_OK;
}

}  // namespace

}  // namespace orbx

using namespace orbx;

extern "C" {

int orbx_vocab_create(int device, int n_nodes, const int32_t* parent, const uint8_t* descriptors, const double* weights, int k,
                      int L, int scoring, int weighting, orbx_vocabulary** out)
{
    if (!out) return fail(ORBX_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (n_nodes < 1 || !parent || !descriptors || !weights || L < 0 || scoring < 0 || scoring > 5 || weighting < 0 || weighting > 3)
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (parent[0] != -1) return fail(ORBX_ERR_INVALID_ARG, "parent[0] must be -1 (node 0 is the root)");
    for (int i = 1; i < n_nodes; ++i)
        if (parent[i] < 0 || parent[i] >= n_nodes || parent[i] == i) return fail(ORBX_ERR_INVALID_ARG, "parent[%d] = %d invalid", i, parent[i]);
    int rc = set_device(device);
    if (rc) return rc;
    // children in creation order == ascending node id (TemplatedVocabulary.h:1391-1394)
    std::vector<int> count(n_nodes, 0), begin(n_nodes, 0), child_id(std::max(n_nodes - 1, 1), 0), word(n_nodes, -1);
    for (int i = 1; i < n_nodes; ++i) count[parent[i]]++;
    for (int i = 0; i < n_nodes; ++i)
        if (count[i] > 255) return fail(ORBX_ERR_UNSUPPORTED, "node %d has %d children (max 255)", i, count[i]);
    for (int i = 1; i < n_nodes; ++i) begin[i] = begin[i - 1] + count[i - 1];
    std::vector<int> fill(begin);
    std::vector<uint8_t> cdesc((size_t)std::max(n_nodes - 1, 1) * 32, 0);
    for (int i = 1; i < n_nodes; ++i) {
        const int slot = fill[parent[i]]++;
        child_id[slot] = i;
        memcpy(&cdesc[(size_t)slot * 32], descriptors + (size_t)i * 32, 32);
    }
    int n_words = 0;
    for (int i = 1; i < n_nodes; ++i)
        if (count[i] == 0) word[i] = n_words++;                 // words numbered in node order (TemplatedVocabulary.h:1408-1415)
    orbx_vocabulary* v = new orbx_vocabulary;
    v->device = device; v->n_nodes = n_nodes; v->n_words = n_words; v->k = k; v->L = L; v->scoring = scoring; v->weighting = weighting;
    cudaError_t e;
    auto up = [&](auto** dst, const auto* src, size_t cnt) {
        using T = std::remove_cv_t<std::remove_pointer_t<decltype(src)>>;
        if ((e = cudaMalloc((void**)dst, std::max<size_t>(cnt, 1) * sizeof(T))) != cudaSuccess) return false;
        return (e = cudaMemcpy(*dst, src, cnt * sizeof(T), cudaMemcpyHostToDevice)) == cudaSuccess;
    };
    if (!up(&v->d_child_begin, begin.data(), (size_t)n_nodes) || !up(&v->d_child_count, count.data(), (size_t)n_nodes) ||
        !up(&v->d_child_id, child_id.data(), child_id.size()) || !up(&v->d_word_of_node, word.data(), (size_t)n_nodes) ||
        !up(&v->d_cdesc, cdesc.data(), cdesc.size()) || !up(&v->d_weight, weights, (size_t)n_nodes)) {
        orbx_vocab_destroy(v);
        return fail(ORBX_ERR_CUDA, "vocabulary upload: %s", cudaGetErrorString(e));
    }
    v->dev = VocabDev{v->d_child_begin, v->d_child_count, v->d_child_id, v->d_cdesc, v->d_word_of_node, v->d_weight};
    *out = v;
    return ORBX_OK;
}

int orbx_vocab_load_text(int device, const char* path, orbx_vocabulary** out)
{
    if (!out) return fail(ORBX_ERR_INVALID_ARG, "out is NULL");
    *out = nullptr;
    if (!path) return fail(ORBX_ERR_INVALID_ARG, "path is NULL");
    std::ifstream f(path);
    if (!f.is_open()) return fail(ORBX_ERR_INVALID_ARG, "cannot open %s", path);
    std::string line;
    if (!std::getline(f, line)) return fail(ORBX_ERR_INVALID_ARG, "%s: empty file", path);
    int k = -1, L = -1, n1 = -1, n2 = -1;
    { std::stringstream ss(line); ss >> k >> L >> n1 >> n2; }
    if (k < 0 || k > 20 || L < 1 || L > 10 || n1 < 0 || n1 > 5 || n2 < 0 || n2 > 3)          // TemplatedVocabulary.h:1360-1364
        return fail(ORBX_ERR_INVALID_ARG, "%s: not a vocabulary text file", path);
    std::vector<int32_t> parent{-1};
    std::vector<uint8_t> desc(32, 0);
    std::vector<double> weight{0.0};
    while (std::getline(f, line)) {
        // (the reference's while(!f.eof()) loop would turn a trailing blank line into one bogus node with an uninitialised parent;
        //  blank lines are skipped here)
        if (line.find_first_not_of(" \t\r\n") == std::string::npos) continue;
        std::stringstream ss(line);
        int pid = -1, is_leaf = 0;
        ss >> pid >> is_leaf;
        const int nid = (int)parent.size();
        if (ss.fail() || pid < 0 || pid >= nid) return fail(ORBX_ERR_INVALID_ARG, "%s: node %d has parent %d", path, nid, pid);
        uint8_t d[32];
        for (int i = 0; i < 32; ++i) { int b = -1; ss >> b; if (ss.fail() || b < 0 || b > 255) return fail(ORBX_ERR_INVALID_ARG, "%s: node %d descriptor", path, nid); d[i] = (uint8_t)b; }
        double w = 0.0;
        ss >> w;
        if (ss.fail()) return fail(ORBX_ERR_INVALID_ARG, "%s: node %d weight", path, nid);
        parent.push_back(pid);
        desc.insert(desc.end(), d, d + 32);
        weight.push_back(w);
        (void)is_leaf;      // leaves are the nodes without children; in a well-formed file that is the is_leaf column
    }
    return orbx_vocab_create(device, (int)parent.size(), parent.data(), desc.data(), weight.data(), k, L, n1, n2, out);
}

void orbx_vocab_destroy(orbx_vocabulary* v)
{
    if (!v) return;
    cudaSetDevice(v->device);
    cudaFree(v->d_child_begin); cudaFree(v->d_child_count); cudaFree(v->d_child_id); cudaFree(v->d_word_of_node);
    cudaFree(v->d_cdesc); cudaFree(v->d_weight);
    delete v;
}

int orbx_vocab_info(const orbx_vocabulary* v, int* n_nodes, int* n_words, int* k, int* L)
{
    if (!v) return fail(ORBX_ERR_INVALID_ARG, "vocabulary is NULL");
    if (n_nodes) *n_nodes = v->n_nodes;
    if (n_words) *n_words = v->n_words;
    if (k) *k = v->k;
    if (L) *L = v->L;
    return ORBX_OK;
}

int orbx_bow_transform(const orbx_vocabulary* v, const uint8_t* descriptors, int n, int levelsup, uint32_t* word_id, double* weight,
                       uint32_t* node_id)
{
    if (!v || n < 0 || (n > 0 && !descriptors)) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (n == 0) return ORBX_OK;
    if (v->n_nodes < 2) return fail(ORBX_ERR_INVALID_ARG, "empty vocabulary");
    int rc = set_device(v->device);
    if (rc) return rc;
    Lease L(v->device);
    if ((rc = L.reserve(lease_pad((size_t)n * 32) + 2 * lease_pad((size_t)n * 4) + lease_pad((size_t)n * 8)))) return rc;
    const size_t o_desc = L.take<uint8_t>((size_t)n * 32);
    L.upload_end = L.off;
    const size_t o_word = L.take<uint32_t>(n), o_node = L.take<uint32_t>(n), o_w = L.take<double>(n);
    memcpy(L.host<uint8_t>(o_desc), descriptors, (size_t)n * 32);
    cudaStream_t st = L.A.st;
    uint32_t* d_word = L.dev<uint32_t>(o_word);
    uint32_t* d_node = L.dev<uint32_t>(o_node);
    double* d_w = L.dev<double>(o_w);
    cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = launch_bow_descend(v->dev, L.dev<uint8_t>(o_desc), n, v->L - levelsup, d_word, d_w, d_node, st);
    if (e == cudaSuccess && word_id) e = cudaMemcpyAsync(word_id, d_word, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && weight) e = cudaMemcpyAsync(weight, d_w, (size_t)n * 8, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess && node_id) e = cudaMemcpyAsync(node_id, d_node, (size_t)n * 4, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "bow_transform: %s", cudaGetErrorString(e));
    return ORBX_OK;
}

int orbx_compute_bow(const orbx_vocabulary* v, const uint8_t* descriptors, int n, int levelsup, uint32_t* bow_ids, double* bow_vals,
                     int* n_bow, uint32_t* fv_nodes, int32_t* fv_offsets, uint32_t* fv_indices, int* n_fv)
{
    if (!v || n < 0 || !n_bow || !n_fv || !fv_offsets || (n > 0 && (!descriptors || !bow_ids || !bow_vals || !fv_nodes || !fv_indices)))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    *n_bow = 0; *n_fv = 0; fv_offsets[0] = 0;
    if (n == 0) return ORBX_OK;
    std::vector<uint32_t> word(n), node(n);
    std::vector<double> w(n);
    int rc = orbx_bow_transform(v, descriptors, n, levelsup, word.data(), w.data(), node.data());
    if (rc) return rc;
    // TemplatedVocabulary::transform(features, v, fv, levelsup) — TemplatedVocabulary.h:1126-1204
    std::map<uint32_t, double> bow;
    std::map<uint32_t, std::vector<uint32_t>> fv;
    const bool tf = v->weighting == ORBX_TF || v->weighting == ORBX_TF_IDF;
    for (int i = 0; i < n; ++i) {
        if (!(w[i] > 0)) continue;                                               // stopped word
        auto it = bow.lower_bound(word[i]);
        if (it != bow.end() && it->first == word[i]) { if (tf) it->second += w[i]; }        // addWeight / addIfNotExist (BowVector.cpp:34-58)
        else bow.insert(it, {word[i], w[i]});
        fv[node[i]].push_back((uint32_t)i);                                      // FeatureVector::addFeature (FeatureVector.cpp:32-46)
    }
    const bool must = v->scoring != ORBX_DOT_PRODUCT;                            // ScoringObject.h:73-89
    if (tf && !bow.empty() && !must) {
        const double nd = (double)bow.size();
        for (auto& kv : bow) kv.second /= nd;
    }
    if (must) {                                                                  // BowVector::normalize (BowVector.cpp:62-86)
        double norm = 0.0;
        if (v->scoring != ORBX_L2_NORM) { for (auto& kv : bow) norm += fabs(kv.second); }
        else { for (auto& kv : bow) norm += kv.second * kv.second; norm = sqrt(norm); }
        if (norm > 0.0) for (auto& kv : bow) kv.second /= norm;
    }
    int nb = 0;
    for (auto& kv : bow) { bow_ids[nb] = kv.first; bow_vals[nb] = kv.second; ++nb; }
    *n_bow = nb;
    int nf = 0, off = 0;
    for (auto& kv : fv) {
        fv_nodes[nf] = kv.first;
        for (uint32_t i : kv.second) fv_indices[off++] = i;
        fv_offsets[++nf] = off;
    }
    *n_fv = nf;
    return ORBX_OK;
}

int orbx_bow_score(const orbx_vocabulary* v, const uint32_t* ids_a, const double* vals_a, int na, const uint32_t* ids_b,
                   const double* vals_b, int nb, double* score)
{
    if (!v || !score || na < 0 || nb < 0 || (na > 0 && (!ids_a || !vals_a)) || (nb > 0 && (!ids_b || !vals_b)))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (v->scoring != ORBX_L1_NORM) return fail(ORBX_ERR_UNSUPPORTED, "only L1_NORM scoring (the ORBvoc.txt setting) is implemented");
    double s = 0;                                                                // L1Scoring::score (ScoringObject.cpp:24-65)
    int i = 0, j = 0;
    while (i < na && j < nb) {
        if (ids_a[i] == ids_b[j]) { s += fabs(vals_a[i] - vals_b[j]) - fabs(vals_a[i]) - fabs(vals_b[j]); ++i; ++j; }
        else if (ids_a[i] < ids_b[j]) ++i;
        else ++j;
    }
    *score = -s / 2.0;
    return ORBX_OK;
}

int orbx_search_by_bow(int device, int mode, const uint8_t* desc_a, const float* angle_a, const uint8_t* valid_a, int n_a,
                       const orbx_feature_vector* fv_a, const uint8_t* desc_b, const float* angle_b, const uint8_t* valid_b, int n_b,
                       const orbx_feature_vector* fv_b, int nleft_b, float nn_ratio, int check_orientation, int32_t* match_a,
                       int32_t* match_b, int* n_matches)
{
    // the one-key-frame batch; these are the arguments the view cannot carry (the batch checks the rest)
    if ((mode != 0 && mode != 1) || n_a < 0 || n_b < 0 || !n_matches || !fv_a || !fv_b) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    const bool kf_frame = mode == 0;
    orbx_bow_view V{};                                       // mode 0: A = pKF, mode 1: B = pKF2
    if (kf_frame) { V.n = n_a; V.desc = desc_a; V.angle = angle_a; V.valid = valid_a; V.fv = *fv_a; }
    else { V.n = n_b; V.desc = desc_b; V.angle = angle_b; V.valid = valid_b; V.fv = *fv_b; }
    const int n = kf_frame ? n_b : n_a;
    std::vector<int32_t> row(n, -1), inv(V.n, -1), inv_right(kf_frame && nleft_b >= 0 ? V.n : 0, -1);
    *n_matches = 0;
    const int rc = kf_frame ? search_by_bow_batch(device, 0, desc_b, angle_b, nullptr, n_b, fv_b, nleft_b, 1, &V, nn_ratio, check_orientation,
                                                  row.data(), n_matches, inv.data(), inv_right.empty() ? nullptr : inv_right.data())
                            : search_by_bow_batch(device, 1, desc_a, angle_a, valid_a, n_a, fv_a, nleft_b, 1, &V, nn_ratio, check_orientation,
                                                  row.data(), n_matches, inv.data(), nullptr);
    if (rc) return rc;
    int32_t* out_row = kf_frame ? match_b : match_a;
    int32_t* out_inv = kf_frame ? match_a : match_b;
    if (out_row) std::copy(row.begin(), row.end(), out_row);
    if (out_inv) std::copy(inv.begin(), inv.end(), out_inv);
    return ORBX_OK;
}

int orbx_search_by_bow_batch(int device, int mode, const uint8_t* desc, const float* angle, const uint8_t* valid, int n,
                             const orbx_feature_vector* fv, int nleft, int n_kf, const orbx_bow_view* kfs, float nn_ratio,
                             int check_orientation, int32_t* match, int* n_matches)
{
    return search_by_bow_batch(device, mode, desc, angle, valid, n, fv, nleft, n_kf, kfs, nn_ratio, check_orientation, match, n_matches,
                               nullptr, nullptr);
}

int orbx_search_for_triangulation(int device, const orbx_keypoint* kp_a, const uint8_t* desc_a, const uint8_t* free_a,
                                  const uint8_t* stereo_a, int n_a, const orbx_feature_vector* fv_a, const orbx_keypoint* kp_b,
                                  const uint8_t* desc_b, const uint8_t* free_b, const uint8_t* stereo_b, int n_b,
                                  const orbx_feature_vector* fv_b, const float* F12, const float* ep, const float* scale_b,
                                  const float* sigma2_b, int n_levels, int only_stereo, int coarse, int check_orientation,
                                  int32_t* match_a, int* n_matches)
{
    // the one-neighbour batch; these are the arguments the view cannot carry (the batch checks the rest)
    if (!n_matches || !F12 || !ep || !fv_b) return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    orbx_triangulation_view V{};
    V.n = n_b; V.kp = kp_b; V.desc = desc_b; V.free = free_b; V.stereo = stereo_b; V.fv = *fv_b;
    memcpy(V.F12, F12, sizeof V.F12); memcpy(V.ep, ep, sizeof V.ep);
    V.scale = scale_b; V.sigma2 = sigma2_b; V.n_levels = n_levels; V.coarse = coarse;
    *n_matches = 0;
    return orbx_search_for_triangulation_batch(device, kp_a, desc_a, free_a, stereo_a, n_a, fv_a, 1, &V, only_stereo, check_orientation,
                                               match_a, n_matches);
}

int orbx_search_for_triangulation_batch(int device, const orbx_keypoint* kp_a, const uint8_t* desc_a, const uint8_t* free_a,
                                        const uint8_t* stereo_a, int n_a, const orbx_feature_vector* fv_a, int n_kf,
                                        const orbx_triangulation_view* kfs, int only_stereo, int check_orientation, int32_t* match,
                                        int* n_matches)
{
    if (n_kf < 0) return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation: n_kf < 0");
    if (n_kf == 0) return ORBX_OK;
    if (n_kf > 65535) return fail(ORBX_ERR_UNSUPPORTED, "search_for_triangulation: more than 65535 neighbours");
    if (!kfs || !n_matches || n_a < 0 || (n_a > 0 && (!kp_a || !desc_a || !free_a || !stereo_a || !match)))
        return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation: bad arguments");
    int rc;
    if ((rc = check_fv(fv_a, n_a, "fv_a"))) return rc;
    // the single call's checks, per neighbour
    size_t n_feat = 0, n_nodes = 0, n_idx = 0;
    for (int k = 0; k < n_kf; ++k) {
        const orbx_triangulation_view& V = kfs[k];
        if (V.n < 0 || !V.scale || !V.sigma2 || V.n_levels < 1 || V.n_levels > kMaxLevels ||
            (V.n > 0 && (!V.kp || !V.desc || !V.free || !V.stereo)))
            return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation: kfs[%d]: bad arguments", k);
        char name[32];
        snprintf(name, sizeof name, "kfs[%d].fv", k);
        if ((rc = check_fv(&V.fv, V.n, name))) return rc;
        for (int j = 0; j < V.n; ++j)
            if (V.kp[j].octave < 0 || V.kp[j].octave >= V.n_levels)
                return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation: kfs[%d].kp[%d].octave out of range", k, j);
        n_feat += (size_t)V.n; n_nodes += (size_t)V.fv.n_nodes; n_idx += V.fv.n_nodes ? (size_t)V.fv.offsets[V.fv.n_nodes] : 0;
    }
    const size_t rows = (size_t)n_kf * n_a;
    if (n_a > 0) {
        if ((rc = set_device(device))) return rc;
        const int a_nodes = fv_a->n_nodes, a_idx = a_nodes ? fv_a->offsets[a_nodes] : 0;
        Lease L(device, g_fuse_arena);
        const size_t total = lease_pad((size_t)n_kf * sizeof(TriKF)) + lease_pad((size_t)n_a * 28) + lease_pad((size_t)n_a * 32) +
                             2 * lease_pad((size_t)n_a) + lease_pad((size_t)a_nodes * 4) + lease_pad((size_t)(a_nodes + 1) * 4) +
                             lease_pad((size_t)a_idx * 4) + lease_pad(n_feat * 28) + lease_pad(n_feat * 32) + 2 * lease_pad(n_feat) +
                             lease_pad(n_nodes * 4) + lease_pad((n_nodes + n_kf) * 4) + lease_pad(n_idx * 4) + lease_pad(rows * 16) +
                             lease_pad((size_t)n_kf * 4) + lease_pad(rows * 4);
        if ((rc = L.reserve(total))) return rc;
        // upload range: the neighbour table, KF1 once, then every neighbour's arrays packed back to back
        const size_t o_kf = L.take<TriKF>(n_kf), o_kpa = L.take<orbx_keypoint>(n_a), o_da = L.take<uint8_t>((size_t)n_a * 32),
                     o_fa = L.take<uint8_t>(n_a), o_sa = L.take<uint8_t>(n_a), o_na = L.take<uint32_t>(a_nodes),
                     o_oa = L.take<int32_t>(a_nodes + 1), o_ia = L.take<uint32_t>(a_idx), o_kpb = L.take<orbx_keypoint>(n_feat),
                     o_db = L.take<uint8_t>(n_feat * 32), o_fb = L.take<uint8_t>(n_feat), o_sb = L.take<uint8_t>(n_feat),
                     o_nb = L.take<uint32_t>(n_nodes), o_ob = L.take<int32_t>(n_nodes + n_kf), o_ib = L.take<uint32_t>(n_idx);
        L.upload_end = L.off;
        // device-only scratch / outputs
        const size_t o_jobs = L.take<int4>(rows), o_cnt = L.take<int>(n_kf), o_match = L.take<int>(rows);
        memcpy(L.host<orbx_keypoint>(o_kpa), kp_a, (size_t)n_a * sizeof(orbx_keypoint));
        memcpy(L.host<uint8_t>(o_da), desc_a, (size_t)n_a * 32);
        memcpy(L.host<uint8_t>(o_fa), free_a, (size_t)n_a);
        memcpy(L.host<uint8_t>(o_sa), stereo_a, (size_t)n_a);
        if (a_nodes) {
            memcpy(L.host<uint32_t>(o_na), fv_a->node_ids, (size_t)a_nodes * 4);
            memcpy(L.host<int32_t>(o_oa), fv_a->offsets, (size_t)(a_nodes + 1) * 4);
            if (a_idx) memcpy(L.host<uint32_t>(o_ia), fv_a->indices, (size_t)a_idx * 4);
        }
        TriKF* T = L.host<TriKF>(o_kf);
        size_t f0 = 0, n0 = 0, i0 = 0, b0 = 0;                   // running bases: features, node ids, indices, offsets
        for (int k = 0; k < n_kf; ++k) {
            const orbx_triangulation_view& V = kfs[k];
            const int nn = V.fv.n_nodes, ni = nn ? V.fv.offsets[nn] : 0;
            TriKF e{};
            e.kp = L.dev<orbx_keypoint>(o_kpb) + f0; e.desc = L.dev<uint8_t>(o_db) + f0 * 32;
            e.free = L.dev<uint8_t>(o_fb) + f0; e.stereo = L.dev<uint8_t>(o_sb) + f0;
            e.node_ids = L.dev<uint32_t>(o_nb) + n0; e.offsets = L.dev<int32_t>(o_ob) + b0; e.indices = L.dev<uint32_t>(o_ib) + i0;
            e.n = V.n; e.n_nodes = nn; e.coarse = V.coarse != 0;
            memcpy(e.F12, V.F12, sizeof e.F12); memcpy(e.ep, V.ep, sizeof e.ep);
            for (int l = 0; l < V.n_levels; ++l) { e.scale[l] = V.scale[l]; e.sigma2[l] = V.sigma2[l]; }
            T[k] = e;
            if (V.n) {
                memcpy(L.host<orbx_keypoint>(o_kpb) + f0, V.kp, (size_t)V.n * sizeof(orbx_keypoint));
                memcpy(L.host<uint8_t>(o_db) + f0 * 32, V.desc, (size_t)V.n * 32);
                memcpy(L.host<uint8_t>(o_fb) + f0, V.free, (size_t)V.n);
                memcpy(L.host<uint8_t>(o_sb) + f0, V.stereo, (size_t)V.n);
            }
            if (nn) {
                memcpy(L.host<uint32_t>(o_nb) + n0, V.fv.node_ids, (size_t)nn * 4);
                if (ni) memcpy(L.host<uint32_t>(o_ib) + i0, V.fv.indices, (size_t)ni * 4);
            }
            for (int p = 0; p <= nn; ++p) L.host<int32_t>(o_ob)[b0 + p] = nn ? V.fv.offsets[p] : 0;
            f0 += (size_t)V.n; n0 += (size_t)nn; i0 += (size_t)ni; b0 += (size_t)nn + 1;
        }
        TriBatchArgs A{};
        A.n_kf = n_kf; A.kfs = L.dev<TriKF>(o_kf);
        A.n_a = n_a; A.kp_a = L.dev<orbx_keypoint>(o_kpa); A.desc_a = L.dev<uint8_t>(o_da); A.free_a = L.dev<uint8_t>(o_fa);
        A.stereo_a = L.dev<uint8_t>(o_sa);
        A.a_nodes = a_nodes; A.a_node_ids = L.dev<uint32_t>(o_na); A.a_offsets = L.dev<int32_t>(o_oa); A.a_indices = L.dev<uint32_t>(o_ia);
        A.only_stereo = only_stereo != 0;
        A.jobs = L.dev<int4>(o_jobs); A.job_count = L.dev<int>(o_cnt); A.match = L.dev<int>(o_match);
        cudaStream_t st = L.A.st;
        cudaError_t e = cudaMemcpyAsync(L.A.d, L.A.h, L.upload_end, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = launch_search_triangulation_batch(A, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(match, A.match, rows * 4, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "search_for_triangulation: %s", cudaGetErrorString(e));
    }
    // the return value and the rotation filter per neighbour, on the host as in the single call
    for (int k = 0; k < n_kf; ++k) {
        int32_t* mA = match + (size_t)k * n_a;
        int nm = 0;
        for (int i = 0; i < n_a; ++i) nm += mA[i] >= 0;
        if (check_orientation && (rc = tri_rotation_filter(kp_a, kfs[k].kp, n_a, mA, &nm))) return rc;
        n_matches[k] = nm;
    }
    return ORBX_OK;
}

}  // extern "C"
