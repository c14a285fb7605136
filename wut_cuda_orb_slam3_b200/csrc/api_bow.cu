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

struct DevBuf {                      // RAII bag of device allocations for one call
    std::vector<void*> ptrs;
    ~DevBuf() { for (void* p : ptrs) cudaFree(p); }
    template <typename T>
    int alloc(T** out, size_t count)
    {
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
        if (e != cudaSuccess) return fail(ORBX_ERR_OOM, "cudaMalloc(%zu): %s", count * sizeof(T), cudaGetErrorString(e));
        ptrs.push_back(p);
        *out = (T*)p;
        return ORBX_OK;
    }
    template <typename T>
    int upload(T** out, const T* host, size_t count)
    {
        int rc = alloc(out, count);
        if (rc) return rc;
        if (count) {
            cudaError_t e = cudaMemcpy(*out, host, count * sizeof(T), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "cudaMemcpy H2D: %s", cudaGetErrorString(e));
        }
        return ORBX_OK;
    }
};

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

// the lock-step walk over two ascending node lists (src/ORBmatcher1.cc:247-251, 397-404): pairs of positions with equal node id
void common_nodes(const orbx_feature_vector* a, const orbx_feature_vector* b, std::vector<std::pair<int, int>>& out)
{
    int i = 0, j = 0;
    while (i < a->n_nodes && j < b->n_nodes) {
        if (a->node_ids[i] == b->node_ids[j]) { out.emplace_back(i, j); ++i; ++j; }
        else if (a->node_ids[i] < b->node_ids[j]) ++i;      // lower_bound on an ascending list == advance
        else ++j;
    }
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
    DevBuf B;
    uint8_t* d_desc; uint32_t *d_word, *d_node; double* d_w;
    if ((rc = B.upload(&d_desc, descriptors, (size_t)n * 32)) || (rc = B.alloc(&d_word, (size_t)n)) || (rc = B.alloc(&d_node, (size_t)n)) ||
        (rc = B.alloc(&d_w, (size_t)n)))
        return rc;
    cudaError_t e = launch_bow_descend(v->dev, d_desc, n, v->L - levelsup, d_word, d_w, d_node, 0);
    if (e == cudaSuccess && word_id) e = cudaMemcpy(word_id, d_word, (size_t)n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && weight) e = cudaMemcpy(weight, d_w, (size_t)n * 8, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess && node_id) e = cudaMemcpy(node_id, d_node, (size_t)n * 4, cudaMemcpyDeviceToHost);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
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
    if ((mode != 0 && mode != 1) || n_a < 0 || n_b < 0 || !n_matches || (n_a > 0 && (!desc_a || !valid_a)) || (n_b > 0 && !desc_b) ||
        (mode == 1 && n_b > 0 && !valid_b) || (check_orientation && ((n_a > 0 && !angle_a) || (n_b > 0 && !angle_b))))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    if (mode == 1 && nleft_b >= 0) return fail(ORBX_ERR_INVALID_ARG, "nleft_b applies to mode 0 only");
    int rc;
    if ((rc = check_fv(fv_a, n_a, "fv_a")) || (rc = check_fv(fv_b, n_b, "fv_b"))) return rc;
    *n_matches = 0;
    std::vector<int32_t> mA(n_a, -1), mAR(n_a, -1), mB(n_b, -1);
    std::vector<std::pair<int, int>> common;
    common_nodes(fv_a, fv_b, common);
    if (!common.empty() && n_a > 0 && n_b > 0) {
        if ((rc = set_device(device))) return rc;
        std::vector<int4> pairs;
        for (auto& c : common)
            pairs.push_back(make_int4(fv_a->offsets[c.first], fv_a->offsets[c.first + 1], fv_b->offsets[c.second], fv_b->offsets[c.second + 1]));
        DevBuf B;
        BowSearchArgs A{};
        int4* d_pairs; uint32_t *d_ia, *d_ib; uint8_t *d_da, *d_db, *d_va, *d_vb = nullptr; int *d_mb, *d_ma, *d_mar;
        if ((rc = B.upload(&d_pairs, pairs.data(), pairs.size())) || (rc = B.upload(&d_ia, fv_a->indices, (size_t)fv_a->offsets[fv_a->n_nodes])) ||
            (rc = B.upload(&d_ib, fv_b->indices, (size_t)fv_b->offsets[fv_b->n_nodes])) || (rc = B.upload(&d_da, desc_a, (size_t)n_a * 32)) ||
            (rc = B.upload(&d_db, desc_b, (size_t)n_b * 32)) || (rc = B.upload(&d_va, valid_a, (size_t)n_a)) ||
            (mode == 1 && (rc = B.upload(&d_vb, valid_b, (size_t)n_b))) || (rc = B.upload(&d_mb, mB.data(), (size_t)n_b)) ||
            (rc = B.upload(&d_ma, mA.data(), (size_t)n_a)) || (rc = B.upload(&d_mar, mAR.data(), (size_t)n_a)))
            return rc;
        A.mode = mode; A.n_pairs = (int)pairs.size(); A.pairs = d_pairs; A.idx_a = d_ia; A.idx_b = d_ib; A.desc_a = d_da; A.desc_b = d_db;
        A.valid_a = d_va; A.valid_b = d_vb; A.nleft_b = nleft_b; A.nn_ratio = nn_ratio; A.match_b = d_mb; A.match_a = d_ma; A.match_a_right = d_mar;
        cudaError_t e = launch_search_by_bow(A, 0);
        if (e == cudaSuccess) e = cudaMemcpy(mB.data(), d_mb, (size_t)n_b * 4, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(mA.data(), d_ma, (size_t)n_a * 4, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess) e = cudaMemcpy(mAR.data(), d_mar, (size_t)n_a * 4, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "search_by_bow: %s", cudaGetErrorString(e));
    }
    // rotation histogram + ComputeThreeMaxima (src/ORBmatcher1.cc:344-356, 406-427; src/ORBmatcher2.cc:127-139, 152-169).
    // One histogram entry per accepted match; the filter depends on bin sizes only, so the entry order is irrelevant.
    int nm = 0;
    if (mode == 0) { for (int j = 0; j < n_b; ++j) nm += mB[j] >= 0; }
    else { for (int i = 0; i < n_a; ++i) nm += mA[i] >= 0; }
    if (check_orientation) {
        const int H = 30;
        int count[H] = {0};
        std::vector<int> bin(mode == 0 ? n_b : n_a, -1);
        for (int t = 0; t < (int)bin.size(); ++t) {
            const int iA = mode == 0 ? mB[t] : t, jB = mode == 0 ? t : mA[t];
            if (iA < 0 || jB < 0) continue;
            const int b = rotation_bin(angle_a[iA], angle_b[jB]);
            if (b < 0) return fail(ORBX_ERR_INVALID_ARG, "keypoint angles out of range (the reference asserts)");
            bin[t] = b; count[b]++;
        }
        int i1, i2, i3;
        three_maxima(count, H, i1, i2, i3);
        for (int t = 0; t < (int)bin.size(); ++t) {
            if (bin[t] < 0 || bin[t] == i1 || bin[t] == i2 || bin[t] == i3) continue;
            if (mode == 0) { const int iA = mB[t]; mB[t] = -1; if (mA[iA] == t) mA[iA] = -1; if (mAR[iA] == t) mAR[iA] = -1; }
            else { mB[mA[t]] = -1; mA[t] = -1; }
            --nm;
        }
    }
    if (match_a) for (int i = 0; i < n_a; ++i) match_a[i] = mA[i];
    if (match_b) for (int j = 0; j < n_b; ++j) match_b[j] = mB[j];
    *n_matches = nm;
    return ORBX_OK;
}

int orbx_search_for_triangulation(int device, const orbx_keypoint* kp_a, const uint8_t* desc_a, const uint8_t* free_a,
                                  const uint8_t* stereo_a, int n_a, const orbx_feature_vector* fv_a, const orbx_keypoint* kp_b,
                                  const uint8_t* desc_b, const uint8_t* free_b, const uint8_t* stereo_b, int n_b,
                                  const orbx_feature_vector* fv_b, const float* F12, const float* ep, const float* scale_b,
                                  const float* sigma2_b, int n_levels, int only_stereo, int coarse, int check_orientation,
                                  int32_t* match_a, int* n_matches)
{
    if (n_a < 0 || n_b < 0 || !n_matches || !F12 || !ep || !scale_b || !sigma2_b || n_levels < 1 || n_levels > kMaxLevels ||
        (n_a > 0 && (!kp_a || !desc_a || !free_a || !stereo_a || !match_a)) || (n_b > 0 && (!kp_b || !desc_b || !free_b || !stereo_b)))
        return fail(ORBX_ERR_INVALID_ARG, "bad arguments");
    int rc;
    if ((rc = check_fv(fv_a, n_a, "fv_a")) || (rc = check_fv(fv_b, n_b, "fv_b"))) return rc;
    for (int j = 0; j < n_b; ++j)
        if (kp_b[j].octave < 0 || kp_b[j].octave >= n_levels) return fail(ORBX_ERR_INVALID_ARG, "kp_b[%d].octave out of range", j);
    *n_matches = 0;
    std::vector<int32_t> mA(n_a, -1);
    std::vector<std::pair<int, int>> common;
    common_nodes(fv_a, fv_b, common);
    std::vector<int4> jobs;
    for (auto& c : common)
        for (int t = fv_a->offsets[c.first]; t < fv_a->offsets[c.first + 1]; ++t) {
            const int iA = (int)fv_a->indices[t];
            if (!free_a[iA]) continue;                                   // already has a MapPoint (src/ORBmatcher2.cc:246-252)
            if (only_stereo && !stereo_a[iA]) continue;                  // :256-258
            jobs.push_back(make_int4(iA, fv_b->offsets[c.second], fv_b->offsets[c.second + 1], 0));
        }
    if (!jobs.empty() && n_b > 0) {
        if ((rc = set_device(device))) return rc;
        DevBuf B;
        TriSearchArgs A{};
        int4* d_jobs; uint32_t* d_ib; orbx_keypoint *d_ka, *d_kb; uint8_t *d_da, *d_db, *d_sa, *d_sb, *d_fb; int* d_ma;
        if ((rc = B.upload(&d_jobs, jobs.data(), jobs.size())) || (rc = B.upload(&d_ib, fv_b->indices, (size_t)fv_b->offsets[fv_b->n_nodes])) ||
            (rc = B.upload(&d_ka, kp_a, (size_t)n_a)) || (rc = B.upload(&d_kb, kp_b, (size_t)n_b)) || (rc = B.upload(&d_da, desc_a, (size_t)n_a * 32)) ||
            (rc = B.upload(&d_db, desc_b, (size_t)n_b * 32)) || (rc = B.upload(&d_sa, stereo_a, (size_t)n_a)) || (rc = B.upload(&d_sb, stereo_b, (size_t)n_b)) ||
            (rc = B.upload(&d_fb, free_b, (size_t)n_b)) || (rc = B.upload(&d_ma, mA.data(), (size_t)n_a)))
            return rc;
        A.n_jobs = (int)jobs.size(); A.jobs = d_jobs; A.idx_b = d_ib; A.kp_a = d_ka; A.kp_b = d_kb; A.desc_a = d_da; A.desc_b = d_db;
        A.stereo_a = d_sa; A.stereo_b = d_sb; A.free_b = d_fb; A.only_stereo = only_stereo; A.coarse = coarse; A.match_a = d_ma;
        memcpy(A.F12, F12, sizeof A.F12); memcpy(A.ep, ep, sizeof A.ep);
        for (int l = 0; l < n_levels; ++l) { A.scale_b[l] = scale_b[l]; A.sigma2_b[l] = sigma2_b[l]; }
        cudaError_t e = launch_search_triangulation(A, 0);
        if (e == cudaSuccess) e = cudaMemcpy(mA.data(), d_ma, (size_t)n_a * 4, cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "search_for_triangulation: %s", cudaGetErrorString(e));
    }
    int nm = 0;
    for (int i = 0; i < n_a; ++i) nm += mA[i] >= 0;
    if (check_orientation && (rc = tri_rotation_filter(kp_a, kp_b, n_a, mA.data(), &nm))) return rc;
    for (int i = 0; i < n_a; ++i) match_a[i] = mA[i];
    *n_matches = nm;
    return ORBX_OK;
}

int orbx_search_for_triangulation_batch(int device, const orbx_keypoint* kp_a, const uint8_t* desc_a, const uint8_t* free_a,
                                        const uint8_t* stereo_a, int n_a, const orbx_feature_vector* fv_a, int n_kf,
                                        const orbx_triangulation_view* kfs, int only_stereo, int check_orientation, int32_t* match,
                                        int* n_matches)
{
    if (n_kf < 0) return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation_batch: n_kf < 0");
    if (n_kf == 0) return ORBX_OK;
    if (n_kf > 65535) return fail(ORBX_ERR_UNSUPPORTED, "search_for_triangulation_batch: more than 65535 neighbours");
    if (!kfs || !n_matches || n_a < 0 || (n_a > 0 && (!kp_a || !desc_a || !free_a || !stereo_a || !match)))
        return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation_batch: bad arguments");
    int rc;
    if ((rc = check_fv(fv_a, n_a, "fv_a"))) return rc;
    // the single call's checks, per neighbour
    size_t n_feat = 0, n_nodes = 0, n_idx = 0;
    for (int k = 0; k < n_kf; ++k) {
        const orbx_triangulation_view& V = kfs[k];
        if (V.n < 0 || !V.scale || !V.sigma2 || V.n_levels < 1 || V.n_levels > kMaxLevels ||
            (V.n > 0 && (!V.kp || !V.desc || !V.free || !V.stereo)))
            return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation_batch: kfs[%d]: bad arguments", k);
        char name[32];
        snprintf(name, sizeof name, "kfs[%d].fv", k);
        if ((rc = check_fv(&V.fv, V.n, name))) return rc;
        for (int j = 0; j < V.n; ++j)
            if (V.kp[j].octave < 0 || V.kp[j].octave >= V.n_levels)
                return fail(ORBX_ERR_INVALID_ARG, "search_for_triangulation_batch: kfs[%d].kp[%d].octave out of range", k, j);
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
        if (e != cudaSuccess) return fail(ORBX_ERR_CUDA, "search_for_triangulation_batch: %s", cudaGetErrorString(e));
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
