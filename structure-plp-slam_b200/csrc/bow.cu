// bow.cu -- DBoW2 vocabulary tree on the device: transform (data/frame.cc:785-795) and match::bow_tree
// (match/bow_tree.cc:41-305) (sm_100a).
//
// transform: the ORB vocabulary (k = 10, L = 6, 1 082 073 nodes x 32 B = 34.6 MB) stays resident in HBM and, once touched,
// in the 126 MB L2.  A group of G = 16 lanes owns one descriptor: at every level each lane takes one child (two 16-byte
// loads), the group reduces min(distance << 32 | child position) -- "first child with the smallest distance", exactly
// DBoW2's strict-'<' scan -- and steps down.  HBM/L2-latency bound; the batch (frames x 1000 descriptors) hides it.
//
// bow_tree matchers: claims only interact inside one vocabulary node (a keypoint lives in exactly one node of its
// feature vector), so the reference's sequential loop factorises over the nodes shared by the two feature vectors:
// one warp per shared node, sequential over the node's side-1 keypoints, lanes over its side-2 candidates (top-2 by
// (distance, list position)), one CTA per (side-1, side-2) pair so that the orientation histogram is a block reduction.
#include "common.cuh"
#include "pack.cuh"
#include "bow_kernels.cuh"

#include <algorithm>
#include <map>
#include <stdio.h>

struct plp_bow_vocab {
    plp_ctx *ctx = nullptr;
    int k = 0, L = 0, num_nodes = 0, num_words = 0, max_children = 0;
    uint8_t *d_desc = nullptr;          // num_nodes x 32
    uint32_t *d_child_begin = nullptr;  // num_nodes + 1
    uint32_t *d_children = nullptr;     // num_nodes - 1 node ids, grouped by parent, ascending id inside a group
    float *d_weight = nullptr;          // num_nodes
    int32_t *d_word_id = nullptr;       // num_nodes (-1 for inner nodes)
};

namespace plp {

namespace {

static VocabDev vocab_dev(const plp_bow_vocab *v) {
    VocabDev V;
    V.desc = v->d_desc;
    V.child_begin = v->d_child_begin;
    V.children = v->d_children;
    V.weight = v->d_weight;
    V.word_id = v->d_word_id;
    return V;
}

static plp_status launch_transform(plp_bow_vocab *v, const uint8_t *d_desc, int n, int levelsup, int32_t *d_word,
                                   int32_t *d_node, float *d_weight) {
    plp_ctx *ctx = v->ctx;
    const int nid_level = v->L - levelsup;  // <= 0: the root (node id 0)
    const VocabDev V = vocab_dev(v);
    const int G = v->max_children <= 4 ? 4 : v->max_children <= 8 ? 8 : v->max_children <= 16 ? 16 : 32;
    const int groups_per_block = 256 / G;
    const int blocks = div_up(n, groups_per_block);
    switch (G) {
        case 4:
            PLP_LAUNCH(ctx, bow_transform_kernel<4>, blocks, 256, 0, V, d_desc, n, nid_level, d_word, d_node, d_weight);
            break;
        case 8:
            PLP_LAUNCH(ctx, bow_transform_kernel<8>, blocks, 256, 0, V, d_desc, n, nid_level, d_word, d_node, d_weight);
            break;
        case 16:
            PLP_LAUNCH(ctx, bow_transform_kernel<16>, blocks, 256, 0, V, d_desc, n, nid_level, d_word, d_node, d_weight);
            break;
        default:
            PLP_LAUNCH(ctx, bow_transform_kernel<32>, blocks, 256, 0, V, d_desc, n, nid_level, d_word, d_node, d_weight);
            break;
    }
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

}  // namespace

}  // namespace plp

using namespace plp;

extern "C" {

plp_status plp_bow_vocab_create(plp_ctx *ctx, int k, int L, int num_nodes, const int32_t *parent, const uint8_t *desc,
                                const float *weight, const uint8_t *is_leaf, plp_bow_vocab **out) {
    PLP_REQUIRE(ctx && out, "null pointer");
    PLP_REQUIRE(k >= 1 && L >= 1 && num_nodes >= 1, "k / L / num_nodes");
    PLP_REQUIRE(num_nodes == 1 || (parent && desc && weight && is_leaf), "node arrays");
    *out = nullptr;
    const size_t N = (size_t)num_nodes;
    // CSR children lists: children of a node in ascending id = the order of m_nodes[parent].children.push_back(n_id)
    std::vector<uint32_t> child_begin(N + 1, 0), children(N > 1 ? N - 1 : 1, 0);
    for (size_t id = 1; id < N; ++id) {
        const int32_t p = parent[id - 1];
        if (p < 0 || (size_t)p >= id) {
            set_error("vocabulary: node %zu has parent %d (parents must precede their children)", id, p);
            return PLP_ERR_INVALID;
        }
        child_begin[(size_t)p + 1]++;
    }
    int max_children = 0;
    for (size_t i = 0; i < N; ++i) {
        max_children = std::max(max_children, (int)child_begin[i + 1]);
        child_begin[i + 1] += child_begin[i];
    }
    std::vector<uint32_t> fill(child_begin.begin(), child_begin.end() - 1);
    for (size_t id = 1; id < N; ++id) children[fill[(size_t)parent[id - 1]]++] = (uint32_t)id;
    std::vector<int32_t> word_id(N, -1);
    std::vector<float> w(N, 0.0f);
    std::vector<uint8_t> dsc(N * 32, 0);
    int num_words = 0;
    for (size_t id = 1; id < N; ++id) {
        const bool has_children = child_begin[id + 1] > child_begin[id];
        if ((is_leaf[id - 1] != 0) == has_children) {
            set_error("vocabulary: node %zu is flagged %s but has %s children", id, is_leaf[id - 1] ? "leaf" : "inner",
                      has_children ? "some" : "no");
            return PLP_ERR_INVALID;
        }
        if (is_leaf[id - 1]) word_id[id] = num_words++;  // words are numbered in file order
        w[id] = weight[id - 1];
        memcpy(&dsc[32 * id], desc + 32 * (id - 1), 32);
    }
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    plp_bow_vocab *v = new plp_bow_vocab;
    v->ctx = ctx;
    v->k = k;
    v->L = L;
    v->num_nodes = num_nodes;
    v->num_words = num_words;
    v->max_children = max_children;
    cudaError_t e = cudaSuccess;
    auto up = [&](void **dst, const void *src, size_t bytes) {
        if (e != cudaSuccess) return;
        e = cudaMalloc(dst, bytes ? bytes : 4);
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
    };
    up((void **)&v->d_desc, dsc.data(), N * 32);
    up((void **)&v->d_child_begin, child_begin.data(), (N + 1) * 4);
    up((void **)&v->d_children, children.data(), (N - 1) * 4);
    up((void **)&v->d_weight, w.data(), N * 4);
    up((void **)&v->d_word_id, word_id.data(), N * 4);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);  // the staging vectors die with this scope
    if (e != cudaSuccess) {
        set_error("vocabulary upload failed: %s", cudaGetErrorString(e));
        plp_bow_vocab_destroy(v);
        return PLP_ERR_CUDA;
    }
    *out = v;
    return PLP_OK;
}

plp_status plp_bow_vocab_load(plp_ctx *ctx, const char *path, plp_bow_vocab **out) {
    PLP_REQUIRE(ctx && path && out, "null pointer");
    *out = nullptr;
    FILE *f = fopen(path, "rb");
    if (!f) {
        set_error("vocabulary: cannot open %s", path);
        return PLP_ERR_INVALID;
    }
    uint32_t n_nodes = 0, node_size = 0;
    int32_t k = 0, L = 0, scoring = 0, weighting = 0;
    bool ok = fread(&n_nodes, 4, 1, f) == 1 && fread(&node_size, 4, 1, f) == 1 && fread(&k, 4, 1, f) == 1 &&
              fread(&L, 4, 1, f) == 1 && fread(&scoring, 4, 1, f) == 1 && fread(&weighting, 4, 1, f) == 1;
    if (!ok || node_size != 41 || n_nodes < 1 || n_nodes > (1u << 30)) {
        fclose(f);
        set_error("vocabulary: %s is not a DBoW2 binary vocabulary (node_size %u)", path, node_size);
        return PLP_ERR_INVALID;
    }
    if (scoring != 0 || weighting != 0) {  // L1_NORM / TF_IDF are what the shipped vocabulary and the adapter's fold use
        fclose(f);
        set_error("vocabulary: unsupported scoring %d / weighting %d (L1_NORM + TF_IDF expected)", scoring, weighting);
        return PLP_ERR_INVALID;
    }
    const size_t cnt = n_nodes - 1;
    std::vector<uint8_t> raw(cnt * 41 + 1);
    ok = fread(raw.data(), 41, cnt, f) == cnt;
    fclose(f);
    if (!ok) {
        set_error("vocabulary: %s is truncated (%u nodes announced)", path, n_nodes);
        return PLP_ERR_INVALID;
    }
    std::vector<int32_t> parent(cnt);
    std::vector<uint8_t> desc(cnt * 32 + 1), leaf(cnt + 1);
    std::vector<float> weight(cnt + 1);
    for (size_t i = 0; i < cnt; ++i) {
        const uint8_t *r = raw.data() + 41 * i;
        memcpy(&parent[i], r, 4);
        memcpy(&desc[32 * i], r + 4, 32);
        memcpy(&weight[i], r + 36, 4);
        leaf[i] = r[40];
    }
    return plp_bow_vocab_create(ctx, k, L, (int)n_nodes, parent.data(), desc.data(), weight.data(), leaf.data(), out);
}

void plp_bow_vocab_destroy(plp_bow_vocab *v) {
    if (!v) return;
    cudaSetDevice(v->ctx->device);
    cudaFree(v->d_desc);
    cudaFree(v->d_child_begin);
    cudaFree(v->d_children);
    cudaFree(v->d_weight);
    cudaFree(v->d_word_id);
    delete v;
}

plp_status plp_bow_vocab_info(const plp_bow_vocab *v, int32_t *k, int32_t *L, int32_t *num_nodes, int32_t *num_words) {
    PLP_REQUIRE(v, "null pointer");
    if (k) *k = v->k;
    if (L) *L = v->L;
    if (num_nodes) *num_nodes = v->num_nodes;
    if (num_words) *num_words = v->num_words;
    return PLP_OK;
}

plp_status plp_bow_transform_dev(plp_bow_vocab *v, const uint8_t *d_desc, int n, int levelsup, int32_t *d_word_id_out,
                                 int32_t *d_node_id_out, float *d_weight_out) {
    PLP_REQUIRE(v && n >= 0, "vocab / n");
    if (n == 0) return PLP_OK;
    PLP_REQUIRE(d_desc && d_word_id_out && d_node_id_out && d_weight_out, "null pointer");
    PLP_CUDA_TRY(cudaSetDevice(v->ctx->device));
    return launch_transform(v, d_desc, n, levelsup, d_word_id_out, d_node_id_out, d_weight_out);
}

plp_status plp_bow_transform(plp_bow_vocab *v, const uint8_t *desc, int n, int levelsup, int32_t *word_id_out,
                             int32_t *node_id_out, float *weight_out) {
    PLP_REQUIRE(v && n >= 0, "vocab / n");
    if (n == 0) return PLP_OK;
    PLP_REQUIRE(desc && word_id_out && node_id_out && weight_out, "null pointer");
    plp_ctx *ctx = v->ctx;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const uint8_t *dd;
    int32_t *dw, *dn;
    float *df;
    lay.in(dd, desc, (size_t)n * 32);
    lay.out(dw, n);
    lay.out(dn, n);
    lay.out(df, n);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_transform(v, dd, n, levelsup, dw, dn, df));
    PLP_CUDA_TRY(cudaMemcpyAsync(word_id_out, dw, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(node_id_out, dn, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(weight_out, df, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

plp_status plp_match_bow_tree(plp_ctx *ctx, plp_bow_pair *pairs, int num_pairs, float lowe_ratio, int check_orientation) {
    PLP_REQUIRE(ctx && num_pairs >= 0, "ctx / num_pairs");
    if (num_pairs == 0) return PLP_OK;
    PLP_REQUIRE(pairs, "pairs");
    struct Side {
        std::vector<uint32_t> flat;  // validated copy of fv.indices
        const uint8_t *desc;
        const float *angle;
        const uint8_t *valid;
        const uint32_t *idx;
    };
    std::map<const plp_bow_side *, Side> sides;
    Layout lay;
    // validate + pack every distinct side once
    for (int p = 0; p < num_pairs; ++p) {
        pairs[p].num_matches = 0;
        PLP_REQUIRE(pairs[p].side1 && pairs[p].side2, "pair sides");
        for (const plp_bow_side *s : {pairs[p].side1, pairs[p].side2}) {
            if (sides.count(s)) continue;
            PLP_REQUIRE(s->n >= 0 && s->fv.num_nodes >= 0, "side sizes");
            PLP_REQUIRE(s->n == 0 || s->desc, "side descriptors");
            PLP_REQUIRE(s->fv.num_nodes == 0 || (s->fv.node_ids && s->fv.offsets && s->fv.indices), "feature vector");
            PLP_REQUIRE(!check_orientation || s->n == 0 || s->angle, "angles required for the orientation check");
            Side so;
            const int total = s->fv.num_nodes ? s->fv.offsets[s->fv.num_nodes] : 0;
            std::vector<uint8_t> seen((size_t)s->n, 0);
            for (int a = 0; a < s->fv.num_nodes; ++a) {
                PLP_REQUIRE(s->fv.offsets[a] <= s->fv.offsets[a + 1], "feature vector offsets must ascend");
                PLP_REQUIRE(a == 0 || s->fv.node_ids[a - 1] < s->fv.node_ids[a], "feature vector node ids must ascend");
            }
            so.flat.assign(s->fv.indices, s->fv.indices + total);
            for (uint32_t i : so.flat) {
                PLP_REQUIRE(i < (uint32_t)s->n, "feature vector index out of range");
                PLP_REQUIRE(!seen[i], "a keypoint appears in two nodes of a feature vector");
                seen[i] = 1;
            }
            sides.emplace(s, std::move(so));
        }
    }
    for (auto &kv : sides) {
        const plp_bow_side *s = kv.first;
        Side &so = kv.second;
        const size_t n = (size_t)s->n;
        lay.in(so.desc, s->desc, n * 32);
        lay.in(so.angle, s->angle, n);
        lay.in(so.valid, s->valid, n);
        lay.in(so.idx, so.flat.data(), so.flat.size());
    }
    // merge-join of the two ascending feature vectors per pair (bow_tree.cc:60-150): the shared nodes
    struct Shared {
        std::vector<int32_t> nb1, ne1, nb2, ne2;
    };
    std::vector<Shared> sh(num_pairs);
    std::vector<BowJob> jobs(num_pairs);
    for (int p = 0; p < num_pairs; ++p) {
        const plp_bow_feature_vector &f1 = pairs[p].side1->fv, &f2 = pairs[p].side2->fv;
        int a = 0, b = 0;
        while (a < f1.num_nodes && b < f2.num_nodes) {
            if (f1.node_ids[a] == f2.node_ids[b]) {
                sh[p].nb1.push_back(f1.offsets[a]);
                sh[p].ne1.push_back(f1.offsets[a + 1]);
                sh[p].nb2.push_back(f2.offsets[b]);
                sh[p].ne2.push_back(f2.offsets[b + 1]);
                ++a;
                ++b;
            } else if (f1.node_ids[a] < f2.node_ids[b]) {
                ++a;  // lower_bound on an ascending map
            } else {
                ++b;
            }
        }
        BowJob &J = jobs[p];
        const Side &s1 = sides[pairs[p].side1], &s2 = sides[pairs[p].side2];
        const size_t nn = sh[p].nb1.size();
        J.n1 = pairs[p].side1->n;
        J.n2 = pairs[p].side2->n;
        J.num_nodes = (int)nn;
        lay.alias(J.desc1, s1.desc);
        lay.alias(J.desc2, s2.desc);
        lay.alias(J.angle1, s1.angle);
        lay.alias(J.angle2, s2.angle);
        lay.alias(J.valid1, s1.valid);
        lay.alias(J.valid2, s2.valid);
        lay.alias(J.idx1, s1.idx);
        lay.alias(J.idx2, s2.idx);
        lay.in(J.nb1, sh[p].nb1.data(), nn);
        lay.in(J.ne1, sh[p].ne1.data(), nn);
        lay.in(J.nb2, sh[p].nb2.data(), nn);
        lay.in(J.ne2, sh[p].ne2.data(), nn);
        lay.out(J.claimed, (size_t)J.n2 + 1);
        lay.out(J.choice, (size_t)J.n1 + 1);
    }
    const BowJob *d_jobs;
    lay.in(d_jobs, jobs.data(), num_pairs);
    // all results in ONE contiguous region -> one D2H copy (a copy per pair and array costs more than the kernel)
    for (BowJob &J : jobs) {
        lay.out(J.matched_2_of_1, (size_t)J.n1 + 1);
        lay.out(J.matched_1_of_2, (size_t)J.n2 + 1);
        lay.out(J.num_matches, 1);
    }
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    PLP_TRY(lay.upload(ctx, 0));
    PLP_LAUNCH(ctx, bow_match_kernel, num_pairs, kMatchThreads, 0, d_jobs, lowe_ratio, check_orientation);
    PLP_CHECK_LAUNCH();
    uint8_t *r0 = (uint8_t *)jobs[0].matched_2_of_1, *r1 = (uint8_t *)(jobs[num_pairs - 1].num_matches + 1);
    PLP_CUDA_TRY(cudaMemcpyAsync(lay.staged(r0), r0, r1 - r0, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    std::vector<uint32_t> nums(num_pairs, 0);
    for (int p = 0; p < num_pairs; ++p) {
        const BowJob &J = jobs[p];
        if (pairs[p].matched_2_of_1_out && J.n1)
            memcpy(pairs[p].matched_2_of_1_out, lay.staged(J.matched_2_of_1), (size_t)J.n1 * 4);
        if (pairs[p].matched_1_of_2_out && J.n2)
            memcpy(pairs[p].matched_1_of_2_out, lay.staged(J.matched_1_of_2), (size_t)J.n2 * 4);
        nums[p] = *lay.staged(J.num_matches);
    }
    for (int p = 0; p < num_pairs; ++p) pairs[p].num_matches = nums[p];
    return PLP_OK;
}

}  // extern "C"
