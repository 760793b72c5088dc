// bow_kernels.cuh -- device code of the DBoW2 transform and of match::bow_tree (bow.cu launches it).  Free of host-side
// CUDA runtime dependencies so that tests/cta_emu can compile the same text for the host.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "../../include/plpslam_b200.h"
#include "devmath.cuh"
#include "match_device.cuh"

namespace plp {

namespace {

constexpr int kMatchThreads = 256;

struct VocabDev {
    const uint8_t *desc;
    const uint32_t *child_begin;
    const uint32_t *children;
    const float *weight;
    const int32_t *word_id;
};

// TemplatedVocabulary::transform(feature, word_id, weight, &nid, levelsup)
template <int G>
__global__ void __launch_bounds__(256) bow_transform_kernel(VocabDev V, const uint8_t *__restrict__ desc, int n,
                                                            int nid_level, int32_t *__restrict__ word_out,
                                                            int32_t *__restrict__ node_out, float *__restrict__ weight_out) {
    const int gid = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) / G);
    const int gl = (int)(threadIdx.x % G);
    const int row = min(gid, n - 1);  // surplus groups shadow the last row (shuffles need every lane) and do not store
    uint4 q0, q1;
    load_desc(desc + 32 * (size_t)row, q0, q1);
    int final_id = 0, nid = 0, level = 0;
    uint32_t beg = V.child_begin[0], end = V.child_begin[1];
    const bool empty_vocab = beg == end;
    while (__any_sync(0xffffffffu, beg < end)) {
        unsigned long long best = ~0ull;
        for (uint32_t c = beg + gl; c < end; c += G) {
            const uint32_t child = V.children[c];
            uint4 d0, d1;
            load_desc(V.desc + 32 * (size_t)child, d0, d1);
            const unsigned long long key = ((unsigned long long)(unsigned)hamming256(q0, q1, d0, d1) << 32) | (c - beg);
            best = key < best ? key : best;
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) {
            const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
            best = other < best ? other : best;
        }
        if (beg < end) {
            ++level;
            final_id = (int)V.children[beg + (uint32_t)(best & 0xffffffffull)];
            if (level == nid_level) nid = final_id;
            beg = V.child_begin[final_id];
            end = V.child_begin[final_id + 1];
        }
    }
    if (gl == 0 && gid < n) {
        word_out[gid] = empty_vocab ? -1 : V.word_id[final_id];
        node_out[gid] = nid;
        weight_out[gid] = empty_vocab ? 0.0f : V.weight[final_id];
    }
}

// ---------------------------------------------------------------------------------------------------------------
// match::bow_tree
// ---------------------------------------------------------------------------------------------------------------
struct BowJob {
    int n1, n2, num_nodes;
    const uint8_t *desc1, *desc2;
    const float *angle1, *angle2;    // may be null
    const uint8_t *valid1, *valid2;  // may be null
    const uint32_t *idx1, *idx2;     // flattened feature-vector index lists
    const int32_t *nb1, *ne1, *nb2, *ne2;  // per shared node: spans in idx1 / idx2
    uint8_t *claimed;                // n2
    int32_t *choice;                 // n1
    int32_t *matched_2_of_1;         // n1
    int32_t *matched_1_of_2;         // n2
    uint32_t *num_matches;
};

__global__ void __launch_bounds__(kMatchThreads) bow_match_kernel(const BowJob *__restrict__ jobs, float lowe_ratio,
                                                                  int check_orientation) {
    __shared__ int s_hist[kHistLen + 2];
    __shared__ uint8_t s_bin_valid[kHistLen + 2];
    __shared__ int s_cnt[2];
    const BowJob &J = jobs[blockIdx.x];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kMatchThreads / 32;
    volatile uint8_t *claimed = J.claimed;
    for (int i = tid; i < J.n1; i += kMatchThreads) J.choice[i] = -1;
    for (int j = tid; j < J.n2; j += kMatchThreads) {
        J.claimed[j] = 0;
        J.matched_1_of_2[j] = -1;
    }
    __syncthreads();
    for (int node = warp; node < J.num_nodes; node += nwarps) {
        const int b1 = J.nb1[node], e1 = J.ne1[node], b2 = J.nb2[node], e2 = J.ne2[node];
        for (int a = b1; a < e1; ++a) {  // bow_tree.cc:67 / :216 -- sequential: later keypoints see earlier claims
            const int i1 = (int)J.idx1[a];
            if (J.valid1 && !J.valid1[i1]) continue;
            uint4 q0, q1;
            load_desc(J.desc1 + 32 * (size_t)i1, q0, q1);
            unsigned long long k1 = ~0ull, k2 = ~0ull;
            for (int c = b2 + lane; c < e2; c += 32) {
                const int j = (int)J.idx2[c];
                if (J.valid2 && !J.valid2[j]) continue;
                if (claimed[j]) continue;
                uint4 d0, d1;
                load_desc(J.desc2 + 32 * (size_t)j, d0, d1);
                const unsigned d = (unsigned)hamming256(q0, q1, d0, d1);
                if (d >= (unsigned)PLP_MAX_HAMMING_DIST) continue;  // can replace neither best nor second (both start at 256)
                const unsigned long long key = ((unsigned long long)d << 32) | (unsigned)(c - b2);
                if (key < k1) {
                    k2 = k1;
                    k1 = key;
                } else if (key < k2) {
                    k2 = key;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long o1 = __shfl_xor_sync(0xffffffffu, k1, o);
                const unsigned long long o2 = __shfl_xor_sync(0xffffffffu, k2, o);
                const unsigned long long lo = k1 < o1 ? k1 : o1, hi = k1 < o1 ? o1 : k1;
                const unsigned long long s2 = k2 < o2 ? k2 : o2;
                k1 = lo;
                k2 = hi < s2 ? hi : s2;
            }
            if (k1 != ~0ull) {
                const unsigned best = (unsigned)(k1 >> 32);
                const unsigned second = k2 != ~0ull ? (unsigned)(k2 >> 32) : (unsigned)PLP_MAX_HAMMING_DIST;
                // :110-119
                if (!((unsigned)PLP_HAMMING_DIST_THR_LOW < best) && !(lowe_ratio * (float)second < (float)best)) {
                    if (lane == 0) {
                        const int j = (int)J.idx2[b2 + (int)(k1 & 0xffffffffull)];
                        claimed[j] = 1;
                        J.choice[i1] = j;
                    }
                }
            }
            __syncwarp();
        }
    }
    // orientation histogram (:123-127, :152-160) and outputs
    const bool do_angle = check_orientation && J.angle1 && J.angle2;
    orientation_filter<kMatchThreads>(
        J.n1, J.choice, do_angle, s_hist, s_bin_valid, s_cnt, J.num_matches,
        [&](int i, int j) { return J.angle1[i] - J.angle2[j]; },
        [&](int i, int j, bool keep) {
            if (keep) J.matched_1_of_2[j] = i;
            J.matched_2_of_1[i] = keep ? j : -1;
        });
}

}  // namespace

}  // namespace plp
