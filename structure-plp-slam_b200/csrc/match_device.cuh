// match_device.cuh -- device building blocks shared by the greedy Hamming matchers (match.cu, point_match_kernels.cuh,
// bow_kernels.cuh): the reference's orientation check (angle_checker.h) and the claim rounds that run its sequential
// "skip candidates claimed by an earlier query" in parallel.  Both must agree with the oracle bit for bit.  Free of
// host-side CUDA runtime dependencies so that tests/cta_emu can compile the same text for the host.
#pragma once
#include <stdint.h>

#include "devmath.cuh"

namespace plp {

constexpr int kHistLen = 30;     // angle_checker.h:47
constexpr int kNumBinsThr = 3;   // angle_checker.h:48
constexpr int kNoOwner = 0x7fffffff;

// angle_checker.h:100-113
__device__ __forceinline__ int angle_bin(float delta_angle) {
    if (delta_angle < 0.0) delta_angle = (float)((double)delta_angle + 360.0);
    if (360.0 <= delta_angle) delta_angle = (float)((double)delta_angle - 360.0);
    const float inv_len = 1.0f / (float)kHistLen;
    return __float2int_rn(delta_angle * inv_len);
}

// angle_checker.h:163-175: rank bins by size (desc), ties by bin index (asc); first 3 are valid.  One thread.
__device__ inline void rank_bins(const int *hist, uint8_t *bin_valid) {
    bool used[kHistLen];
    for (int b = 0; b < kHistLen; ++b) {
        used[b] = false;
        bin_valid[b] = 0;
    }
    for (int k = 0; k < kNumBinsThr; ++k) {
        int best = -1, best_cnt = -1;
        for (int b = 0; b < kHistLen; ++b)
            if (!used[b] && hist[b] > best_cnt) {
                best_cnt = hist[b];
                best = b;
            }
        used[best] = true;
        bin_valid[best] = 1;
    }
}

// The orientation check of a matcher's result, run by the whole CTA: choice[q] (< 0: unmatched) is the candidate of
// query q, delta(q, c) the angle difference in the reference's operand order for that matcher.  With do_angle, a choice
// is kept only if its angle bin is among the three fullest.  emit(q, c, keep) is called once per query and writes the
// matcher's outputs; *num_matches (if not null) = accepted - rejected.  hist (kHistLen), bin_valid (kHistLen) and cnt (2)
// are shared memory that the filter clears itself.  Four barriers, the first one right after the clearing.
// num_matches is a reference to the job's field so that the pointer is loaded only for the final store: a copy would stay
// live through rank_bins and costs the window matcher 8 registers.
template <int kThreads, class Delta, class Emit>
__device__ __forceinline__ void orientation_filter(int m, const int32_t *choice, bool do_angle, int *hist,
                                                   uint8_t *bin_valid, int *cnt, uint32_t *const &num_matches,
                                                   Delta delta, Emit emit) {
    const int tid = threadIdx.x;
    for (int b = tid; b < kHistLen; b += kThreads) hist[b] = 0;
    if (tid < 2) cnt[tid] = 0;
    __syncthreads();
    for (int q = tid; q < m; q += kThreads) {
        const int c = choice[q];
        if (c < 0) continue;
        atomicAdd(&cnt[0], 1);
        if (do_angle) atomicAdd(&hist[angle_bin(delta(q, c))], 1);
    }
    __syncthreads();
    if (tid == 0 && do_angle) rank_bins(hist, bin_valid);
    __syncthreads();
    for (int q = tid; q < m; q += kThreads) {
        const int c = choice[q];
        bool keep = c >= 0;
        if (keep && do_angle) {
            keep = bin_valid[angle_bin(delta(q, c))] != 0;
            if (!keep) atomicAdd(&cnt[1], 1);
        }
        emit(q, c, keep);
    }
    __syncthreads();
    if (tid == 0 && num_matches) *num_matches = (uint32_t)(cnt[0] - cnt[1]);
}

struct NoChange {
    __device__ void operator()(int) const {}
};

// The reference's matchers serve queries in order and skip candidates claimed by an earlier query.  In parallel, every
// round each query rescans, skipping candidates `owned_before` it in the previous round, and `claim`s its choice for the
// next; the smallest claiming query owns a candidate.  Query q depends only on queries < q, so after round r the first r
// queries are final, and the fixed point (a round that changes no owner) is the sequential result.  prev / next (n
// entries each) and the flag `changed` are shared memory; the CTA calls every member together.
template <int kThreads>
struct ClaimRounds {
    int *prev, *next;  // owner of each candidate in the previous / current round
    int *changed;
    int n;

    __device__ __forceinline__ void reset(int tid) {
        for (int c = tid; c < n; c += kThreads) {
            prev[c] = kNoOwner;
            next[c] = kNoOwner;
        }
        if (tid == 0) *changed = 0;
    }
    __device__ __forceinline__ bool owned_before(int c, int q) const { return prev[c] < q; }
    __device__ __forceinline__ void claim(int c, int q) { atomicMin(&next[c], q); }

    // After every query of the round has claimed: true at the fixed point, else the owners move on to the next round.
    // on_change(c) is called for each candidate whose owner changed.
    template <class OnChange = NoChange>
    __device__ __forceinline__ bool settled(int tid, OnChange on_change = OnChange()) {
        __syncthreads();
        for (int c = tid; c < n; c += kThreads)
            if (next[c] != prev[c]) {
                *changed = 1;
                on_change(c);
            }
        __syncthreads();
        const int any = *changed;
        __syncthreads();
        if (!any) return true;
        if (tid == 0) *changed = 0;
        int *t = prev;
        prev = next;
        next = t;
        for (int c = tid; c < n; c += kThreads) next[c] = kNoOwner;
        __syncthreads();
        return false;
    }
};

}  // namespace plp
