// point_match_kernels.cuh -- device code of the window matcher over the 64 x 48 keypoint grid (match.cu launches it):
// projection::match_frame_and_landmarks (match/projection.cc:37-121), the matching stage of
// match_current_and_last_frames (:294-335) and match_frame_and_keyframe (:584-640), with the grid helpers
// data/common.cc:205-313.  Free of host-side CUDA runtime dependencies so that tests/cta_emu can compile the same text
// for the host.
//
// One CTA (1024 threads) per frame.
//   1-3  stable counting sort of the keypoints by (cell_x, cell_y, index) -- exactly the traversal order of
//        get_keypoints_in_cell (data/common.cc:275-309): cell histogram (shared-memory atomics), block-wide exclusive scan,
//        scatter with per-cell cursors (any order), then every cell is put back into index order by one thread (cells hold
//        ~0.4 keypoints on average, 10 x 10 px) -- O(n), replaces the O(n^2) rank sort;
//   4    the reference's sequential greedy ("skip keypoints claimed by an earlier query") as a fixed point, see below;
//        a GROUP of kGroup lanes owns one query: the lanes take the grid columns of the query window round-robin (a
//        column's cells [min_cy, max_cy] are one contiguous span of the sorted arrays) and scan their spans
//        sequentially, keeping the two smallest keys  key = distance << 12 | sorted position  -- top-2 by (distance,
//        traversal order) is exactly the reference's strict-'<' scan -- merged over the group by log2(kGroup) shuffles.
//        (The first generation used one WARP per query: windows hold 10-40 candidates spread over 5-15 columns with
//        ~2 candidates each, so 30 of 32 lanes idled through every column iteration.)
//   5    orientation histogram (angle_checker.h:86-175) and outputs.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "../../include/plpslam_b200.h"
#include "devmath.cuh"
#include "match_device.cuh"
#include "match_jobs.h"

namespace plp {

namespace pm {

constexpr int kThreads = 1024;
constexpr int kGroup = 4;        // lanes per query
constexpr int kNoKey = 0x7fffffff;

struct PointSmem {
    uint4 *desc;     // 2 per keypoint, sorted order
    float *x, *y, *xr;
    int *meta;       // octave (bits 0-7, signed) | cell_y (8-15) | claimed (16) | cell_x (17..)
    int *orig;       // original index of the keypoint at each sorted position
    int *owner_a, *owner_b;
    int *col_start;  // cell start table: num_cols * num_rows + 2
    int *cursor;     // scatter cursors of the counting sort: num_cols * num_rows + 2
    int *hist;       // kHistLen
    int *flags;      // [0] changed, [1] num accepted, [2] num invalid, [3] spare
    int *warp_sums;  // 32
    uint8_t *bin_valid;
    uint8_t *colchg;  // per grid column: did an owner change there in the last round?
};

__device__ __forceinline__ PointSmem carve_point_smem(uint8_t *base, int cap, int num_cols, int num_rows) {
    PointSmem s;
    const size_t cells2 = (size_t)(num_cols * num_rows + 2);
    s.desc = reinterpret_cast<uint4 *>(base);
    base += (size_t)cap * 32;
    s.x = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    s.y = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    s.xr = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    s.meta = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    s.orig = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    s.owner_a = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    s.owner_b = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    s.col_start = reinterpret_cast<int *>(base);
    base += cells2 * 4;
    s.cursor = reinterpret_cast<int *>(base);
    base += cells2 * 4;
    s.hist = reinterpret_cast<int *>(base);
    base += kHistLen * 4;
    s.flags = reinterpret_cast<int *>(base);
    base += 4 * 4;
    s.warp_sums = reinterpret_cast<int *>(base);
    base += 32 * 4;
    s.bin_valid = base;
    s.colchg = base + 32;
    return s;
}

static inline size_t point_smem_bytes(int cap, int num_cols, int num_rows) {
    return (size_t)cap * (32 + 7 * 4) + (size_t)(num_cols * num_rows + 2) * 8 + kHistLen * 4 + 16 + 128 + 32 +
           (size_t)(num_cols + 16);
}

// the window of query q in grid cells (data/common.cc:249-272); false if it misses the grid
struct Window {
    int min_cx, max_cx, min_cy, max_cy;
};
__device__ __forceinline__ bool query_window(const plp_grid &grid, float ref_x, float ref_y, float r, Window &w) {
    w.min_cx = max(0, cv_floor((double)(ref_x - grid.min_x - r) * grid.inv_cell_width));
    w.max_cx = min(grid.num_cols - 1, cv_ceil((double)(ref_x - grid.min_x + r) * grid.inv_cell_width));
    w.min_cy = max(0, cv_floor((double)(ref_y - grid.min_y - r) * grid.inv_cell_height));
    w.max_cy = min(grid.num_rows - 1, cv_ceil((double)(ref_y - grid.min_y + r) * grid.inv_cell_height));
    return w.min_cx < grid.num_cols && w.max_cx >= 0 && w.min_cy < grid.num_rows && w.max_cy >= 0;
}

// Top-2 keys of query q over its window, computed by the kGroup lanes of a group (all lanes of the WARP must call it
// together: the merge uses shuffles).  `active` = this group has a query to scan; `owner` (may be null): skip candidates
// owned by a smaller query; `floor`: only keys strictly greater (-1 = none).
__device__ __forceinline__ void group_scan(const PointSmem &S, const PointMatchJob &J, const plp_grid &grid, bool active,
                                           int q, int gl, const int *owner, int floor, int &k1, int &k2) {
    k1 = kNoKey;
    k2 = kNoKey;
    if (active) {
        const float ref_x = J.qx[q], ref_y = J.qy[q], r = J.qradius[q];
        const int min_level = J.qmin[q], max_level = J.qmax[q];
        Window w;
        if (query_window(grid, ref_x, ref_y, r, w)) {
            const bool check_level = (0 < min_level) || (0 <= max_level);
            const float qxr = J.qxr ? J.qxr[q] : 0.0f;
            uint4 q0, q1;
            load_desc(J.qdesc + 32 * (size_t)q, q0, q1);
            for (int c = w.min_cx + gl; c <= w.max_cx; c += kGroup) {
                const int p_begin = S.col_start[c * grid.num_rows + w.min_cy];
                const int p_end = S.col_start[c * grid.num_rows + w.max_cy + 1];
                for (int p = p_begin; p < p_end; ++p) {
                    const int meta = S.meta[p];
                    const int oct = (int)(signed char)(meta & 0xff);
                    if (check_level) {
                        if (oct < min_level) continue;
                        if (0 <= max_level && max_level < oct) continue;
                    }
                    const float dx = S.x[p] - ref_x, dy = S.y[p] - ref_y;
                    if (!(fabsf(dx) < r && fabsf(dy) < r)) continue;
                    if ((meta >> 16) & 1) continue;       // already has a landmark with observations
                    if (owner && owner[p] < q) continue;  // claimed by an earlier query
                    const float xr = S.xr[p];
                    if (0 < xr) {  // projection.cc:76-83 / 310-317
                        const float err = fabsf(qxr - xr);
                        if (r < err) continue;
                    }
                    const int d = hamming256(q0, q1, S.desc[2 * p], S.desc[2 * p + 1]);
                    if (d >= PLP_MAX_HAMMING_DIST) continue;  // can never replace the initial best / second
                    const int key = (d << 12) | p;
                    if (key <= floor) continue;
                    if (key < k1) {
                        k2 = k1;
                        k1 = key;
                    } else if (key < k2) {
                        k2 = key;
                    }
                }
            }
        }
    }
#pragma unroll
    for (int o = kGroup / 2; o > 0; o >>= 1) {
        const int o1 = __shfl_xor_sync(0xffffffffu, k1, o);
        const int o2 = __shfl_xor_sync(0xffffffffu, k2, o);
        const int lo = k1 < o1 ? k1 : o1, hi = k1 < o1 ? o1 : k1;
        const int s2 = k2 < o2 ? k2 : o2;
        k1 = lo;
        k2 = hi < s2 ? hi : s2;
    }
}

__device__ __forceinline__ bool group_any(bool v) {
    int x = v ? 1 : 0;
#pragma unroll
    for (int o = kGroup / 2; o > 0; o >>= 1) x |= __shfl_xor_sync(0xffffffffu, x, o);
    return x != 0;
}

__global__ void __launch_bounds__(kThreads, 1)
    point_match_kernel(const PointMatchJob *__restrict__ jobs, plp_grid grid, int cap, int ratio_test, float lowe_ratio,
                       int check_orientation) {
    PLP_DYNAMIC_SMEM(smem_raw);
    const PointMatchJob &J = jobs[blockIdx.x];
    if (J.m < 0) return;  // job disabled (e.g. the widened-margin retry is not needed for this frame)
    PointSmem S = carve_point_smem(smem_raw, cap, grid.num_cols, grid.num_rows);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kThreads / 32;
    if (J.n > cap) {  // more keypoints than the shared-memory tables hold: report "no matches" loudly (0xffffffff)
        if (J.matched_out)
            for (int i = tid; i < J.n; i += kThreads) J.matched_out[i] = -1;
        if (J.best_idx_out)
            for (int q = tid; q < J.m; q += kThreads) J.best_idx_out[q] = -1;
        if (tid == 0 && J.num_matches) *J.num_matches = 0xffffffffu;
        return;
    }
    const int n = J.n, m = J.m;
    const int cells = grid.num_cols * grid.num_rows;

    // ---- 1. cell key of every keypoint (data/common.h:104-109) and the cell histogram; owner_a doubles as key buffer
    int *key = S.owner_a;
    for (int k = tid; k < cells + 2; k += kThreads) S.col_start[k] = 0;
    if (tid < 4) S.flags[tid] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        const float px = J.x[i], py = J.y[i];
        const int cx = cv_floor((double)(px - grid.min_x) * grid.inv_cell_width);
        const int cy = cv_floor((double)(py - grid.min_y) * grid.inv_cell_height);
        const bool in = (0 <= cx && cx < grid.num_cols && 0 <= cy && cy < grid.num_rows);
        const int k = in ? cx * grid.num_rows + cy : cells;  // out-of-grid keypoints sort last and are never visited
        key[i] = k;
        atomicAdd(&S.col_start[k], 1);
    }
    __syncthreads();
    // ---- 2. exclusive scan of the histogram: col_start[k] = first sorted position whose cell key >= k
    //         (k = cell_x * num_rows + cell_y), so the cells [min_cy, max_cy] of one grid column are ONE contiguous span
    {
        const int total = cells + 1;  // keys 0 .. cells
        const int per = (total + kThreads - 1) / kThreads;
        const int b0 = min(total, tid * per), b1 = min(total, b0 + per);
        int sum = 0;
        for (int k = b0; k < b1; ++k) sum += S.col_start[k];
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) S.warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int v = lane < nwarps ? S.warp_sums[lane] : 0;
            int sc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, sc, o);
                if (lane >= o) sc += u;
            }
            if (lane < nwarps) S.warp_sums[lane] = sc - v;  // exclusive prefix of the warp totals
        }
        __syncthreads();
        int run = S.warp_sums[warp] + incl - sum;
        for (int k = b0; k < b1; ++k) {
            const int v = S.col_start[k];
            S.col_start[k] = run;
            S.cursor[k] = run;
            run += v;
        }
        if (tid == 0) S.col_start[cells + 1] = n;
    }
    __syncthreads();
    // ---- 3. scatter (order inside a cell arbitrary), then restore index order inside every cell: together a stable
    //         sort by (cell key, index) = the traversal order of get_keypoints_in_cell (data/common.cc:275-309)
    for (int i = tid; i < n; i += kThreads) S.orig[atomicAdd(&S.cursor[key[i]], 1)] = i;
    __syncthreads();
    const int n_in = S.col_start[cells];
    for (int k = tid; k < cells; k += kThreads) {
        const int b0 = S.col_start[k], b1 = S.col_start[k + 1];
        for (int a = b0 + 1; a < b1; ++a) {  // insertion sort of the (few) indices of one cell
            const int v = S.orig[a];
            int b = a - 1;
            while (b >= b0 && S.orig[b] > v) {
                S.orig[b + 1] = S.orig[b];
                --b;
            }
            S.orig[b + 1] = v;
        }
    }
    __syncthreads();
    // gather the sorted keypoint data into shared memory
    for (int p = tid; p < n_in; p += kThreads) {
        const int i = S.orig[p];
        const int k = key[i];
        const int cy = k % grid.num_rows;
        S.x[p] = J.x[i];
        S.y[p] = J.y[i];
        S.xr[p] = J.x_right ? J.x_right[i] : -1.0f;
        const int cl = J.claimed ? (J.claimed[i] != 0) : 0;
        S.meta[p] = (J.octave[i] & 0xff) | (cy << 8) | (cl << 16) | ((k / grid.num_rows) << 17);
        uint4 d0, d1;
        load_desc(J.desc + 32 * (size_t)i, d0, d1);
        S.desc[2 * p] = d0;
        S.desc[2 * p + 1] = d1;
    }
    __syncthreads();  // key[] (owner_a) no longer needed after this point

    ClaimRounds<kThreads> claims{S.owner_a, S.owner_b, &S.flags[0], n_in};
    claims.reset(tid);
    __syncthreads();

    // ---- 4. the sequential greedy assignment, in parallel
    const int gl = tid & (kGroup - 1);          // lane inside the group
    const int grp = tid / kGroup;               // group of this thread
    constexpr int kGroups = kThreads / kGroup;  // queries in flight
    const int m_pad = ((m + kGroups - 1) / kGroups) * kGroups;  // every warp runs the same number of passes (shuffles)

    if (!ratio_test) {
        // No ratio test (match_current_and_last_frames): "best unclaimed candidate, queries served in index order"
        // is a serial dictatorship = the unique stable matching when every keypoint prefers the smallest query
        // index.  Deferred acceptance reaches it with work proportional to the number of conflicts: every query
        // proposes to its best candidate; a keypoint keeps its smallest proposer; only bumped queries re-propose
        // to their next candidate in (distance, order).
        int *owner = claims.prev;  // min proposer so far; never reset
        const int hamm_thr = J.hamm_thr_p1 ? (int)J.hamm_thr_p1 - 1 : PLP_HAMMING_DIST_THR_HIGH;
        // A proposal returns the previous owner from its atomicMin: smaller -> the proposer lost at once and moves to its
        // next candidate; larger -> that owner has just been bumped, and the SAME group re-proposes for it right away
        // (it knows the lost keypoint, hence the floor).  A query is in the hands of at most one group at any time (it
        // holds one proposal; only the group that displaces it takes it over), every step lowers an owner or exhausts a
        // candidate list, so the chains end -- without a single block barrier or work list.  The first generation re-ran
        // whole rounds separated by barriers: 46-68 % of the kernel's stall samples were 1000 threads waiting for the few
        // bumped queries of a round (profiles/source_hotspots_r02*.md).
        // Queries are handed out by a shared counter (the result of deferred acceptance does not depend on the order of
        // the proposals): a group whose chain has ended takes the next query at once, so the 8 groups of a warp stay busy
        // while one of them follows a long chain, and only the last few chains of the frame run alone.  A proposal that
        // loses moves on to the second-best key of the same scan before the window is scanned again.
        int cur = -1, floor = -1;
        const int leader = lane & ~(kGroup - 1);
        for (;;) {
            {
                int q = -1;
                if (cur < 0 && gl == 0) {
                    q = atomicAdd(&S.flags[3], 1);
                    while (q < m && J.qvalid && J.qvalid[q] == 0) {
                        J.choice[q] = -1;
                        q = atomicAdd(&S.flags[3], 1);
                    }
                    if (q >= m) q = -1;
                }
                const int got = __shfl_sync(0xffffffffu, q, leader);  // every lane of the warp takes part
                if (cur < 0) {
                    cur = got;
                    floor = -1;
                }
            }
            if (!__any_sync(0xffffffffu, cur >= 0)) break;
            int k1, k2;
            group_scan(S, J, grid, cur >= 0, cur, gl, nullptr, floor, k1, k2);
            int next = -1, nfloor = -1;
            if (gl == 0 && cur >= 0) {
                J.choice[cur] = -1;
#pragma unroll
                for (int t = 0; t < 2; ++t) {
                    const int key = t == 0 ? k1 : k2;
                    if (key == kNoKey || (key >> 12) > hamm_thr) {
                        // keys come in ascending (distance, order): nothing acceptable is left, the query stays unmatched
                        next = -1;
                        break;
                    }
                    const int choice = key & 0xfff;
                    J.choice[cur] = choice;
                    __threadfence_block();  // the choice is visible before another group can take the query over
                    const int old = atomicMin(&owner[choice], cur);
                    if (old < cur) {  // lost at once: continue behind this candidate (second key, then a new scan)
                        J.choice[cur] = -1;
                        next = cur;
                        nfloor = key;
                        continue;
                    }
                    next = -1;
                    if (old != kNoOwner) {  // bumped `old` off this keypoint: find its next candidate
                        uint4 o0, o1;
                        load_desc(J.qdesc + 32 * (size_t)old, o0, o1);
                        next = old;
                        nfloor = (hamming256(o0, o1, S.desc[2 * choice], S.desc[2 * choice + 1]) << 12) | choice;
                    }
                    break;
                }
            }
            cur = __shfl_sync(0xffffffffu, next, leader);
            floor = __shfl_sync(0xffffffffu, nfloor, leader);
        }
        __syncthreads();
    } else {
        // Ratio test (match_frame_and_landmarks): acceptance depends on the second-best AVAILABLE candidate, so we
        // iterate choice[q] = f(claims of queries < q) to its (unique) fixed point.
        for (int round = 0; round <= m; ++round) {
            for (int q0 = 0; q0 < m_pad; q0 += kGroups) {
                const int q = q0 + grp;
                const bool valid = q < m && (J.qvalid ? (J.qvalid[q] != 0) : true);
                bool rescan = valid;
                if (valid && round > 0) {
                    // a query's result depends only on the owners inside its column span: if none of them changed
                    // in the previous round the previous choice stands (it only re-issues its claim)
                    const float ref_x = J.qx[q], r = J.qradius[q];
                    const int min_cx = max(0, cv_floor((double)(ref_x - grid.min_x - r) * grid.inv_cell_width));
                    const int max_cx = min(grid.num_cols - 1, cv_ceil((double)(ref_x - grid.min_x + r) * grid.inv_cell_width));
                    bool dirty = false;
                    for (int c = min_cx + gl; c <= max_cx; c += kGroup) dirty = dirty || S.colchg[c];
                    rescan = dirty;
                }
                if (round > 0) rescan = group_any(rescan);
                if (!__any_sync(0xffffffffu, rescan)) {
                    if (gl == 0 && valid) {
                        const int choice = J.choice[q];
                        if (choice >= 0) claims.claim(choice, q);
                    }
                    continue;
                }
                int k1, k2;
                group_scan(S, J, grid, rescan, q, gl, claims.prev, -1, k1, k2);
                if (gl == 0 && q < m) {
                    int choice = -1;
                    if (!valid) {
                        choice = -1;
                    } else if (!rescan) {
                        choice = J.choice[q];
                    } else if (k1 != kNoKey) {
                        const int best = k1 >> 12, best_p = k1 & 0xfff;
                        const int best_lvl = (int)(signed char)(S.meta[best_p] & 0xff);
                        const int second = k2 != kNoKey ? (k2 >> 12) : PLP_MAX_HAMMING_DIST;
                        const int second_lvl = k2 != kNoKey ? (int)(signed char)(S.meta[k2 & 0xfff] & 0xff) : -1;
                        if (best <= PLP_HAMMING_DIST_THR_HIGH) {
                            bool ok = true;
                            if (best_lvl == second_lvl && (float)best > lowe_ratio * (float)second) ok = false;
                            if (ok) choice = best_p;
                        }
                    }
                    J.choice[q] = choice;
                    if (choice >= 0) claims.claim(choice, q);
                }
            }
            __syncthreads();  // every query has read colchg
            for (int c = tid; c < grid.num_cols; c += kThreads) S.colchg[c] = 0;
            if (claims.settled(tid, [&](int p) { S.colchg[(S.meta[p] >> 17) & 0x3fff] = 1; })) break;
        }
    }
    // choice[] now holds the sequential result

    // ---- 5. orientation histogram (projection.cc:337-354) and outputs
    if (J.matched_out)
        for (int i = tid; i < n; i += kThreads) J.matched_out[i] = -1;
    const bool do_angle = check_orientation && J.qangle != nullptr && J.angle != nullptr;
    orientation_filter<kThreads>(
        m, J.choice, do_angle, S.hist, S.bin_valid, &S.flags[1], J.num_matches,
        [&](int q, int p) { return J.qangle[q] - J.angle[S.orig[p]]; },
        [&](int q, int p, bool keep) {
            const int i = keep ? S.orig[p] : -1;
            if (keep && J.matched_out) J.matched_out[i] = q;
            if (J.best_idx_out) J.best_idx_out[q] = i;
        });
}

}  // namespace pm

}  // namespace plp
