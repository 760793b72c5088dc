// orb_quadtree.cuh -- quadtree keypoint distribution of the ORB extractor (orb_extractor.cc:468-685) in the array
// formulation of tools/quadtree_parallel_model.py: one CTA per (level, frame).  Free of host-side CUDA runtime calls, so
// tests/cta_emu compiles the same text for the host.
//
// The kernel is a template on its thread count, node capacity and shared-memory candidate window; orb.cu picks an
// instance per level from the level's node need (4 * budget + 8) so that small levels do not pay for a CTA sized for the
// largest one.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "devmath.cuh"

namespace plp {
namespace qt {

constexpr int kMaxLevels = 16;
constexpr int kPatchRadius = 19;  // orb_extractor.h:161 orb_patch_radius_
constexpr int kCellCap = 1024;    // max NMS survivors of a 64x64 tested area (one cell list of cell_buf)
constexpr int kMaxCands = 65535;  // candidates of one level beyond this are dropped (status 1)
constexpr int kBytesPerCand = 4 + 2 * 5 + 1;  // cand, perm x2, owner x2, rank, cls

struct LevelKp {  // quadtree output, level coordinates (border already added)
    short x, y;
    int response;
};

struct QtLevel {
    int w, h;
    int cell_base, num_cells;  // this level's cells in the per-frame cell list
    int budget;                // num_keypts_per_level_
    int slot_base, slot_cap;   // output slots of this level (per-level keypoint lists)
};

struct QtDev {
    int num_levels;   // per frame
    int num_cells;    // per frame
    int total_slots;  // per frame
    int level_base;   // level of blockIdx.x == 0 (one launch covers a contiguous range of levels)
    QtLevel lv[kMaxLevels];
    const uint32_t *cell_buf;  // batch x num_cells x kCellCap packed (x:11 | y:10 | score:8), row-major in the cell
    const int *cell_cnt;       // batch x num_cells
    LevelKp *lvl_kp;           // batch x total_slots
    int *lvl_cnt;              // batch x num_levels
    uint8_t *scratch;          // global work area of jobs whose candidates exceed the shared-memory window
    size_t scratch_per_job;    // >= kMaxCands * kBytesPerCand
    int *status;               // batch: 1 = candidates dropped, 3 = output slots exceeded
};

struct QtArrays {
    uint32_t *cand;             // packed candidates in gather order
    unsigned short *perm[2];    // permutation (indices into cand), ping-pong
    unsigned short *owner[2];   // list position of the node owning each perm slot, ping-pong
};

struct QtNodes {  // struct of arrays in list order
    short4 *rect;              // bx, by, ex, ey
    unsigned short *start;     // segment start in perm
    unsigned short *cnt;
    uint8_t *leaf;
};

__device__ __forceinline__ int cand_x(uint32_t c) { return (int)(c & 0x7ff); }
__device__ __forceinline__ int cand_y(uint32_t c) { return (int)((c >> 11) & 0x3ff); }
__device__ __forceinline__ int cand_score(uint32_t c) { return (int)(c >> 21); }

// block-wide exclusive scan of `v` (one value per thread); returns the exclusive prefix, *total = sum.  The warp totals
// are scanned by warp 0 with shuffles: kThreads / 32 <= 32 lanes.
template <int kThreads>
__device__ __forceinline__ int block_exclusive_scan(int v, int *smem_warp /*[kThreads / 32 + 1]*/, int *total) {
    constexpr int kWarps = kThreads / 32;
    static_assert(kThreads % 32 == 0 && kWarps <= 32, "1..32 whole warps");
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    __syncthreads();  // protect smem_warp reuse
    if (lane == 31) smem_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int s = lane < kWarps ? smem_warp[lane] : 0;
        int si = s;
#pragma unroll
        for (int o = 1; o < kWarps; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, si, o);
            if (lane >= o) si += t;
        }
        if (lane < kWarps) smem_warp[lane] = si - s;
        if (lane == kWarps - 1) smem_warp[kWarps] = si;
    }
    __syncthreads();
    *total = smem_warp[kWarps];
    return smem_warp[warp] + incl - v;
}

// exclusive scan over an array of length n in shared memory (in place); returns the total
template <int kThreads, class V>
__device__ int block_scan_array(V *data, int n, int *smem_warp) {
    const int per = (n + kThreads - 1) / kThreads;
    const int i0 = min(n, (int)threadIdx.x * per), i1 = min(n, i0 + per);
    int sum = 0;
    for (int i = i0; i < i1; ++i) sum += data[i];
    int total;
    int run = block_exclusive_scan<kThreads>(sum, smem_warp, &total);
    for (int i = i0; i < i1; ++i) {
        const int v = data[i];
        data[i] = (V)run;
        run += v;
    }
    __syncthreads();
    return total;
}

// child class of a keypoint inside node rect (orb_extractor_node.cc:67-78)
__device__ __forceinline__ int classify(const short4 r, uint32_t c) {
    const unsigned half_x = (unsigned)cv_ceil((r.z - r.x) / 2.0);
    const unsigned half_y = (unsigned)cv_ceil((r.w - r.y) / 2.0);
    int q = 0;
    if ((float)((unsigned)r.x + half_x) <= (float)cand_x(c)) q += 1;
    if ((float)((unsigned)r.y + half_y) <= (float)cand_y(c)) q += 2;
    return q;
}

__device__ __forceinline__ short4 child_rect(const short4 r, int q) {
    const int half_x = cv_ceil((r.z - r.x) / 2.0), half_y = cv_ceil((r.w - r.y) / 2.0);
    short4 c;
    c.x = (q & 1) ? (short)(r.x + half_x) : r.x;
    c.z = (q & 1) ? r.z : (short)(r.x + half_x);
    c.y = (q & 2) ? (short)(r.y + half_y) : r.y;
    c.w = (q & 2) ? r.w : (short)(r.y + half_y);
    return c;
}

// Segmented scan of per-element class counters.  For every perm slot i whose node is selected (sel[owner]),
// computes rank[i] = number of earlier slots of the same node with the same class, and per node the four
// class totals tot[node*4 + q].  The four counters of a slot are packed as 4 x 16 bits.
template <int kThreads>
__device__ void segmented_class_scan(const QtArrays &A, int cur, int n, const QtNodes &N, const uint8_t *sel,
                                     unsigned short *rank, uint8_t *cls, unsigned short *tot,
                                     unsigned long long *carry_tail, uint8_t *carry_head) {
    const int tid = threadIdx.x;
    const int per = (n + kThreads - 1) / kThreads;
    const int i0 = min(n, tid * per), i1 = min(n, i0 + per);
    const unsigned short *perm = A.perm[cur], *owner = A.owner[cur];
    // pass 1: local tail since the last segment head in this chunk
    unsigned long long acc = 0;
    bool head = false;
    int prev_owner = (i0 > 0 && i0 < n) ? owner[i0 - 1] : -1;
    for (int i = i0; i < i1; ++i) {
        const int o = owner[i];
        if (o != prev_owner) {
            head = true;
            acc = 0;
        }
        prev_owner = o;
        int q = 0;
        if (sel[o]) q = classify(N.rect[o], A.cand[perm[i]]);
        cls[i] = (uint8_t)q;
        if (sel[o]) acc += 1ull << (16 * q);
    }
    // the first element of a chunk starts a new segment iff its owner differs from the previous slot's owner;
    // that case is covered above because prev_owner was initialised from owner[i0-1].
    carry_tail[tid] = acc;
    carry_head[tid] = head ? 1 : 0;
    __syncthreads();
    // pass 2: carry-in per thread = segmented exclusive scan over the kThreads (tail, head) pairs, done by warp 0:
    // each lane folds kThreads / 32 consecutive entries, the 32 lane aggregates are scanned with shuffles.
    if (tid < 32) {
        constexpr int kPer = kThreads / 32;
        unsigned long long run = 0;
        bool hf = false;
        for (int t = tid * kPer; t < (tid + 1) * kPer; ++t) {
            const bool h = carry_head[t] != 0;
            run = h ? carry_tail[t] : run + carry_tail[t];
            hf = hf || h;
        }
        unsigned long long v = run;
        int f = hf ? 1 : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long pv = __shfl_up_sync(0xffffffffu, v, o);
            const int pf = __shfl_up_sync(0xffffffffu, f, o);
            if (tid >= o) {
                if (!f) v += pv;
                f |= pf;
            }
        }
        unsigned long long carry = __shfl_up_sync(0xffffffffu, v, 1);
        if (tid == 0) carry = 0;
        run = carry;
        for (int t = tid * kPer; t < (tid + 1) * kPer; ++t) {
            const bool h = carry_head[t] != 0;
            const unsigned long long tail = carry_tail[t];
            carry_tail[t] = run;  // carry-in of thread t
            run = h ? tail : run + tail;
        }
    }
    __syncthreads();
    // pass 3: ranks and node totals
    acc = carry_tail[tid];
    prev_owner = (i0 > 0 && i0 < n) ? owner[i0 - 1] : -1;
    for (int i = i0; i < i1; ++i) {
        const int o = owner[i];
        if (o != prev_owner) acc = 0;
        prev_owner = o;
        const int q = cls[i];
        if (sel[o]) {
            rank[i] = (unsigned short)((acc >> (16 * q)) & 0xffff);
            acc += 1ull << (16 * q);
        }
        const bool last = (i + 1 == n) || (owner[i + 1] != o);
        if (last && sel[o]) {
            tot[o * 4 + 0] = (unsigned short)(acc & 0xffff);
            tot[o * 4 + 1] = (unsigned short)((acc >> 16) & 0xffff);
            tot[o * 4 + 2] = (unsigned short)((acc >> 32) & 0xffff);
            tot[o * 4 + 3] = (unsigned short)((acc >> 48) & 0xffff);
        }
    }
    __syncthreads();
}

// Shared memory of one CTA: node lists (ping-pong) and per-node scratch.  NC = node capacity (>= 4 * budget + 8 of every
// level the instance serves, and >= the level's cell count: the cell-count prefix of the gather lives in `scan`).
// 45 bytes per node.
template <int kThreads, int NC>
struct QtSharedT {
    short4 rect[2][NC];
    unsigned short start[2][NC];
    unsigned short cnt[2][NC];
    uint8_t leaf[2][NC];
    uint8_t sel[NC];
    unsigned short tot[NC * 4];
    unsigned short newpos[NC];  // list position of the first (front-most) child / of the kept node
    int scan[NC];               // scratch for scans over the list
    unsigned short pool[NC];    // nodes with more than one keypoint, in creation order (read before it is rewritten)
    unsigned short pool_sorted[NC];
    unsigned long long carry_tail[kThreads];
    uint8_t carry_head[kThreads];
    int warp_tmp[kThreads / 32 + 1];
    int misc[8];
};

// dynamic shared memory of an instance: the node lists plus a window of CC candidates
template <int kThreads, int NC, int CC>
__host__ __device__ constexpr size_t qt_smem_bytes() {
    return ((sizeof(QtSharedT<kThreads, NC>) + 15) & ~(size_t)15) + (size_t)CC * kBytesPerCand;
}

// Applies the division of all nodes with sel[p] != 0 of list `cur_n` (length len): builds the new list
// (children of processed nodes in front, later-processed first, classes reversed; then the untouched nodes in
// order), partitions the keypoints, builds the new pool (children with more than one keypoint, creation
// order).  `proc_list`: the selected nodes in processing order (for phase 1 it is the list order).  Returns the
// new list length.
template <int kThreads, int NC>
__device__ int apply_division(QtSharedT<kThreads, NC> &S, QtArrays &A, int &cur, int n_cand, int &cur_n, int len,
                              int num_proc, const unsigned short *proc_list, unsigned short *rank, uint8_t *cls,
                              int *pool_len_out) {
    const int tid = threadIdx.x;
    const int nxt_n = cur_n ^ 1;
    // children count per processed node, in processing order -> S.scan[k]
    for (int k = tid; k < num_proc; k += kThreads) {
        const int p = proc_list[k];
        const unsigned short *t = S.tot + p * 4;
        S.scan[k] = (t[0] > 0) + (t[1] > 0) + (t[2] > 0) + (t[3] > 0);
    }
    __syncthreads();
    const int total_children = block_scan_array<kThreads>(S.scan, num_proc, S.warp_tmp);  // exclusive prefix over k
    // kept nodes: positions after all children, in list order (exclusive scan of kept flags over the list)
    for (int p = tid; p < len; p += kThreads) S.newpos[p] = S.sel[p] ? 0 : 1;
    __syncthreads();
    const int kept = block_scan_array<kThreads>(S.newpos, len, S.warp_tmp);
    const int new_len = total_children + kept;
    for (int p = tid; p < len; p += kThreads) {
        if (!S.sel[p]) {
            const int pos = total_children + S.newpos[p];
            S.rect[nxt_n][pos] = S.rect[cur_n][p];
            S.start[nxt_n][pos] = S.start[cur_n][p];
            S.cnt[nxt_n][pos] = S.cnt[cur_n][p];
            S.leaf[nxt_n][pos] = S.leaf[cur_n][p];
            S.newpos[p] = (unsigned short)pos;
        }
    }
    __syncthreads();
    // children: processed node k has prefix S.scan[k] children before it (in processing order); its children
    // occupy list positions [total_children - S.scan[k] - nch, total_children - S.scan[k]) with class order
    // reversed (orb_extractor.cc:639-657 pushes to the front).
    for (int k = tid; k < num_proc; k += kThreads) {
        const int p = proc_list[k];
        const unsigned short *t = S.tot + p * 4;
        const int nch = (t[0] > 0) + (t[1] > 0) + (t[2] > 0) + (t[3] > 0);
        const int base = total_children - S.scan[k] - nch;
        const short4 r = S.rect[cur_n][p];
        int o = S.start[cur_n][p];
        int rnk = 0;
        for (int q = 0; q < 4; ++q) {
            if (t[q] == 0) continue;
            const int pos = base + (nch - 1 - rnk);
            S.rect[nxt_n][pos] = child_rect(r, q);
            S.start[nxt_n][pos] = (unsigned short)o;
            S.cnt[nxt_n][pos] = t[q];
            S.leaf[nxt_n][pos] = 0;
            o += t[q];
            ++rnk;
        }
        S.newpos[p] = (unsigned short)base;  // front-most child position; class q child = base + (nch-1-rank_q)
    }
    __syncthreads();
    // keypoints: stable 4-way partition inside each processed node, owner update for everybody
    {
        const unsigned short *perm = A.perm[cur], *owner = A.owner[cur];
        unsigned short *perm2 = A.perm[cur ^ 1], *owner2 = A.owner[cur ^ 1];
        for (int i = tid; i < n_cand; i += kThreads) {
            const int o = owner[i];
            if (S.sel[o]) {
                const unsigned short *t = S.tot + o * 4;
                const int q = cls[i];
                int off = 0, rnk = 0;
                for (int c = 0; c < q; ++c) {
                    off += t[c];
                    rnk += (t[c] > 0);
                }
                const int nch = (t[0] > 0) + (t[1] > 0) + (t[2] > 0) + (t[3] > 0);
                const int dst = S.start[cur_n][o] + off + rank[i];
                perm2[dst] = perm[i];
                owner2[dst] = (unsigned short)(S.newpos[o] + (nch - 1 - rnk));
            } else {
                perm2[i] = perm[i];
                owner2[i] = (unsigned short)S.newpos[o];
            }
        }
    }
    __syncthreads();
    // new pool: children with cnt > 1 in creation order (processing order, classes ascending)
    for (int k = tid; k < num_proc; k += kThreads) {
        const unsigned short *t = S.tot + proc_list[k] * 4;
        S.scan[k] = (t[0] > 1) + (t[1] > 1) + (t[2] > 1) + (t[3] > 1);
    }
    __syncthreads();
    const int pool_len = block_scan_array<kThreads>(S.scan, num_proc, S.warp_tmp);
    for (int k = tid; k < num_proc; k += kThreads) {
        const int p = proc_list[k];
        const unsigned short *t = S.tot + p * 4;
        const int nch = (t[0] > 0) + (t[1] > 0) + (t[2] > 0) + (t[3] > 0);
        int w = S.scan[k], rnk = 0;
        for (int q = 0; q < 4; ++q) {
            if (t[q] == 0) continue;
            if (t[q] > 1) S.pool[w++] = (unsigned short)(S.newpos[p] + (nch - 1 - rnk));
            ++rnk;
        }
    }
    __syncthreads();
    *pool_len_out = pool_len;
    cur ^= 1;
    cur_n = nxt_n;
    return new_len;
}

// One CTA per (level, frame): blockIdx.x + P.level_base is the level, blockIdx.y the frame.  A level with more candidates
// than the shared-memory window CC works in its global scratch block (decided per job).
template <int kThreads, int NC, int CC, int kMinBlocks>
__global__ void __launch_bounds__(kThreads, kMinBlocks) quadtree_kernel(QtDev P) {
    PLP_DYNAMIC_SMEM(qsmem);
    using QtShared = QtSharedT<kThreads, NC>;
    QtShared &S = *reinterpret_cast<QtShared *>(qsmem);
    const int l = P.level_base + (int)blockIdx.x, b = blockIdx.y, tid = threadIdx.x;
    const QtLevel &LV = P.lv[l];
    int *lvl_cnt = P.lvl_cnt + (size_t)b * P.num_levels + l;
    LevelKp *out = P.lvl_kp + (size_t)b * P.total_slots + LV.slot_base;

    // ---- candidates of this level in cell order (prefix over cell counts)
    const int num_cells = LV.num_cells;
    const int *cc = P.cell_cnt + (size_t)b * P.num_cells + LV.cell_base;
    for (int c = tid; c < num_cells; c += kThreads) S.scan[c] = cc[c];
    __syncthreads();
    int n = block_scan_array<kThreads>(S.scan, num_cells, S.warp_tmp);
    if (n == 0) {
        if (tid == 0) *lvl_cnt = 0;
        return;
    }
    if (n > kMaxCands) {
        n = kMaxCands;
        if (tid == 0) P.status[b] = 1;
    }
    // work arrays: shared memory when they fit, else the global scratch block of this (frame, level)
    QtArrays A;
    unsigned short *rank;
    uint8_t *cls;
    {
        uint8_t *base;
        if (n <= CC) {
            base = qsmem + ((sizeof(QtShared) + 15) & ~(size_t)15);
        } else {
            base = P.scratch + ((size_t)b * P.num_levels + l) * P.scratch_per_job;
        }
        const size_t cap = n <= CC ? CC : kMaxCands + 1;
        A.cand = reinterpret_cast<uint32_t *>(base);
        base += cap * 4;
        A.perm[0] = reinterpret_cast<unsigned short *>(base);
        base += cap * 2;
        A.perm[1] = reinterpret_cast<unsigned short *>(base);
        base += cap * 2;
        A.owner[0] = reinterpret_cast<unsigned short *>(base);
        base += cap * 2;
        A.owner[1] = reinterpret_cast<unsigned short *>(base);
        base += cap * 2;
        rank = reinterpret_cast<unsigned short *>(base);
        base += cap * 2;
        cls = base;
    }
    {
        // gather: candidate i belongs to the last cell whose prefix is <= i (empty cells share their successor's prefix),
        // so every thread finds its cell by a binary search and all loads of the level are in flight together.  The
        // order is cell order, then the FAST kernel's row-major order inside the cell.
        const uint32_t *cb = P.cell_buf + ((size_t)b * P.num_cells + LV.cell_base) * kCellCap;
        for (int i = tid; i < n; i += kThreads) {
            int lo = 0, hi = num_cells - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (S.scan[mid] <= i)
                    lo = mid;
                else
                    hi = mid - 1;
            }
            A.cand[i] = cb[(size_t)lo * kCellCap + (i - S.scan[lo])];
        }
    }
    __syncthreads();

    // ---- initialize_nodes (orb_extractor.cc:557-637)
    const int min_x = kPatchRadius, max_x = LV.w - kPatchRadius, min_y = kPatchRadius, max_y = LV.h - kPatchRadius;
    const double ratio = (double)(max_x - min_x) / (max_y - min_y);
    int gx, gy;
    double dx, dy;
    if (ratio > 1) {
        gx = (int)round(ratio);
        gy = 1;
        dx = (double)(max_x - min_x) / gx;
        dy = max_y - min_y;
    } else {
        gx = 1;
        gy = (int)round(1 / ratio);
        dx = max_x - min_y;  // sic, orb_extractor.cc:580
        dy = (double)(max_y - min_y) / gy;
    }
    const int g = gx * gy;  // number of initial nodes (small)
    int cur = 0, cur_n = 0, len = 0;
    {
        // stable counting sort of the candidates by initial node
        int *cnts = S.scan;  // g entries
        for (int i = tid; i < g; i += kThreads) cnts[i] = 0;
        __syncthreads();
        for (int i = tid; i < n; i += kThreads) {
            const uint32_t c = A.cand[i];
            const unsigned ix = (unsigned)((float)cand_x(c) / dx), iy = (unsigned)((float)cand_y(c) / dy);
            int node = (int)(ix + iy * gx);
            node = min(node, g - 1);
            cls[i] = 0;
            A.owner[0][i] = (unsigned short)node;  // temporarily the initial node index
            atomicAdd(&cnts[node], 1);
        }
        __syncthreads();
        // node offsets + list (thread 0; g is tiny)
        if (tid == 0) {
            int off = 0, pos = 0;
            for (int i = 0; i < g; ++i) {
                const int c = cnts[i];
                S.newpos[i] = (unsigned short)off;  // segment start of initial node i
                if (c > 0) {
                    const int ix = i % gx, iy = i / gx;
                    short4 r;
                    r.x = (short)(int)(dx * ix);
                    r.y = (short)(int)(dy * iy);
                    r.z = (short)(int)(dx * (ix + 1));
                    r.w = (short)(int)(dy * (iy + 1));
                    S.rect[0][pos] = r;
                    S.start[0][pos] = (unsigned short)off;
                    S.cnt[0][pos] = (unsigned short)c;
                    S.leaf[0][pos] = (c == 1);
                    S.tot[i] = (unsigned short)pos;  // initial node -> list position
                    ++pos;
                }
                off += c;
            }
            S.misc[0] = pos;
        }
        __syncthreads();
        len = S.misc[0];
        // stable placement: rank of element i inside its initial node = #earlier elements of the same node.
        // g is tiny, so do one ordered pass per initial node with a block scan of flags.
        for (int node = 0; node < g; ++node) {
            if (cnts[node] == 0) continue;
            const int per = (n + kThreads - 1) / kThreads;
            const int i0 = min(n, tid * per), i1 = min(n, i0 + per);
            int c = 0;
            for (int i = i0; i < i1; ++i) c += (A.owner[0][i] == node);
            int tot;
            int run = block_exclusive_scan<kThreads>(c, S.warp_tmp, &tot);
            const int base = S.newpos[node];
            const unsigned short lp = S.tot[node];
            for (int i = i0; i < i1; ++i)
                if (A.owner[0][i] == node) {
                    A.perm[1][base + run] = (unsigned short)i;
                    A.owner[1][base + run] = lp;
                    ++run;
                }
            __syncthreads();
        }
        cur = 1;
    }
    const int budget = LV.budget;
    int pool_len = 0;
    bool filled = false;
    unsigned short *proc_list = S.pool_sorted;

    // ---- phase 1 (orb_extractor.cc:482-518)
    while (true) {
        const int prev = len;
        for (int p = tid; p < len; p += kThreads) S.sel[p] = S.leaf[cur_n][p] ? 0 : 1;
        __syncthreads();
        // processing order = list order of the selected nodes
        for (int p = tid; p < len; p += kThreads) S.scan[p] = S.sel[p];
        __syncthreads();
        const int num_proc = block_scan_array<kThreads>(S.scan, len, S.warp_tmp);
        for (int p = tid; p < len; p += kThreads)
            if (S.sel[p]) proc_list[S.scan[p]] = (unsigned short)p;
        __syncthreads();
        segmented_class_scan<kThreads>(A, cur, n, QtNodes{S.rect[cur_n], S.start[cur_n], S.cnt[cur_n], S.leaf[cur_n]},
                                       S.sel, rank, cls, S.tot, S.carry_tail, S.carry_head);
        len = apply_division(S, A, cur, n, cur_n, len, num_proc, proc_list, rank, cls, &pool_len);
        if (budget <= len || len == prev) {
            filled = true;
            break;
        }
        if (budget < len + pool_len) break;
    }
    // ---- phase 2 (orb_extractor.cc:520-552)
    while (!filled) {
        const int prev = len;
        const unsigned short *pool = S.pool;
        for (int p = tid; p < len; p += kThreads) S.sel[p] = 0;
        __syncthreads();
        for (int k = tid; k < pool_len; k += kThreads) S.sel[pool[k]] = 1;
        __syncthreads();
        segmented_class_scan<kThreads>(A, cur, n, QtNodes{S.rect[cur_n], S.start[cur_n], S.cnt[cur_n], S.leaf[cur_n]},
                                       S.sel, rank, cls, S.tot, S.carry_tail, S.carry_head);
        // sort the pool by (cnt desc, creation desc): rank sort
        for (int k = tid; k < pool_len; k += kThreads) {
            const int ck = S.cnt[cur_n][pool[k]];
            int r = 0;
            for (int j = 0; j < pool_len; ++j) {
                const int cj = S.cnt[cur_n][pool[j]];
                r += (cj > ck) || (cj == ck && j > k);
            }
            proc_list[r] = pool[k];
        }
        __syncthreads();
        // cut: first t with prev + sum_{i<=t}(nch_i - 1) >= budget
        for (int k = tid; k < pool_len; k += kThreads) {
            const unsigned short *t = S.tot + proc_list[k] * 4;
            S.scan[k] = (t[0] > 0) + (t[1] > 0) + (t[2] > 0) + (t[3] > 0) - 1;
        }
        if (tid == 0) {
            S.misc[1] = pool_len;
            S.misc[2] = 0;
        }
        __syncthreads();
        block_scan_array<kThreads>(S.scan, pool_len, S.warp_tmp);  // exclusive prefix of (nch-1)
        for (int k = tid; k < pool_len; k += kThreads) {
            const unsigned short *t = S.tot + proc_list[k] * 4;
            const int inc = (t[0] > 0) + (t[1] > 0) + (t[2] > 0) + (t[3] > 0) - 1;
            if (prev + S.scan[k] + inc >= budget) {  // list size after dividing the k-th pool node
                atomicMin(&S.misc[1], k + 1);
                S.misc[2] = 1;
            }
        }
        __syncthreads();
        const int num_proc = S.misc[1];
        const bool reached = S.misc[2] != 0;
        __syncthreads();
        // only the first num_proc pool nodes are divided
        for (int k = num_proc + tid; k < pool_len; k += kThreads) S.sel[proc_list[k]] = 0;
        __syncthreads();
        len = apply_division(S, A, cur, n, cur_n, len, num_proc, proc_list, rank, cls, &pool_len);
        if (reached) filled = true;
        if (filled || budget <= len || len == prev) break;
    }

    // ---- find_keypoints_with_max_response (orb_extractor.cc:659-685): first maximum wins
    const int n_out = min(len, LV.slot_cap);
    if (len > LV.slot_cap && tid == 0) P.status[b] = 3;
    for (int p = tid; p < n_out; p += kThreads) {
        const int st = S.start[cur_n][p], c = S.cnt[cur_n][p];
        uint32_t best = A.cand[A.perm[cur][st]];
        for (int k = 1; k < c; ++k) {
            const uint32_t v = A.cand[A.perm[cur][st + k]];
            if (cand_score(v) > cand_score(best)) best = v;
        }
        LevelKp kp;
        kp.x = (short)(cand_x(best) + kPatchRadius);  // orb_extractor.cc:450-454
        kp.y = (short)(cand_y(best) + kPatchRadius);
        kp.response = cand_score(best);
        out[p] = kp;
    }
    if (tid == 0) *lvl_cnt = n_out;
}

}  // namespace qt
}  // namespace plp
