// fuse_kernels.cuh -- device code of the match::fuse search (fuse.cu launches it).  Free of host-side CUDA runtime
// dependencies so that tests/cta_emu can compile the same text for the host.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/plpslam_b200.h"
#include "devmath.cuh"

namespace plp {

namespace {

constexpr int kThreads = 512;
constexpr int kFuseMaxPoints = 3072;  // keypoints per target keyframe (shared-memory bound, like the window matcher)
constexpr int kFuseMaxLines = 2048;   // keylines per target keyframe
constexpr int kMaxLevels = 32;

struct FusePointTarget {
    int n;
    const float *x, *y, *xr;  // xr may be null (monocular keyframe)
    const int32_t *octave;
    const uint8_t *desc;
    const uint8_t *skip;  // may be null
    double R[9], t[3], c[3];
};

struct FuseLineTarget {
    int n;
    const float *sx, *sy, *ex, *ey;
    const int32_t *octave;
    const uint8_t *desc;
    const uint8_t *skip;  // may be null
    double R[9], t[3], c[3];
};

struct FuseLandmarks {
    int m;
    const double *pos_w;
    const double *normal;  // points only
    const float *min_d, *max_d, *max_raw;
    const uint8_t *desc;
    const uint8_t *valid;  // may be null
};

struct FuseParams {
    plp_camera cam;
    plp_grid grid;  // points only
    float scale_factors[kMaxLevels];
    float inv_sigma_sq[kMaxLevels];
    float level_thr[kMaxLevels];  // level_thr[k], 1 <= k < num_levels: smallest ratio whose predicted level is >= k
    int num_levels;
    float margin;
    int mode;
};

// data/landmark.cc:341-362 through the host-derived threshold table
__device__ __forceinline__ int predict_level(float ratio, const FuseParams &P) {
    int lvl = 0;
    for (int k = 1; k < P.num_levels; ++k) lvl += (ratio >= P.level_thr[k]) ? 1 : 0;
    return lvl;
}

struct Proj {
    double u, v;
    float x_right;
    bool in_image;
};

// camera/perspective.cc:190-209; a point behind the camera leaves (u, v) = (0, 0) (the reference leaves them unset)
__device__ __forceinline__ Proj reproject(const plp_camera &cam, const double *R, const double *t, const double *X) {
    Proj r;
    r.u = 0.0;
    r.v = 0.0;
    r.x_right = 0.0f;
    r.in_image = false;
    const double pc0 = R[0] * X[0] + R[1] * X[1] + R[2] * X[2] + t[0];
    const double pc1 = R[3] * X[0] + R[4] * X[1] + R[5] * X[2] + t[1];
    const double pc2 = R[6] * X[0] + R[7] * X[1] + R[8] * X[2] + t[2];
    if (pc2 <= 0.0) return r;
    const double z_inv = 1.0 / pc2;
    r.u = cam.fx * pc0 * z_inv + cam.cx;
    r.v = cam.fy * pc1 * z_inv + cam.cy;
    r.x_right = (float)(r.u - cam.focal_x_baseline * z_inv);
    r.in_image = (cam.min_x < r.u && r.u < cam.max_x && cam.min_y < r.v && r.v < cam.max_y);
    return r;
}

__device__ __forceinline__ unsigned long long warp_min_u64(unsigned long long k) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, k, o);
        k = other < k ? other : k;
    }
    return k;
}

static size_t fuse_point_smem_bytes(int cap, int cells) {
    return (size_t)cap * (32 + 6 * 4) + (size_t)(cells + 2) * 8 + 32 * 4;
}

// ---------------------------------------------------------------------------------------------------------------
// points: fuse.cc:40-151 (mode 0) / :153-300 (mode 1)
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
    fuse_points_kernel(const FusePointTarget *__restrict__ targets, FuseLandmarks L, FuseParams P, int cap, int chunk,
                       int32_t *__restrict__ best_idx_out, uint16_t *__restrict__ best_dist_out) {
    PLP_DYNAMIC_SMEM(smem_raw);
    const FusePointTarget &T = targets[blockIdx.y];
    const plp_grid &grid = P.grid;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kThreads / 32;
    const int cells = grid.num_cols * grid.num_rows;
    const int n = T.n;
    const int i0 = blockIdx.x * chunk, i1 = min(L.m, i0 + chunk);
    int32_t *out_idx = best_idx_out + (size_t)blockIdx.y * L.m;
    uint16_t *out_dist = best_dist_out ? best_dist_out + (size_t)blockIdx.y * L.m : nullptr;

    // carve
    uint8_t *base = smem_raw;
    uint4 *s_desc = reinterpret_cast<uint4 *>(base);
    base += (size_t)cap * 32;
    float *s_x = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    float *s_y = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    float *s_xr = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    int *s_oct = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    int *s_orig = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    int *s_key = reinterpret_cast<int *>(base);
    base += (size_t)cap * 4;
    int *s_cell_start = reinterpret_cast<int *>(base);
    base += (size_t)(cells + 2) * 4;
    int *s_cursor = reinterpret_cast<int *>(base);
    base += (size_t)(cells + 2) * 4;
    int *s_warp = reinterpret_cast<int *>(base);

    // ---- 1. cell key of every keypoint (data/common.h:104-109) and the cell histogram
    for (int k = tid; k < cells + 2; k += kThreads) s_cell_start[k] = 0;
    __syncthreads();
    for (int i = tid; i < n; i += kThreads) {
        const float px = T.x[i], py = T.y[i];
        const int cx = cv_floor((double)(px - grid.min_x) * grid.inv_cell_width);
        const int cy = cv_floor((double)(py - grid.min_y) * grid.inv_cell_height);
        const bool in = (0 <= cx && cx < grid.num_cols && 0 <= cy && cy < grid.num_rows);
        const int key = in ? cx * grid.num_rows + cy : cells;  // out-of-grid keypoints sort last and are never visited
        s_key[i] = key;
        atomicAdd(&s_cell_start[key], 1);
    }
    __syncthreads();
    // ---- 2. stable counting sort by (cell key, index) = traversal order of get_keypoints_in_cell
    //         (data/common.cc:275-309).  (a) exclusive scan of the histogram: cell_start[k] = first sorted position
    //         whose key >= k; (b) one warp walks the keypoints in index order, __match_any groups equal keys and gives
    //         every lane its rank inside the group, the group leader advances the cell cursor.
    {
        const int total = cells + 1;  // keys 0 .. cells
        const int per = (total + kThreads - 1) / kThreads;
        const int b0 = min(total, tid * per), b1 = min(total, b0 + per);
        int sum = 0;
        for (int k = b0; k < b1; ++k) sum += s_cell_start[k];
        int incl = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const int v = lane < nwarps ? s_warp[lane] : 0;
            int sc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, sc, o);
                if (lane >= o) sc += u;
            }
            if (lane < nwarps) s_warp[lane] = sc - v;  // exclusive prefix of the warp totals
        }
        __syncthreads();
        int run = s_warp[warp] + incl - sum;
        for (int k = b0; k < b1; ++k) {
            const int v = s_cell_start[k];
            s_cell_start[k] = run;
            s_cursor[k] = run;
            run += v;
        }
        if (tid == 0) s_cell_start[cells + 1] = n;
        __syncthreads();
        if (warp == 0) {
            for (int base = 0; base < n; base += 32) {
                const int i = base + lane;
                const int key = i < n ? s_key[i] : (0x40000000 | lane);  // idle lanes get unique keys
                const unsigned peers = __match_any_sync(0xffffffffu, key);
                const int leader = __ffs(peers) - 1;
                const int rank = __popc(peers & ((1u << lane) - 1));
                int b = 0;
                if (lane == leader && i < n) {
                    b = s_cursor[key];
                    s_cursor[key] = b + __popc(peers);
                }
                b = __shfl_sync(0xffffffffu, b, leader);
                if (i < n) s_orig[b + rank] = i;
                __syncwarp();
            }
        }
    }
    __syncthreads();
    const int n_in = s_cell_start[cells];
    // ---- 3. gather in sorted order; s_oct keeps the octave, the cell key is re-read from s_key through s_orig
    for (int p = tid; p < n_in; p += kThreads) {
        const int i = s_orig[p];
        s_x[p] = T.x[i];
        s_y[p] = T.y[i];
        s_xr[p] = T.xr ? T.xr[i] : -1.0f;
        s_oct[p] = T.octave[i];
        uint4 d0, d1;
        load_desc(T.desc + 32 * (size_t)i, d0, d1);
        s_desc[2 * p] = d0;
        s_desc[2 * p + 1] = d1;
    }
    __syncthreads();

    // ---- 4. one warp per landmark
    for (int i = i0 + warp; i < i1; i += nwarps) {
        int out = -1;
        unsigned outd = 0xFFFFu;
        bool ok = (L.valid ? L.valid[i] != 0 : true) && (T.skip ? T.skip[i] == 0 : true);
        double u = 0.0, v = 0.0;
        float q_xr = 0.0f;
        unsigned pred = 0;
        if (ok) {
            const double X[3] = {L.pos_w[3 * (size_t)i], L.pos_w[3 * (size_t)i + 1], L.pos_w[3 * (size_t)i + 2]};
            const Proj pr = reproject(P.cam, T.R, T.t, X);
            ok = pr.in_image;
            u = pr.u;
            v = pr.v;
            q_xr = pr.x_right;
            if (ok) {
                const double d0 = X[0] - T.c[0], d1 = X[1] - T.c[1], d2 = X[2] - T.c[2];
                const double dist = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
                const float max_d = L.max_d[i], min_d = L.min_d[i];
                if (dist < (double)min_d || (double)max_d < dist) ok = false;
                const double *nm = L.normal + 3 * (size_t)i;
                if (ok && (d0 * nm[0] + d1 * nm[1] + d2 * nm[2] < 0.5 * dist)) ok = false;
                if (ok) pred = (unsigned)predict_level(L.max_raw[i] / (float)dist, P);
            }
        }
        if (ok && n_in > 0) {
            const float ref_x = (float)u, ref_y = (float)v, r = P.margin * P.scale_factors[pred];
            // data/common.cc:249-272
            const int min_cx = max(0, cv_floor((double)(ref_x - grid.min_x - r) * grid.inv_cell_width));
            const int max_cx = min(grid.num_cols - 1, cv_ceil((double)(ref_x - grid.min_x + r) * grid.inv_cell_width));
            const int min_cy = max(0, cv_floor((double)(ref_y - grid.min_y - r) * grid.inv_cell_height));
            const int max_cy = min(grid.num_rows - 1, cv_ceil((double)(ref_y - grid.min_y + r) * grid.inv_cell_height));
            unsigned long long best = ~0ull;
            if (min_cx < grid.num_cols && max_cx >= 0 && min_cy < grid.num_rows && max_cy >= 0) {
                uint4 q0, q1;
                load_desc(L.desc + 32 * (size_t)i, q0, q1);
                const int pred_i = (int)pred;
                for (int c = min_cx; c <= max_cx; ++c) {
                    const int p_begin = s_cell_start[c * grid.num_rows + min_cy];
                    const int p_end = s_cell_start[c * grid.num_rows + max_cy + 1];
                    for (int p = p_begin + lane; p < p_end; p += 32) {
                        const float kx = s_x[p], ky = s_y[p];
                        const float dx = kx - ref_x, dy = ky - ref_y;
                        if (!(fabsf(dx) < r && fabsf(dy) < r)) continue;  // data/common.cc:300-306
                        const int oct = s_oct[p];
                        if (P.mode == PLP_FUSE_DETECT) {
                            if (oct < pred_i - 1 || pred_i < oct) continue;  // fuse.cc:117-121 (int)
                        } else {
                            const unsigned sl = (unsigned)oct;
                            if (sl < pred - 1u || pred < sl) continue;  // fuse.cc:232-236 (unsigned, wraps at pred == 0)
                            if (sl >= (unsigned)P.num_levels) continue;  // inv_level_sigma_sq_.at() would throw
                            const double e_x = u - (double)kx, e_y = v - (double)ky;
                            const float kxr = s_xr[p];
                            if (kxr >= 0) {  // :238-251
                                const float e_xr = q_xr - kxr;
                                const double err = e_x * e_x + e_y * e_y + (double)(e_xr * e_xr);
                                if ((double)7.81473f < err * (double)P.inv_sigma_sq[sl]) continue;
                            } else {  // :252-265
                                const double err = e_x * e_x + e_y * e_y;
                                if ((double)5.99146f < err * (double)P.inv_sigma_sq[sl]) continue;
                            }
                        }
                        const unsigned d = (unsigned)hamming256(q0, q1, s_desc[2 * p], s_desc[2 * p + 1]);
                        const unsigned long long key = ((unsigned long long)d << 32) | (unsigned)p;
                        best = key < best ? key : best;
                    }
                }
            }
            best = warp_min_u64(best);
            if (best != ~0ull) {
                const unsigned d = (unsigned)(best >> 32);
                // best_dist starts at MAX_HAMMING_DIST with a strict '<' (:221-276), then HAMMING_DIST_THR_LOW (:279-282)
                if (d < (unsigned)PLP_MAX_HAMMING_DIST && d <= (unsigned)PLP_HAMMING_DIST_THR_LOW) {
                    out = s_orig[(int)(best & 0xffffffffull)];
                    outd = d;
                }
            }
        }
        if (lane == 0) {
            out_idx[i] = out;
            if (out_dist) out_dist[i] = (uint16_t)outd;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// lines: fuse.cc:304-503
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
    fuse_lines_kernel(const FuseLineTarget *__restrict__ targets, FuseLandmarks L, FuseParams P, int cap, int chunk,
                      int32_t *__restrict__ best_idx_out, uint16_t *__restrict__ best_dist_out) {
    PLP_DYNAMIC_SMEM(smem_raw);
    const FuseLineTarget &T = targets[blockIdx.y];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = kThreads / 32;
    const int n = T.n;
    const int i0 = blockIdx.x * chunk, i1 = min(L.m, i0 + chunk);
    int32_t *out_idx = best_idx_out + (size_t)blockIdx.y * L.m;
    uint16_t *out_dist = best_dist_out ? best_dist_out + (size_t)blockIdx.y * L.m : nullptr;

    uint8_t *base = smem_raw;
    uint4 *s_desc = reinterpret_cast<uint4 *>(base);
    base += (size_t)cap * 32;
    float *s_sx = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    float *s_sy = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    float *s_ex = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    float *s_ey = reinterpret_cast<float *>(base);
    base += (size_t)cap * 4;
    int *s_oct = reinterpret_cast<int *>(base);
    for (int p = tid; p < n; p += kThreads) {
        s_sx[p] = T.sx[p];
        s_sy[p] = T.sy[p];
        s_ex[p] = T.ex[p];
        s_ey[p] = T.ey[p];
        s_oct[p] = T.octave[p];
        uint4 d0, d1;
        load_desc(T.desc + 32 * (size_t)p, d0, d1);
        s_desc[2 * p] = d0;
        s_desc[2 * p + 1] = d1;
    }
    __syncthreads();

    for (int i = i0 + warp; i < i1; i += nwarps) {
        int out = -1;
        unsigned outd = 0xFFFFu;
        bool ok = (L.valid ? L.valid[i] != 0 : true) && (T.skip ? T.skip[i] == 0 : true);
        double su = 0.0, sv = 0.0, eu = 0.0, ev = 0.0;
        unsigned pred = 0;
        if (ok) {
            const double *pw = L.pos_w + 6 * (size_t)i;
            const double S[3] = {pw[0], pw[1], pw[2]}, E[3] = {pw[3], pw[4], pw[5]};
            const Proj ps = reproject(P.cam, T.R, T.t, S), pe = reproject(P.cam, T.R, T.t, E);
            su = ps.u;
            sv = ps.v;
            eu = pe.u;
            ev = pe.v;
            if (!ps.in_image && !pe.in_image) ok = false;  // :341-345
            const double M[3] = {0.5 * (S[0] + E[0]), 0.5 * (S[1] + E[1]), 0.5 * (S[2] + E[2])};
            if (ok && (!ps.in_image || !pe.in_image)) {  // :347-366
                const Proj pm = reproject(P.cam, T.R, T.t, M);
                if (!pm.in_image) ok = false;
            }
            if (ok) {  // :368-392
                const double a0 = S[0] - T.c[0], a1 = S[1] - T.c[1], a2 = S[2] - T.c[2];
                const double b0 = E[0] - T.c[0], b1 = E[1] - T.c[1], b2 = E[2] - T.c[2];
                const double dist_sp = sqrt(a0 * a0 + a1 * a1 + a2 * a2), dist_ep = sqrt(b0 * b0 + b1 * b1 + b2 * b2);
                const double min_d = (double)L.min_d[i], max_d = (double)L.max_d[i];
                if (dist_sp < min_d || max_d < dist_sp || dist_ep < min_d || max_d < dist_ep) ok = false;
                const double m0 = M[0] - T.c[0], m1 = M[1] - T.c[1], m2 = M[2] - T.c[2];
                const double dist_mp = sqrt(m0 * m0 + m1 * m1 + m2 * m2);
                if (ok) pred = (unsigned)predict_level(L.max_raw[i] / (float)dist_mp, P);
            }
        }
        if (ok && n > 0) {
            const float r = P.margin * P.scale_factors[pred];
            // data/common.cc:315-364: the candidate test builds the line from the FLOAT reprojections ...
            const double ax = (double)(float)su, ay = (double)(float)sv, bx = (double)(float)eu, by = (double)(float)ev;
            const double f0 = ay * 1.0 - 1.0 * by, f1 = 1.0 * bx - ax * 1.0, f2 = ax * by - ay * bx;
            const double fden = sqrt(f0 * f0 + f1 * f1);
            // ... and the chi-square gate from the double ones (fuse.cc:417-431)
            const double l0 = sv * 1.0 - 1.0 * ev, l1 = 1.0 * eu - su * 1.0, l2 = su * ev - sv * eu;
            const double lden = sqrt(l0 * l0 + l1 * l1);
            uint4 q0, q1;
            load_desc(L.desc + 32 * (size_t)i, q0, q1);
            unsigned long long best = ~0ull;
            for (int p = lane; p < n; p += 32) {
                const double ksx = (double)s_sx[p], ksy = (double)s_sy[p], kex = (double)s_ex[p], key_ = (double)s_ey[p];
                const float dsp = (float)((ksx * f0 + ksy * f1 + f2) / fden);
                const float dep = (float)((kex * f0 + key_ * f1 + f2) / fden);
                if (fabsf(dsp) > r || fabsf(dep) > r) continue;
                const unsigned sl = (unsigned)s_oct[p];
                if (sl >= (unsigned)P.num_levels) continue;  // _inv_level_sigma_sq_lsd.at() would throw
                const double e_sp = (ksx * l0 + ksy * l1 + l2) / lden;
                const double e_ep = (kex * l0 + key_ * l1 + l2) / lden;
                if ((double)5.99146f < (e_sp * e_sp + e_ep * e_ep) * (double)P.inv_sigma_sq[sl]) continue;
                const unsigned d = (unsigned)hamming256(q0, q1, s_desc[2 * p], s_desc[2 * p + 1]);
                const unsigned long long key = ((unsigned long long)d << 32) | (unsigned)p;
                best = key < best ? key : best;
            }
            best = warp_min_u64(best);
            if (best != ~0ull) {
                const unsigned d = (unsigned)(best >> 32);
                if (d < (unsigned)PLP_MAX_HAMMING_DIST && d <= (unsigned)PLP_HAMMING_DIST_THR_LOW) {
                    out = (int)(best & 0xffffffffull);
                    outd = d;
                }
            }
        }
        if (lane == 0) {
            out_idx[i] = out;
            if (out_dist) out_dist[i] = (uint16_t)outd;
        }
    }
}

}  // namespace

}  // namespace plp
