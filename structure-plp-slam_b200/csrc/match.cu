// match.cu -- 256-bit Hamming matchers (sm_100a).
//
// Replaces match/base.h:43-93, match/projection.cc:37-527, match/robust.cc:257-385 and the
// grid helpers data/common.cc:205-364 of the reference.
//
// Parallelisation of the reference's *sequential greedy* matchers.  Every matcher walks its
// queries in order and skips candidates already claimed by an earlier query.  We run one CTA per
// frame and iterate to the fixed point of
//     choice[q] = best candidate among { c : no q' < q with choice[q'] == c }
// Query q only depends on queries < q, so after round r the first r queries are final and any
// fixed point equals the sequential result; conflicts are rare so 2-4 rounds suffice in practice.
// Candidate traversal order (cell-x, cell-y, insertion -- data/common.cc:275-309) decides '<' ties:
// keypoints are counting-sorted by (cell_x, cell_y, index) into shared memory once per frame, so a
// query scans one contiguous span per grid column of its window in exactly the reference's order
// (the window matcher lives in point_match_kernels.cuh).  Descriptors live in shared memory as
// 2 x uint4; distances are 8 x __popc.
//
// Compiled with -fmad=false: float/double expressions must round exactly like the oracle.
#include "match_kernels.cuh"
#include "match_device.cuh"
#include "point_match_kernels.cuh"
#include "detmath.h"
#include "pack.cuh"

namespace plp {

namespace {

constexpr int kThreads = 512;

// ---------------------------------------------------------------------------------------
// dense Hamming matrix and exact 1-NN
// ---------------------------------------------------------------------------------------
__global__ void hamming_matrix_kernel(const uint8_t *__restrict__ a, int na, const uint8_t *__restrict__ b,
                                      int nb, uint16_t *__restrict__ out) {
    // block = 32 x 8 threads; tile 32 (b) x 32 (a); b-descriptors of the tile in smem
    __shared__ uint4 sb[32][2];
    const int j0 = blockIdx.x * 32, i0 = blockIdx.y * 32;
    const int tx = threadIdx.x, ty = threadIdx.y;
    if (ty < 2 && j0 + tx < nb) sb[tx][ty] = __ldg(reinterpret_cast<const uint4 *>(b + 32 * (size_t)(j0 + tx)) + ty);
    __syncthreads();
    for (int r = ty; r < 32; r += 8) {
        const int i = i0 + r;
        if (i >= na) break;
        uint4 a0, a1;
        load_desc(a + 32 * (size_t)i, a0, a1);
        if (j0 + tx < nb) out[(size_t)i * nb + j0 + tx] = (uint16_t)hamming256(a0, a1, sb[tx][0], sb[tx][1]);
    }
}

__global__ void hamming_nn_kernel(const uint8_t *__restrict__ q, int nq, const uint8_t *__restrict__ t, int nt,
                                  int32_t *__restrict__ nn_idx, uint16_t *__restrict__ nn_dist) {
    // one warp per query; lanes stride the train set; (dist, idx) min via shuffles
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (warp >= nq) return;
    uint4 q0, q1;
    load_desc(q + 32 * (size_t)warp, q0, q1);
    unsigned long long best = ~0ull;
    for (int j = lane; j < nt; j += 32) {
        uint4 t0, t1;
        load_desc(t + 32 * (size_t)j, t0, t1);
        const unsigned long long key = ((unsigned long long)hamming256(q0, q1, t0, t1) << 32) | (unsigned)j;
        best = key < best ? key : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, best, o);
        best = other < best ? other : best;
    }
    if (lane == 0) {
        nn_idx[warp] = nt > 0 ? (int32_t)(best & 0xffffffffu) : -1;
        nn_dist[warp] = nt > 0 ? (uint16_t)(best >> 32) : (uint16_t)0xFFFF;
    }
}

// ---------------------------------------------------------------------------------------
// reprojection pre-pass of match_current_and_last_frames (projection.cc:240-292)
// ---------------------------------------------------------------------------------------
struct Reproj {
    double u, v;
    float x_right;
    bool in_image;
    bool in_front;
};

// camera/perspective.cc:190-209
__device__ __forceinline__ Reproj reproject(const plp_camera &cam, const double *P, const double *X) {
    Reproj r;
    const double pc0 = P[0] * X[0] + P[1] * X[1] + P[2] * X[2] + P[3];
    const double pc1 = P[4] * X[0] + P[5] * X[1] + P[6] * X[2] + P[7];
    const double pc2 = P[8] * X[0] + P[9] * X[1] + P[10] * X[2] + P[11];
    r.u = 0.0;
    r.v = 0.0;
    r.x_right = 0.0f;
    r.in_image = false;
    r.in_front = pc2 > 0.0;
    if (!r.in_front) return r;
    const double z_inv = 1.0 / pc2;
    r.u = cam.fx * pc0 * z_inv + cam.cx;
    r.v = cam.fy * pc1 * z_inv + cam.cy;
    r.x_right = (float)(r.u - cam.focal_x_baseline * z_inv);
    r.in_image = (cam.min_x < r.u && r.u < cam.max_x && cam.min_y < r.v && r.v < cam.max_y);
    return r;
}

__global__ void project_points_kernel(const ProjectJob *__restrict__ jobs, plp_camera cam,
                                      const float *__restrict__ scale_factors, int num_levels, float margin) {
    const ProjectJob &J = jobs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= J.n_last) return;  // also skips disabled jobs (n_last < 0)
    bool valid = J.valid ? (J.valid[i] != 0) : true;
    const int lvl = J.octave[i];
    Reproj r = reproject(cam, J.pose_cw, J.pos_w + 3 * (size_t)i);
    valid = valid && r.in_image;
    J.qx[i] = (float)r.u;
    J.qy[i] = (float)r.v;
    J.qxr[i] = r.x_right;
    J.qradius[i] = margin * scale_factors[lvl];
    int mn, mx;
    if (J.assume_forward) {  // projection.cc:268-273
        mn = lvl;
        mx = num_levels - 1;
    } else if (J.assume_backward) {  // :274-279
        mn = 0;
        mx = lvl;
    } else {  // :280-285
        mn = lvl - 1;
        mx = lvl + 1;
    }
    J.qmin[i] = mn;
    J.qmax[i] = mx;
    J.qvalid[i] = valid ? 1 : 0;
}

// projection.cc:392-470
__global__ void project_lines_kernel(const ProjectJob *__restrict__ jobs, plp_camera cam,
                                     const float *__restrict__ scale_factors, int num_levels, float margin) {
    const ProjectJob &J = jobs[blockIdx.y];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= J.n_last) return;
    bool valid = J.valid ? (J.valid[i] != 0) : true;
    const double *pw = J.pos_w + 6 * (size_t)i;
    const Reproj sp = reproject(cam, J.pose_cw, pw);
    const Reproj ep = reproject(cam, J.pose_cw, pw + 3);
    if (!sp.in_image && !ep.in_image) valid = false;
    if (valid && (!sp.in_image || !ep.in_image)) {
        const double mp[3] = {0.5 * (pw[0] + pw[3]), 0.5 * (pw[1] + pw[4]), 0.5 * (pw[2] + pw[5])};
        const Reproj mid = reproject(cam, J.pose_cw, mp);
        if (!mid.in_image) valid = false;
    }
    const int lvl = J.octave[i];
    J.qx[i] = (float)sp.u;
    J.qy[i] = (float)sp.v;
    J.qxr[i] = sp.x_right;
    J.qx2[i] = (float)ep.u;
    J.qy2[i] = (float)ep.v;
    J.qxr2[i] = ep.x_right;
    J.qradius[i] = margin * scale_factors[lvl];
    int mn, mx;
    if (J.assume_forward) {  // projection.cc:441-447
        mn = lvl;
        mx = num_levels;
    } else if (J.assume_backward) {  // :448-454
        mn = 0;
        mx = lvl + 1;
    } else {  // :455-461
        mn = lvl - 1;
        mx = lvl + 1;
    }
    J.qmin[i] = mn;
    J.qmax[i] = mx;
    J.qvalid[i] = valid ? 1 : 0;
}

// ---------------------------------------------------------------------------------------
// keyline matcher: candidates = linear scan (data/common.cc:315-364)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
    line_match_kernel(const LineMatchJob *__restrict__ jobs, int ratio_test, float lowe_ratio, int rgbd_gate) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const LineMatchJob &J = jobs[blockIdx.x];
    const int tid = threadIdx.x;
    const int n = J.n, m = J.m;
    int *owner_prev = reinterpret_cast<int *>(smem_raw);
    int *owner_next = owner_prev + n;
    int *flags = owner_next + n;  // [0] changed, [1] num matches
    ClaimRounds<kThreads> claims{owner_prev, owner_next, &flags[0], n};
    claims.reset(tid);
    if (tid == 0) flags[1] = 0;
    __syncthreads();
    for (int round = 0; round <= m; ++round) {
        for (int q = tid; q < m; q += kThreads) {
            int choice = -1;
            const bool valid = J.qvalid ? (J.qvalid[q] != 0) : true;
            if (valid) {
                const float margin = J.qradius[q];
                const int min_level = J.qmin[q], max_level = J.qmax[q];
                const bool check_level = (0 < min_level) || (0 <= max_level);
                // proj_line = (x1,y1,1) x (x2,y2,1) in double (data/common.cc:325-327)
                const double ax = J.q_spx[q], ay = J.q_spy[q], bx = J.q_epx[q], by = J.q_epy[q];
                const double l0 = ay * 1.0 - 1.0 * by;
                const double l1 = 1.0 * bx - ax * 1.0;
                const double l2 = ax * by - ay * bx;
                const double den = sqrt(l0 * l0 + l1 * l1);
                uint4 q0, q1;
                load_desc(J.qdesc + 32 * (size_t)q, q0, q1);
                unsigned best = PLP_MAX_HAMMING_DIST, second = PLP_MAX_HAMMING_DIST;
                int best_lvl = -1, second_lvl = -1, best_p = -1;
                for (int p = 0; p < n; ++p) {
                    const float dsp = (float)((J.sx[p] * l0 + J.sy[p] * l1 + l2) / den);
                    const float dep = (float)((J.ex[p] * l0 + J.ey[p] * l1 + l2) / den);
                    if (fabsf(dsp) > margin || fabsf(dep) > margin) continue;
                    if (check_level) {
                        const int oct = J.octave[p];
                        if (oct < min_level) continue;
                        if (max_level > 0 && oct > max_level) continue;
                    }
                    if (J.claimed && J.claimed[p]) continue;
                    if (claims.owned_before(p, q)) continue;
                    if (rgbd_gate && J.xr_sp && J.xr_ep && J.q_xr_sp && J.q_xr_ep) {  // projection.cc:487-500
                        if (J.xr_sp[p] > 0 && J.xr_ep[p] > 0) {
                            const float e_sp = fabsf(J.q_xr_sp[q] - J.xr_sp[p]);
                            const float e_ep = fabsf(J.q_xr_ep[q] - J.xr_ep[p]);
                            if (margin < e_sp || margin < e_ep) continue;
                        }
                    }
                    uint4 d0, d1;
                    load_desc(J.desc + 32 * (size_t)p, d0, d1);
                    const unsigned d = (unsigned)hamming256(q0, q1, d0, d1);
                    const int lvl = J.ratio_level ? J.ratio_level[p] : J.octave[p];
                    if (d < best) {
                        second = best;
                        best = d;
                        second_lvl = best_lvl;
                        best_lvl = lvl;
                        best_p = p;
                    } else if (d < second) {
                        second_lvl = lvl;
                        second = d;
                    }
                }
                if (best_p >= 0 && best <= (J.hamm_thr_p1 ? J.hamm_thr_p1 - 1u : (unsigned)PLP_HAMMING_DIST_THR_HIGH)) {
                    bool ok = true;
                    if (ratio_test && best_lvl == second_lvl && (float)best > lowe_ratio * (float)second) ok = false;
                    if (ok) choice = best_p;
                }
            }
            J.choice[q] = choice;
            if (choice >= 0) claims.claim(choice, q);
        }
        if (claims.settled(tid)) break;
    }
    if (J.matched_out)
        for (int i = tid; i < n; i += kThreads) J.matched_out[i] = -1;
    __syncthreads();
    for (int q = tid; q < m; q += kThreads) {
        const int p = J.choice[q];
        if (p >= 0) {
            atomicAdd(&flags[1], 1);
            if (J.matched_out) J.matched_out[p] = q;
        }
        if (J.best_idx_out) J.best_idx_out[q] = p;
    }
    __syncthreads();
    if (tid == 0 && J.num_matches) *J.num_matches = (uint32_t)flags[1];
}

// ---------------------------------------------------------------------------------------
// robust::brute_force_match (robust.cc:257-385)
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1)
    brute_match_kernel(const BruteJob *__restrict__ jobs, int cap, float lowe_ratio, int check_orientation) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const BruteJob &J = jobs[blockIdx.x];
    const int tid = threadIdx.x;
    const int n1 = J.n_frm, n2 = J.n_kf;
    uint4 *sdesc = reinterpret_cast<uint4 *>(smem_raw);
    int *owner_prev = reinterpret_cast<int *>(smem_raw + (size_t)cap * 32);
    int *owner_next = owner_prev + cap;
    int *hist = owner_next + cap;
    int *flags = hist + kHistLen;  // [0] changed, [1..2] orientation filter counts
    uint8_t *bin_valid = reinterpret_cast<uint8_t *>(flags + 4);
    ClaimRounds<kThreads> claims{owner_prev, owner_next, &flags[0], n1};
    // left to itself the compiler unrolls this copy 16 deep, which costs the whole kernel 128 registers instead of 48
#pragma unroll 4
    for (int i = tid; i < n1; i += kThreads) {
        uint4 d0, d1;
        load_desc(J.frm_desc + 32 * (size_t)i, d0, d1);
        sdesc[2 * i] = d0;
        sdesc[2 * i + 1] = d1;
    }
    claims.reset(tid);
    __syncthreads();
    for (int round = 0; round <= n2; ++round) {
        for (int q = tid; q < n2; q += kThreads) {
            int choice = -1;
            const bool valid = J.kf_valid ? (J.kf_valid[q] != 0) : true;
            if (valid) {
                uint4 q0, q1;
                load_desc(J.kf_desc + 32 * (size_t)q, q0, q1);
                unsigned best = PLP_MAX_HAMMING_DIST, second = PLP_MAX_HAMMING_DIST;
                int best_i = -1;
                for (int i = 0; i < n1; ++i) {
                    if (claims.owned_before(i, q)) continue;  // already_matched_indices_1
                    const unsigned d = (unsigned)hamming256(q0, q1, sdesc[2 * i], sdesc[2 * i + 1]);
                    if (d < best) {
                        second = best;
                        best = d;
                        best_i = i;
                    } else if (d < second) {
                        second = d;
                    }
                }
                // robust.cc:335-349
                if (!(PLP_HAMMING_DIST_THR_LOW < best) && best_i >= 0 && !(lowe_ratio * (float)second < (float)best))
                    choice = best_i;
            }
            J.choice[q] = choice;
            if (choice >= 0) claims.claim(choice, q);
        }
        if (claims.settled(tid)) break;
    }
    for (int i = tid; i < n1; i += kThreads) J.matched_out[i] = -1;
    const bool do_angle = check_orientation && J.frm_angle && J.kf_angle;
    orientation_filter<kThreads>(
        n2, J.choice, do_angle, hist, bin_valid, &flags[1], J.num_matches,
        [&](int q, int i) { return J.frm_angle[i] - J.kf_angle[q]; },
        [&](int q, int i, bool keep) {
            if (keep) J.matched_out[i] = q;
        });
}

// ---------------------------------------------------------------------------------------
// robust::match_for_triangulation (match/robust.cc:43-216)
// ---------------------------------------------------------------------------------------
struct TriJob {
    int n1, n2, num_seq;
    const uint8_t *desc1, *desc2;
    const float *angle1, *angle2;
    const int32_t *octave1;
    const double *bearing1, *bearing2;   // n x 3
    const uint8_t *has_lm2;
    const uint8_t *stereo1, *stereo2;    // 0 <= stereo_x_right; may be null (monocular)
    const int32_t *seq_idx1;             // processing order: keyframe-1 keypoint of step p (landmark-free ones only)
    const int32_t *seq_cbeg, *seq_cend;  // candidate span of step p in cand2 (the keyframe-2 indices of the same BoW node)
    const int32_t *cand2;
    const float *scale_factors1;
    double E[9], epipole[3];
    int32_t *choice;       // num_seq
    int32_t *matched_out;  // n1
    uint32_t *num_matches;
};

// robust.cc:387-406; acos(c) is evaluated as atan2(sqrt((1 - c)(1 + c)), c) with the deterministic kernel of detmath.h
__device__ __forceinline__ bool check_epipolar_constraint(const double *b1, const double *b2, const double *E, float sf1) {
    const double e0 = E[0] * b2[0] + E[1] * b2[1] + E[2] * b2[2];
    const double e1 = E[3] * b2[0] + E[4] * b2[1] + E[5] * b2[2];
    const double e2 = E[6] * b2[0] + E[7] * b2[1] + E[8] * b2[2];
    const double cos_residual = (e0 * b1[0] + e1 * b1[1] + e2 * b1[2]) / sqrt(e0 * e0 + e1 * e1 + e2 * e2);
    const double ac = det_atan2(sqrt((1.0 - cos_residual) * (1.0 + cos_residual)), cos_residual);
    const double residual_rad = 3.14159265358979323846 / 2.0 - fabs(ac);
    const double residual_rad_thr = 0.2 * 3.14159265358979323846 / 180.0;
    return residual_rad < residual_rad_thr * (double)sf1;
}

__global__ void __launch_bounds__(kThreads, 1) triangulation_match_kernel(const TriJob *__restrict__ jobs, int cap2,
                                                                          int check_orientation) {
    extern __shared__ __align__(16) uint8_t smem_raw[];
    const TriJob &J = jobs[blockIdx.x];
    const int tid = threadIdx.x;
    const int n1 = J.n1, n2 = J.n2, P = J.num_seq;
    int *owner_prev = reinterpret_cast<int *>(smem_raw);
    int *owner_next = owner_prev + cap2;
    int *hist = owner_next + cap2;
    int *flags = hist + kHistLen;  // [0] changed, [1..2] orientation filter counts
    uint8_t *bin_valid = reinterpret_cast<uint8_t *>(flags + 4);
    // Sequential semantics: step p takes the best candidate not taken by an earlier step.
    ClaimRounds<kThreads> claims{owner_prev, owner_next, &flags[0], n2};
    claims.reset(tid);
    __syncthreads();
    for (int round = 0; round <= P; ++round) {
        for (int p = tid; p < P; p += kThreads) {
            const int i1 = J.seq_idx1[p];
            uint4 q0, q1;
            load_desc(J.desc1 + 32 * (size_t)i1, q0, q1);
            const double *b1 = J.bearing1 + 3 * (size_t)i1;
            const bool st1 = J.stereo1 ? (J.stereo1[i1] != 0) : false;
            const float sf1 = J.scale_factors1[J.octave1[i1]];
            unsigned best = PLP_HAMMING_DIST_THR_LOW;
            int best_j = -1;
            for (int c = J.seq_cbeg[p]; c < J.seq_cend[p]; ++c) {
                const int j = J.cand2[c];
                if (J.has_lm2[j]) continue;
                if (claims.owned_before(j, p)) continue;  // is_already_matched_in_keyfrm_2
                uint4 d0, d1;
                load_desc(J.desc2 + 32 * (size_t)j, d0, d1);
                const unsigned d = (unsigned)hamming256(q0, q1, d0, d1);
                if (PLP_HAMMING_DIST_THR_LOW < d || best < d) continue;
                const double *b2 = J.bearing2 + 3 * (size_t)j;
                const bool st2 = J.stereo2 ? (J.stereo2[j] != 0) : false;
                if (!st1 && !st2) {
                    const double cos_dist = J.epipole[0] * b2[0] + J.epipole[1] * b2[1] + J.epipole[2] * b2[2];
                    if (0.99862953475 < cos_dist) continue;
                }
                if (check_epipolar_constraint(b1, b2, J.E, sf1)) {
                    best_j = j;
                    best = d;
                }
            }
            J.choice[p] = best_j;
            if (best_j >= 0) claims.claim(best_j, p);
        }
        if (claims.settled(tid)) break;
    }
    for (int i = tid; i < n1; i += kThreads) J.matched_out[i] = -1;
    const bool do_angle = check_orientation && J.angle1 && J.angle2;
    orientation_filter<kThreads>(
        P, J.choice, do_angle, hist, bin_valid, &flags[1], J.num_matches,
        [&](int p, int j) { return J.angle1[J.seq_idx1[p]] - J.angle2[j]; },
        [&](int p, int j, bool keep) {
            if (keep) J.matched_out[J.seq_idx1[p]] = j;
        });
}

// ---------------------------------------------------------------------------------------
// landmark::compute_descriptor / Line::compute_descriptor (data/landmark.cc:181-247, data/landmark_line.cc:215-283):
// the observation whose median Hamming distance to all observations is smallest (first such observation wins).
// One warp per landmark; per row a 257-bin histogram of the distances gives the element of rank floor(0.5 (k - 1)).
// ---------------------------------------------------------------------------------------
constexpr int kMedWarps = 4;
__global__ void __launch_bounds__(kMedWarps * 32) median_descriptor_kernel(const uint8_t *__restrict__ descs,
                                                                             const int32_t *__restrict__ offsets,
                                                                             int num_landmarks,
                                                                             int32_t *__restrict__ best_out) {
    __shared__ int s_hist[kMedWarps][264];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int lm = blockIdx.x * kMedWarps + warp;
    if (lm >= num_landmarks) return;
    const int beg = offsets[lm], k = offsets[lm + 1] - beg;
    if (k <= 0) {
        if (lane == 0) best_out[lm] = -1;
        return;
    }
    int *hist = s_hist[warp];
    const int rank = (int)(0.5 * (double)(k - 1));
    unsigned best_median = PLP_MAX_HAMMING_DIST;
    int best_idx = 0;
    for (int i = 0; i < k; ++i) {
        for (int b = lane; b < 264; b += 32) hist[b] = 0;
        __syncwarp();
        uint4 a0, a1;
        load_desc(descs + 32 * (size_t)(beg + i), a0, a1);
        for (int j = lane; j < k; j += 32) {
            uint4 b0, b1;
            load_desc(descs + 32 * (size_t)(beg + j), b0, b1);
            atomicAdd(&hist[hamming256(a0, a1, b0, b1)], 1);
        }
        __syncwarp();
        // element of rank `rank` in ascending order: first bin whose inclusive prefix exceeds rank
        int cnt[9], local = 0;
#pragma unroll
        for (int q = 0; q < 9; ++q) {
            const int b = lane * 9 + q;
            cnt[q] = b < 257 ? hist[b] : 0;
            local += cnt[q];
        }
        int incl = local;
        for (int off = 1; off < 32; off <<= 1) {
            const int nb = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= off) incl += nb;
        }
        int run = incl - local, med = 0x7fffffff;
#pragma unroll
        for (int q = 0; q < 9; ++q) {
            if (med == 0x7fffffff && run <= rank && rank < run + cnt[q]) med = lane * 9 + q;
            run += cnt[q];
        }
        for (int off = 16; off >= 1; off >>= 1) med = min(med, __shfl_xor_sync(0xffffffffu, med, off));
        if ((unsigned)med < best_median) {
            best_median = (unsigned)med;
            best_idx = i;
        }
        __syncwarp();
    }
    if (lane == 0) best_out[lm] = best_idx;
}

}  // namespace

// ---------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------
plp_status launch_point_match(plp_ctx *ctx, const PointMatchJob *d_jobs, int num_jobs, int max_n,
                              const plp_grid &grid, int ratio_test, float lowe_ratio, int check_orientation) {
    if (num_jobs <= 0) return PLP_OK;
    if (max_n > kMatchMaxPoints) {
        set_error("window matcher: %d keypoints exceed the per-frame capacity %d", max_n, kMatchMaxPoints);
        return PLP_ERR_CAPACITY;
    }
    if (grid.num_rows > 255 || grid.num_cols < 1 || grid.num_cols > 16383 || grid.num_rows < 1) {
        set_error("window matcher: unsupported grid %d x %d", grid.num_cols, grid.num_rows);
        return PLP_ERR_INVALID;
    }
    const int cap = max_n < 64 ? 64 : ((max_n + 63) / 64) * 64;
    const size_t smem = pm::point_smem_bytes(cap, grid.num_cols, grid.num_rows);
    using pm::point_match_kernel;
    PLP_SMEM_OPTIN(point_match_kernel, smem);
    PLP_LAUNCH(ctx, point_match_kernel, num_jobs, pm::kThreads, smem, d_jobs, grid, cap, ratio_test, lowe_ratio,
               check_orientation);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

plp_status launch_line_match(plp_ctx *ctx, const LineMatchJob *d_jobs, int num_jobs, int ratio_test,
                             float lowe_ratio, int rgbd_gate) {
    if (num_jobs <= 0) return PLP_OK;
    // shared memory: 2 owner arrays of the fixed keyline capacity, then the flags
    const size_t smem = (size_t)2 * kLineMaxLines * 4 + 32;
    PLP_SMEM_OPTIN(line_match_kernel, smem);
    PLP_LAUNCH(ctx, line_match_kernel, num_jobs, kThreads, smem, d_jobs, ratio_test, lowe_ratio, rgbd_gate);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

plp_status launch_brute_match(plp_ctx *ctx, const BruteJob *d_jobs, int num_jobs, int max_n_frm, float lowe_ratio,
                              int check_orientation) {
    if (num_jobs <= 0) return PLP_OK;
    if (max_n_frm > kBruteMaxPoints) {
        set_error("brute-force matcher: %d keypoints exceed the capacity %d", max_n_frm, kBruteMaxPoints);
        return PLP_ERR_CAPACITY;
    }
    const int cap = max_n_frm < 64 ? 64 : ((max_n_frm + 63) / 64) * 64;
    const size_t smem = (size_t)cap * 32 + (size_t)cap * 8 + kHistLen * 4 + 16 + 32;
    PLP_SMEM_OPTIN(brute_match_kernel, smem);
    PLP_LAUNCH(ctx, brute_match_kernel, num_jobs, kThreads, smem, d_jobs, cap, lowe_ratio, check_orientation);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

plp_status launch_project_points(plp_ctx *ctx, const ProjectJob *d_jobs, int num_jobs, int max_n,
                                 const plp_camera &cam, const float *d_scale_factors, int num_levels, float margin) {
    if (num_jobs <= 0 || max_n <= 0) return PLP_OK;
    dim3 grid(div_up(max_n, 128), num_jobs);
    PLP_LAUNCH(ctx, project_points_kernel, grid, 128, 0, d_jobs, cam, d_scale_factors, num_levels, margin);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

plp_status launch_project_lines(plp_ctx *ctx, const ProjectJob *d_jobs, int num_jobs, int max_n,
                                const plp_camera &cam, const float *d_scale_factors, int num_levels, float margin) {
    if (num_jobs <= 0 || max_n <= 0) return PLP_OK;
    dim3 grid(div_up(max_n, 128), num_jobs);
    PLP_LAUNCH(ctx, project_lines_kernel, grid, 128, 0, d_jobs, cam, d_scale_factors, num_levels, margin);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

void motion_assumption(const plp_camera &cam, const double *Tc, const double *Tl, int *fwd, int *bwd) {
    // projection.cc:220-238: trans_wc = -R_cw^T t_cw ; trans_lc = R_lw trans_wc + t_lw
    double twc[3];
    for (int r = 0; r < 3; ++r) twc[r] = -(Tc[0 * 4 + r] * Tc[3] + Tc[1 * 4 + r] * Tc[7] + Tc[2 * 4 + r] * Tc[11]);
    const double tlc_z = Tl[8] * twc[0] + Tl[9] * twc[1] + Tl[10] * twc[2] + Tl[11];
    const bool mono = cam.setup_type == 0;
    *fwd = mono ? 0 : (tlc_z > cam.true_baseline);
    *bwd = mono ? 0 : (-tlc_z > cam.true_baseline);
}

}  // namespace plp

// =========================================================================================
// C ABI (host pointers)
// =========================================================================================
using namespace plp;

extern "C" {

// copy a matcher's result array and its match count back, then wait for the stream
static plp_status read_matches(plp_ctx *ctx, int32_t *host_out, const int32_t *dev_out, size_t count,
                               const uint32_t *dev_num, uint32_t *num_out) {
    uint32_t num = 0;
    PLP_CUDA_TRY(cudaMemcpyAsync(host_out, dev_out, count * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(&num, dev_num, 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (num_out) *num_out = num;
    return PLP_OK;
}

// search window of each query, computed on the host in float: radius = margin * scale factor of the query's level,
// levels [level - 1, level + level_span]
static plp_status query_windows(const int32_t *q_level, int m, const float *scale_factors, int num_levels, float margin,
                                int level_span, std::vector<float> &radius, std::vector<int32_t> &qmin,
                                std::vector<int32_t> &qmax) {
    radius.resize(m);
    qmin.resize(m);
    qmax.resize(m);
    for (int i = 0; i < m; ++i) {
        const int lvl = q_level[i];
        PLP_REQUIRE(lvl >= 0 && lvl < num_levels, "scale_level out of range");
        radius[i] = margin * scale_factors[lvl];
        qmin[i] = lvl - 1;
        qmax[i] = lvl + level_span;
    }
    return PLP_OK;
}

plp_status plp_hamming_matrix(plp_ctx *ctx, const uint8_t *a, int na, const uint8_t *b, int nb, uint16_t *dist_out) {
    PLP_REQUIRE(ctx && na >= 0 && nb >= 0, "ctx/na/nb");
    if (na == 0 || nb == 0) return PLP_OK;
    PLP_REQUIRE(a && b && dist_out, "null pointer");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const uint8_t *da, *db;
    uint16_t *dist;
    lay.in(da, a, (size_t)na * 32);
    lay.in(db, b, (size_t)nb * 32);
    lay.out(dist, (size_t)na * nb);
    PLP_TRY(lay.upload(ctx, 0));
    dim3 grid(div_up(nb, 32), div_up(na, 32)), block(32, 8);
    PLP_LAUNCH(ctx, hamming_matrix_kernel, grid, block, 0, da, na, db, nb, dist);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(dist_out, dist, (size_t)na * nb * 2, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

plp_status plp_hamming_nn(plp_ctx *ctx, const uint8_t *query, int nq, const uint8_t *train, int nt, int32_t *nn_idx,
                          uint16_t *nn_dist) {
    PLP_REQUIRE(ctx && nq >= 0 && nt >= 0, "ctx/nq/nt");
    if (nq == 0) return PLP_OK;
    PLP_REQUIRE(query && nn_idx && nn_dist && (train || nt == 0), "null pointer");
    if (nt == 0) {
        for (int i = 0; i < nq; ++i) {
            nn_idx[i] = -1;
            nn_dist[i] = 0xFFFF;
        }
        return PLP_OK;
    }
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const uint8_t *dq, *dt;
    int32_t *di;
    uint16_t *dd;
    lay.in(dq, query, (size_t)nq * 32);
    lay.in(dt, train, (size_t)nt * 32);
    lay.out(di, nq);
    lay.out(dd, nq);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_LAUNCH(ctx, hamming_nn_kernel, div_up(nq * 32, 256), 256, 0, dq, nq, dt, nt, di, dd);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(nn_idx, di, (size_t)nq * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(nn_dist, dd, (size_t)nq * 2, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

// the frame's keypoints as the candidate side of a window-matcher job
static void add_frame_points(Layout &lay, const plp_frame_points &f, PointMatchJob &J) {
    const size_t n = (size_t)f.n;
    J.n = f.n;
    lay.in(J.x, f.x, n);
    lay.in(J.y, f.y, n);
    lay.in(J.octave, f.octave, n);
    lay.in(J.angle, f.angle, n);
    lay.in(J.x_right, f.x_right, n);
    lay.in(J.desc, f.desc, n * 32);
    lay.in(J.claimed, f.claimed, n);
}

plp_status plp_match_frame_and_landmarks(plp_ctx *ctx, const plp_frame_points *frm, const plp_grid *grid,
                                         const float *scale_factors, int num_levels, const plp_landmark_queries *q,
                                         float margin, float lowe_ratio, int32_t *best_idx_out,
                                         uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && frm && grid && scale_factors && q && best_idx_out, "null pointer");
    PLP_REQUIRE(frm->n >= 0 && q->m >= 0 && num_levels > 0, "sizes");
    if (num_matches_out) *num_matches_out = 0;
    if (q->m == 0) return PLP_OK;
    if (frm->n == 0) {
        for (int i = 0; i < q->m; ++i) best_idx_out[i] = -1;
        return PLP_OK;
    }
    PLP_REQUIRE(frm->x && frm->y && frm->octave && frm->desc, "frame arrays");
    PLP_REQUIRE(q->reproj_x && q->reproj_y && q->scale_level && q->desc, "query arrays");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const int m = q->m;
    std::vector<float> radius;
    std::vector<int32_t> qmin, qmax;
    // projection.cc:54-58
    PLP_TRY(query_windows(q->scale_level, m, scale_factors, num_levels, margin, 0, radius, qmin, qmax));
    Layout lay;
    PointMatchJob J;
    memset(&J, 0, sizeof(J));
    plp_frame_points f = *frm;
    f.angle = nullptr;  // no orientation check here: the matcher never reads the frame's angles
    add_frame_points(lay, f, J);
    J.m = m;
    lay.in(J.qx, q->reproj_x, m);
    lay.in(J.qy, q->reproj_y, m);
    lay.in(J.qxr, q->x_right, m);
    lay.in(J.qradius, radius.data(), m);
    lay.in(J.qmin, qmin.data(), m);
    lay.in(J.qmax, qmax.data(), m);
    lay.in(J.qdesc, q->desc, (size_t)m * 32);
    lay.in(J.qvalid, q->valid, m);
    const PointMatchJob *d_job;
    lay.in(d_job, &J, 1);
    lay.out(J.choice, m);
    lay.out(J.best_idx_out, m);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_point_match(ctx, d_job, 1, frm->n, *grid, 1, lowe_ratio, 0));
    return read_matches(ctx, best_idx_out, J.best_idx_out, m, J.num_matches, num_matches_out);
}

plp_status plp_match_current_and_last_frames(plp_ctx *ctx, const plp_frame_points *curr, const plp_grid *grid,
                                             const float *scale_factors, int num_levels, const plp_camera *cam,
                                             const double *pose_cw_curr, const double *pose_cw_last,
                                             const plp_last_frame_points *last, float margin, int check_orientation,
                                             int32_t *matched_last_idx_out, uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && curr && grid && scale_factors && cam && pose_cw_curr && pose_cw_last && last &&
                    matched_last_idx_out,
                "null pointer");
    PLP_REQUIRE(curr->n >= 0 && last->n >= 0 && num_levels > 0, "sizes");
    if (num_matches_out) *num_matches_out = 0;
    for (int i = 0; i < curr->n; ++i) matched_last_idx_out[i] = -1;
    if (curr->n == 0 || last->n == 0) return PLP_OK;
    PLP_REQUIRE(curr->x && curr->y && curr->octave && curr->desc, "frame arrays");
    PLP_REQUIRE(last->pos_w && last->octave && last->desc, "last-frame arrays");
    PLP_REQUIRE(!check_orientation || (curr->angle && last->angle), "angles required for the orientation check");
    for (int i = 0; i < last->n; ++i) PLP_REQUIRE(last->octave[i] >= 0 && last->octave[i] < num_levels, "octave range");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const int m = last->n, n = curr->n;
    Layout lay;
    PointMatchJob J;
    memset(&J, 0, sizeof(J));
    ProjectJob P;
    memset(&P, 0, sizeof(P));
    add_frame_points(lay, *curr, J);
    P.n_last = m;
    lay.in(P.pos_w, last->pos_w, (size_t)m * 3);
    lay.in(P.octave, last->octave, m);
    lay.in(J.qangle, last->angle, m);
    lay.in(J.qdesc, last->desc, (size_t)m * 32);
    lay.in(P.valid, last->valid, m);
    const float *d_sf;
    lay.in(d_sf, scale_factors, num_levels);
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) P.pose_cw[r * 4 + c] = pose_cw_curr[r * 4 + c];
    motion_assumption(*cam, pose_cw_curr, pose_cw_last, &P.assume_forward, &P.assume_backward);
    J.m = m;
    const PointMatchJob *d_job;
    const ProjectJob *d_pjob;
    lay.in(d_job, &J, 1);
    lay.in(d_pjob, &P, 1);
    // the projection pre-pass writes the queries the matcher reads
    lay.out(P.qx, m);
    lay.out(P.qy, m);
    lay.out(P.qxr, m);
    lay.out(P.qradius, m);
    lay.out(P.qmin, m);
    lay.out(P.qmax, m);
    lay.out(P.qvalid, m);
    lay.alias(J.qx, P.qx);
    lay.alias(J.qy, P.qy);
    lay.alias(J.qxr, P.qxr);
    lay.alias(J.qradius, P.qradius);
    lay.alias(J.qmin, P.qmin);
    lay.alias(J.qmax, P.qmax);
    lay.alias(J.qvalid, P.qvalid);
    lay.out(J.choice, m);
    lay.out(J.matched_out, n);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_project_points(ctx, d_pjob, 1, m, *cam, d_sf, num_levels, margin));
    PLP_TRY(launch_point_match(ctx, d_job, 1, n, *grid, 0, 0.0f, check_orientation));
    return read_matches(ctx, matched_last_idx_out, J.matched_out, n, J.num_matches, num_matches_out);
}

// the frame's keylines as the candidate side of a keyline-matcher job
static void add_frame_lines(Layout &lay, const plp_frame_lines &f, LineMatchJob &J) {
    const size_t n = (size_t)f.n;
    J.n = f.n;
    lay.in(J.sx, f.sx, n);
    lay.in(J.sy, f.sy, n);
    lay.in(J.ex, f.ex, n);
    lay.in(J.ey, f.ey, n);
    lay.in(J.octave, f.octave, n);
    lay.in(J.ratio_level, f.ratio_level, n);
    lay.in(J.xr_sp, f.x_right_sp, n);
    lay.in(J.xr_ep, f.x_right_ep, n);
    lay.in(J.desc, f.desc, n * 32);
    lay.in(J.claimed, f.claimed, n);
}

plp_status plp_match_frame_and_landmarks_line(plp_ctx *ctx, const plp_frame_lines *frm, const float *scale_factors_lsd,
                                              int num_levels_lsd, const plp_line_queries *q, float margin,
                                              float lowe_ratio, int32_t *best_idx_out, uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && frm && scale_factors_lsd && q && best_idx_out, "null pointer");
    PLP_REQUIRE(frm->n >= 0 && q->m >= 0 && num_levels_lsd > 0, "sizes");
    PLP_REQUIRE(frm->n <= kLineMaxLines, "keyline capacity 16384");
    if (num_matches_out) *num_matches_out = 0;
    if (q->m == 0) return PLP_OK;
    if (frm->n == 0) {
        for (int i = 0; i < q->m; ++i) best_idx_out[i] = -1;
        return PLP_OK;
    }
    PLP_REQUIRE(frm->sx && frm->sy && frm->ex && frm->ey && frm->octave && frm->desc, "frame arrays");
    PLP_REQUIRE(q->sp_x && q->sp_y && q->ep_x && q->ep_y && q->scale_level && q->desc, "query arrays");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const int m = q->m;
    std::vector<float> radius;
    std::vector<int32_t> qmin, qmax;
    // projection.cc:151-153
    PLP_TRY(query_windows(q->scale_level, m, scale_factors_lsd, num_levels_lsd, margin, 0, radius, qmin, qmax));
    Layout lay;
    LineMatchJob J;
    memset(&J, 0, sizeof(J));
    add_frame_lines(lay, *frm, J);
    J.m = m;
    lay.in(J.q_spx, q->sp_x, m);
    lay.in(J.q_spy, q->sp_y, m);
    lay.in(J.q_epx, q->ep_x, m);
    lay.in(J.q_epy, q->ep_y, m);
    lay.in(J.qradius, radius.data(), m);
    lay.in(J.qmin, qmin.data(), m);
    lay.in(J.qmax, qmax.data(), m);
    lay.in(J.qdesc, q->desc, (size_t)m * 32);
    lay.in(J.qvalid, q->valid, m);
    const LineMatchJob *d_job;
    lay.in(d_job, &J, 1);
    lay.out(J.choice, m);
    lay.out(J.best_idx_out, m);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_line_match(ctx, d_job, 1, 1, lowe_ratio, 0));
    return read_matches(ctx, best_idx_out, J.best_idx_out, m, J.num_matches, num_matches_out);
}

plp_status plp_match_current_and_last_frames_line(plp_ctx *ctx, const plp_frame_lines *curr,
                                                  const float *scale_factors_lsd, int num_levels_lsd,
                                                  const plp_camera *cam, const double *pose_cw_curr,
                                                  const double *pose_cw_last, const plp_last_frame_lines *last,
                                                  float margin, int32_t *matched_last_idx_out,
                                                  uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && curr && scale_factors_lsd && cam && pose_cw_curr && pose_cw_last && last &&
                    matched_last_idx_out,
                "null pointer");
    PLP_REQUIRE(curr->n >= 0 && last->n >= 0 && num_levels_lsd > 0, "sizes");
    PLP_REQUIRE(curr->n <= kLineMaxLines, "keyline capacity 16384");
    if (num_matches_out) *num_matches_out = 0;
    for (int i = 0; i < curr->n; ++i) matched_last_idx_out[i] = -1;
    if (curr->n == 0 || last->n == 0) return PLP_OK;
    PLP_REQUIRE(curr->sx && curr->sy && curr->ex && curr->ey && curr->octave && curr->desc, "frame arrays");
    PLP_REQUIRE(last->pos_w && last->octave && last->desc, "last-frame arrays");
    for (int i = 0; i < last->n; ++i)
        PLP_REQUIRE(last->octave[i] >= 0 && last->octave[i] < num_levels_lsd, "octave range");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const int m = last->n, n = curr->n;
    Layout lay;
    LineMatchJob J;
    memset(&J, 0, sizeof(J));
    ProjectJob P;
    memset(&P, 0, sizeof(P));
    plp_frame_lines f = *curr;
    f.ratio_level = nullptr;  // no ratio test here: the matcher never reads the ratio levels
    add_frame_lines(lay, f, J);
    P.n_last = m;
    lay.in(P.pos_w, last->pos_w, (size_t)m * 6);
    lay.in(P.octave, last->octave, m);
    lay.in(J.qdesc, last->desc, (size_t)m * 32);
    lay.in(P.valid, last->valid, m);
    const float *d_sf;
    lay.in(d_sf, scale_factors_lsd, num_levels_lsd);
    for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 4; ++c) P.pose_cw[r * 4 + c] = pose_cw_curr[r * 4 + c];
    motion_assumption(*cam, pose_cw_curr, pose_cw_last, &P.assume_forward, &P.assume_backward);
    J.m = m;
    const LineMatchJob *d_job;
    const ProjectJob *d_pjob;
    lay.in(d_job, &J, 1);
    lay.in(d_pjob, &P, 1);
    // the projection pre-pass writes the queries the matcher reads
    lay.out(P.qx, m);
    lay.out(P.qy, m);
    lay.out(P.qxr, m);
    lay.out(P.qx2, m);
    lay.out(P.qy2, m);
    lay.out(P.qxr2, m);
    lay.out(P.qradius, m);
    lay.out(P.qmin, m);
    lay.out(P.qmax, m);
    lay.out(P.qvalid, m);
    lay.alias(J.q_spx, P.qx);
    lay.alias(J.q_spy, P.qy);
    lay.alias(J.q_xr_sp, P.qxr);
    lay.alias(J.q_epx, P.qx2);
    lay.alias(J.q_epy, P.qy2);
    lay.alias(J.q_xr_ep, P.qxr2);
    lay.alias(J.qradius, P.qradius);
    lay.alias(J.qmin, P.qmin);
    lay.alias(J.qmax, P.qmax);
    lay.alias(J.qvalid, P.qvalid);
    lay.out(J.choice, m);
    lay.out(J.matched_out, n);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_project_lines(ctx, d_pjob, 1, m, *cam, d_sf, num_levels_lsd, margin));
    PLP_TRY(launch_line_match(ctx, d_job, 1, 0, 0.0f, cam->setup_type == 2));
    return read_matches(ctx, matched_last_idx_out, J.matched_out, n, J.num_matches, num_matches_out);
}

plp_status plp_match_frame_and_keyframe(plp_ctx *ctx, const plp_frame_points *frm, const plp_grid *grid,
                                        const float *scale_factors, int num_levels, const plp_landmark_queries *q,
                                        const float *q_angle, float margin, unsigned hamm_dist_thr, int check_orientation,
                                        int32_t *matched_kf_idx_out, uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && frm && grid && scale_factors && q && matched_kf_idx_out, "null pointer");
    PLP_REQUIRE(frm->n >= 0 && q->m >= 0 && num_levels > 0, "sizes");
    if (num_matches_out) *num_matches_out = 0;
    for (int i = 0; i < frm->n; ++i) matched_kf_idx_out[i] = -1;
    if (frm->n == 0 || q->m == 0) return PLP_OK;
    PLP_REQUIRE(frm->x && frm->y && frm->octave && frm->desc, "frame arrays");
    PLP_REQUIRE(q->reproj_x && q->reproj_y && q->scale_level && q->desc, "query arrays");
    PLP_REQUIRE(!check_orientation || (frm->angle && q_angle), "angles required for the orientation check");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const int m = q->m, n = frm->n;
    std::vector<float> radius;
    std::vector<int32_t> qmin, qmax;
    // projection.cc:586-588
    PLP_TRY(query_windows(q->scale_level, m, scale_factors, num_levels, margin, 1, radius, qmin, qmax));
    Layout lay;
    PointMatchJob J;
    memset(&J, 0, sizeof(J));
    plp_frame_points f = *frm;
    f.x_right = nullptr;  // no stereo gate in match_frame_and_keyframe
    add_frame_points(lay, f, J);
    J.m = m;
    lay.in(J.qx, q->reproj_x, m);
    lay.in(J.qy, q->reproj_y, m);
    lay.in(J.qradius, radius.data(), m);
    lay.in(J.qmin, qmin.data(), m);
    lay.in(J.qmax, qmax.data(), m);
    lay.in(J.qangle, q_angle, m);
    lay.in(J.qdesc, q->desc, (size_t)m * 32);
    lay.in(J.qvalid, q->valid, m);
    J.hamm_thr_p1 = hamm_dist_thr + 1u;
    const PointMatchJob *d_job;
    lay.in(d_job, &J, 1);
    lay.out(J.choice, m);
    lay.out(J.matched_out, n);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_point_match(ctx, d_job, 1, n, *grid, 0, 0.0f, check_orientation));
    return read_matches(ctx, matched_kf_idx_out, J.matched_out, n, J.num_matches, num_matches_out);
}

plp_status plp_match_frame_and_keyframe_line(plp_ctx *ctx, const plp_frame_lines *frm, const float *scale_factors_lsd,
                                             int num_levels_lsd, const plp_line_queries *q, float margin,
                                             unsigned hamm_dist_thr, int32_t *matched_kf_idx_out,
                                             uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && frm && scale_factors_lsd && q && matched_kf_idx_out, "null pointer");
    PLP_REQUIRE(frm->n >= 0 && q->m >= 0 && num_levels_lsd > 0, "sizes");
    PLP_REQUIRE(frm->n <= kLineMaxLines, "keyline capacity 16384");
    if (num_matches_out) *num_matches_out = 0;
    for (int i = 0; i < frm->n; ++i) matched_kf_idx_out[i] = -1;
    if (frm->n == 0 || q->m == 0) return PLP_OK;
    PLP_REQUIRE(frm->sx && frm->sy && frm->ex && frm->ey && frm->octave && frm->desc, "frame arrays");
    PLP_REQUIRE(q->sp_x && q->sp_y && q->ep_x && q->ep_y && q->scale_level && q->desc, "query arrays");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const int m = q->m, n = frm->n;
    std::vector<float> radius;
    std::vector<int32_t> qmin, qmax;
    // projection.cc:734-737
    PLP_TRY(query_windows(q->scale_level, m, scale_factors_lsd, num_levels_lsd, margin, 1, radius, qmin, qmax));
    Layout lay;
    LineMatchJob J;
    memset(&J, 0, sizeof(J));
    plp_frame_lines f = *frm;
    f.ratio_level = nullptr;  // no ratio test here: the matcher never reads the ratio levels
    add_frame_lines(lay, f, J);
    J.m = m;
    lay.in(J.q_spx, q->sp_x, m);
    lay.in(J.q_spy, q->sp_y, m);
    lay.in(J.q_epx, q->ep_x, m);
    lay.in(J.q_epy, q->ep_y, m);
    lay.in(J.qradius, radius.data(), m);
    lay.in(J.qmin, qmin.data(), m);
    lay.in(J.qmax, qmax.data(), m);
    lay.in(J.qdesc, q->desc, (size_t)m * 32);
    lay.in(J.qvalid, q->valid, m);
    J.hamm_thr_p1 = hamm_dist_thr + 1u;
    const LineMatchJob *d_job;
    lay.in(d_job, &J, 1);
    lay.out(J.choice, m);
    lay.out(J.matched_out, n);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_line_match(ctx, d_job, 1, 0, 0.0f, 0));
    return read_matches(ctx, matched_kf_idx_out, J.matched_out, n, J.num_matches, num_matches_out);
}

plp_status plp_match_brute_force(plp_ctx *ctx, const uint8_t *frm_desc, const float *frm_angle, int n_frm,
                                 const uint8_t *kf_desc, const float *kf_angle, const uint8_t *kf_valid, int n_kf,
                                 float lowe_ratio, int check_orientation, int32_t *matched_kf_idx_in_frm_out,
                                 uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && matched_kf_idx_in_frm_out, "null pointer");
    PLP_REQUIRE(n_frm >= 0 && n_kf >= 0, "sizes");
    if (num_matches_out) *num_matches_out = 0;
    for (int i = 0; i < n_frm; ++i) matched_kf_idx_in_frm_out[i] = -1;
    if (n_frm == 0 || n_kf == 0) return PLP_OK;
    PLP_REQUIRE(frm_desc && kf_desc, "descriptors");
    PLP_REQUIRE(!check_orientation || (frm_angle && kf_angle), "angles required for the orientation check");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    BruteJob J;
    memset(&J, 0, sizeof(J));
    J.n_frm = n_frm;
    lay.in(J.frm_desc, frm_desc, (size_t)n_frm * 32);
    lay.in(J.frm_angle, frm_angle, n_frm);
    J.n_kf = n_kf;
    lay.in(J.kf_desc, kf_desc, (size_t)n_kf * 32);
    lay.in(J.kf_angle, kf_angle, n_kf);
    lay.in(J.kf_valid, kf_valid, n_kf);
    const BruteJob *d_job;
    lay.in(d_job, &J, 1);
    lay.out(J.choice, n_kf);
    lay.out(J.matched_out, n_frm);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(launch_brute_match(ctx, d_job, 1, n_frm, lowe_ratio, check_orientation));
    return read_matches(ctx, matched_kf_idx_in_frm_out, J.matched_out, n_frm, J.num_matches, num_matches_out);
}

plp_status plp_match_for_triangulation(plp_ctx *ctx, const plp_keyframe_points *kf1, const plp_keyframe_points *kf2,
                                       const plp_bow_feature_vector *fv1, const plp_bow_feature_vector *fv2,
                                       const double *E_12, const double *epipole_bearing_in_2, const float *scale_factors_1,
                                       int num_levels, int check_orientation, int32_t *matched_idx2_in_1_out,
                                       uint32_t *num_matches_out) {
    PLP_REQUIRE(ctx && kf1 && kf2 && fv1 && fv2 && E_12 && epipole_bearing_in_2 && scale_factors_1 && matched_idx2_in_1_out,
                "null pointer");
    PLP_REQUIRE(kf1->n >= 0 && kf2->n >= 0 && num_levels > 0 && fv1->num_nodes >= 0 && fv2->num_nodes >= 0, "sizes");
    if (num_matches_out) *num_matches_out = 0;
    for (int i = 0; i < kf1->n; ++i) matched_idx2_in_1_out[i] = -1;
    if (kf1->n == 0 || kf2->n == 0 || fv1->num_nodes == 0 || fv2->num_nodes == 0) return PLP_OK;
    PLP_REQUIRE(kf1->desc && kf1->octave && kf1->bearings && kf1->has_landmark, "keyframe 1 arrays");
    PLP_REQUIRE(kf2->desc && kf2->bearings && kf2->has_landmark, "keyframe 2 arrays");
    PLP_REQUIRE(!check_orientation || (kf1->angle && kf2->angle), "angles required for the orientation check");
    PLP_REQUIRE(fv1->node_ids && fv1->offsets && fv1->indices && fv2->node_ids && fv2->offsets && fv2->indices,
                "feature vectors");
    PLP_REQUIRE(kf2->n <= 24000, "keyframe 2 keypoint capacity 24000");
    // merge-join of the two (ascending) feature vectors, robust.cc:78-199: processing order and candidate spans
    std::vector<int32_t> seq_idx1, seq_cbeg, seq_cend, cand2;
    int a = 0, b = 0;
    while (a < fv1->num_nodes && b < fv2->num_nodes) {
        if (fv1->node_ids[a] == fv2->node_ids[b]) {
            const int cb = (int)cand2.size();
            for (int k = fv2->offsets[b]; k < fv2->offsets[b + 1]; ++k) {
                PLP_REQUIRE(fv2->indices[k] < (uint32_t)kf2->n, "feature vector index out of range");
                cand2.push_back((int32_t)fv2->indices[k]);
            }
            const int ce = (int)cand2.size();
            for (int k = fv1->offsets[a]; k < fv1->offsets[a + 1]; ++k) {
                const uint32_t i1 = fv1->indices[k];
                PLP_REQUIRE(i1 < (uint32_t)kf1->n, "feature vector index out of range");
                PLP_REQUIRE(kf1->octave[i1] >= 0 && kf1->octave[i1] < num_levels, "octave range");
                if (kf1->has_landmark[i1]) continue;  // robust.cc:99-103
                seq_idx1.push_back((int32_t)i1);
                seq_cbeg.push_back(cb);
                seq_cend.push_back(ce);
            }
            ++a;
            ++b;
        } else if (fv1->node_ids[a] < fv2->node_ids[b]) {
            ++a;  // lower_bound(itr_2->first) on an ascending map == skip the smaller ids
        } else {
            ++b;
        }
    }
    const int P = (int)seq_idx1.size();
    if (P == 0) return PLP_OK;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t n1 = kf1->n, n2 = kf2->n;
    std::vector<uint8_t> st1(n1, 0), st2(n2, 0);
    if (kf1->x_right)
        for (size_t i = 0; i < n1; ++i) st1[i] = 0 <= kf1->x_right[i];
    if (kf2->x_right)
        for (size_t i = 0; i < n2; ++i) st2[i] = 0 <= kf2->x_right[i];
    Layout lay;
    TriJob J;
    memset(&J, 0, sizeof(J));
    J.n1 = (int)n1;
    J.n2 = (int)n2;
    J.num_seq = P;
    lay.in(J.desc1, kf1->desc, n1 * 32);
    lay.in(J.desc2, kf2->desc, n2 * 32);
    lay.in(J.angle1, kf1->angle, n1);
    lay.in(J.angle2, kf2->angle, n2);
    lay.in(J.octave1, kf1->octave, n1);
    lay.in(J.bearing1, kf1->bearings, n1 * 3);
    lay.in(J.bearing2, kf2->bearings, n2 * 3);
    lay.in(J.has_lm2, kf2->has_landmark, n2);
    lay.in(J.stereo1, st1.data(), n1);
    lay.in(J.stereo2, st2.data(), n2);
    lay.in(J.seq_idx1, seq_idx1.data(), P);
    lay.in(J.seq_cbeg, seq_cbeg.data(), P);
    lay.in(J.seq_cend, seq_cend.data(), P);
    lay.in(J.cand2, cand2.data(), cand2.size());
    lay.in(J.scale_factors1, scale_factors_1, num_levels);
    for (int k = 0; k < 9; ++k) J.E[k] = E_12[k];
    for (int k = 0; k < 3; ++k) J.epipole[k] = epipole_bearing_in_2[k];
    const TriJob *d_job;
    lay.in(d_job, &J, 1);
    lay.out(J.choice, P);
    lay.out(J.matched_out, n1);
    lay.out(J.num_matches, 1);
    PLP_TRY(lay.upload(ctx, 0));
    const size_t smem = (size_t)n2 * 8 + (kHistLen + 4) * 4 + kHistLen + 16;
    PLP_SMEM_OPTIN(triangulation_match_kernel, smem);
    PLP_LAUNCH(ctx, triangulation_match_kernel, 1, kThreads, smem, d_job, (int)n2, check_orientation);
    PLP_CHECK_LAUNCH();
    return read_matches(ctx, matched_idx2_in_1_out, J.matched_out, n1, J.num_matches, num_matches_out);
}

plp_status plp_landmark_compute_descriptor_batch(plp_ctx *ctx, const uint8_t *descs, const int32_t *offsets,
                                                 int num_landmarks, int32_t *best_idx_out) {
    PLP_REQUIRE(ctx && offsets && best_idx_out, "null pointer");
    PLP_REQUIRE(num_landmarks >= 0, "sizes");
    if (num_landmarks == 0) return PLP_OK;
    const int total = offsets[num_landmarks];
    PLP_REQUIRE(offsets[0] == 0 && total >= 0 && (total == 0 || descs), "offsets");
    for (int i = 0; i < num_landmarks; ++i) PLP_REQUIRE(offsets[i] <= offsets[i + 1], "offsets must ascend");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const uint8_t *dd;
    const int32_t *doff;
    int32_t *dbest;
    lay.in(dd, descs, (size_t)total * 32);
    lay.in(doff, offsets, (size_t)num_landmarks + 1);
    lay.out(dbest, num_landmarks);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_LAUNCH(ctx, median_descriptor_kernel, div_up(num_landmarks, kMedWarps), kMedWarps * 32, 0, dd, doff,
               num_landmarks, dbest);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(best_idx_out, dbest, (size_t)num_landmarks * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

}  // extern "C"
