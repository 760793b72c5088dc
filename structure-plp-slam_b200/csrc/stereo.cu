// stereo.cu -- match::stereo::compute (match/stereo.cc:45-302) for batches of rectified stereo frames, sm_100a.
//
// One CTA per frame.  The right keypoints (row band, x, octave, 256-bit descriptor) are staged in shared memory once;
// a warp owns one left keypoint at a time: lanes scan the right keypoints in ascending index order (the order of the
// reference's per-row candidate lists), the 256-bit Hamming distance is 8 x __popc, and the warp minimum of
// (distance << 16 | index) is exactly the reference's "first strictly smaller distance wins".  The 11 x 11 L1 patch
// slide (11 offsets) reads the image pyramids the two ORB handles keep in HBM (orb_extractor::image_pyramid_,
// frame.cc:475); all patch sums are integers.  The final "reject above 2 x median correlation" needs the element of
// rank n/2 of the (correlation, index) pairs: a rank count in shared memory.
#include <vector>

#include "common.cuh"
#include "pack.cuh"

using namespace plp;

namespace {

constexpr int kThreads = 512;
constexpr unsigned kHammThr = (PLP_HAMMING_DIST_THR_HIGH + PLP_HAMMING_DIST_THR_LOW) / 2;  // stereo.h:126
constexpr int kMaxLevels = 16;
constexpr unsigned kFull = 0xffffffffu;

struct StereoLevel {
    const uint8_t *left, *right;  // frame 0
    size_t step_l, step_r, stride_l, stride_r;  // row pitch, frame stride
    int w, h;
};

struct StereoDev {
    int num_levels, cap, rows;
    StereoLevel lv[kMaxLevels];
    float scale_factors[kMaxLevels], inv_scale_factors[kMaxLevels];
    float fxb, max_disp;
    const plp_keypoint *kp_l, *kp_r;
    const uint8_t *desc_l, *desc_r;
    const int32_t *n_l, *n_r;
    float *x_right, *depth;
    int32_t *best_right;  // optional parity tap
};

__global__ void __launch_bounds__(kThreads, 1) stereo_kernel(StereoDev D) {
    extern __shared__ uint4 s_dyn[];
    // layout: desc_r [cap][2 x uint4] | band [cap] short2 | xr [cap] float | oct [cap] int8 | corr [cap] int
    uint4 *s_desc = s_dyn;
    short2 *s_band = reinterpret_cast<short2 *>(s_desc + 2 * (size_t)D.cap);
    float *s_x = reinterpret_cast<float *>(s_band + D.cap);
    int *s_corr = reinterpret_cast<int *>(s_x + D.cap);
    int8_t *s_oct = reinterpret_cast<int8_t *>(s_corr + D.cap);
    __shared__ int s_nvalid, s_median;
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nl = D.n_l[b], nr = D.n_r[b];
    const plp_keypoint *kpl = D.kp_l + (size_t)b * D.cap, *kpr = D.kp_r + (size_t)b * D.cap;
    const uint4 *dl = reinterpret_cast<const uint4 *>(D.desc_l + (size_t)b * D.cap * 32);
    const uint4 *dr = reinterpret_cast<const uint4 *>(D.desc_r + (size_t)b * D.cap * 32);
    float *xr_out = D.x_right + (size_t)b * D.cap, *dp_out = D.depth + (size_t)b * D.cap;
    for (int i = tid; i < nr; i += kThreads) {
        const plp_keypoint k = kpr[i];
        const float r = 2.0f * D.scale_factors[k.octave];  // get_right_keypoint_indices_in_each_row(2.0)
        s_band[i] = make_short2((short)cv_floor((double)(k.y - r)), (short)cv_ceil((double)(k.y + r)));
        s_x[i] = k.x;
        s_oct[i] = (int8_t)k.octave;
        s_desc[2 * i] = dr[2 * i];
        s_desc[2 * i + 1] = dr[2 * i + 1];
    }
    for (int i = tid; i < nl; i += kThreads) {
        s_corr[i] = -1;
        xr_out[i] = -1.0f;
        dp_out[i] = -1.0f;
        if (D.best_right) D.best_right[(size_t)b * D.cap + i] = -1;
    }
    if (tid == 0) s_nvalid = 0;
    __syncthreads();
    for (int il = warp; il < nl; il += kThreads / 32) {
        const plp_keypoint kl = kpl[il];
        const int lvl = kl.octave;
        const int row = (int)(size_t)kl.y;
        const float min_x_right = kl.x - D.max_disp, max_x_right = kl.x - 0.0f;
        if (max_x_right < 0) continue;
        const uint4 a0 = dl[2 * il], a1 = dl[2 * il + 1];
        unsigned best = 0xffffffffu;
        for (int i0 = 0; i0 < nr; i0 += 32) {
            const int ir = i0 + lane;
            if (ir < nr) {
                const short2 bd = s_band[ir];
                const int oc = s_oct[ir];
                const float x = s_x[ir];
                if (row >= bd.x && row <= bd.y && !(oc < lvl - 1 || oc > lvl + 1) && !(x < min_x_right || max_x_right < x)) {
                    const unsigned d = (unsigned)hamming256(a0, a1, s_desc[2 * ir], s_desc[2 * ir + 1]);
                    best = min(best, (d << 16) | (unsigned)ir);
                }
            }
        }
        best = __reduce_min_sync(kFull, best);
        if (best == 0xffffffffu || (best >> 16) >= kHammThr) continue;
        const int ir = (int)(best & 0xffff);
        if (D.best_right && lane == 0) D.best_right[(size_t)b * D.cap + il] = ir;
        // compute_subpixel_disparity (stereo.cc:226-299)
        const float x_right = s_x[ir];
        const float isf = D.inv_scale_factors[lvl];
        const int sxl = cv_round_f(kl.x * isf), syl = cv_round_f(kl.y * isf), sxr = cv_round_f(x_right * isf);
        constexpr int win = 5, slide = 5;
        const StereoLevel &V = D.lv[lvl];
        if (sxr - slide - win < 0 || V.w <= sxr + slide + win) continue;
        const uint8_t *L = V.left + (size_t)b * V.stride_l, *R = V.right + (size_t)b * V.stride_r;
        const int lc = L[(size_t)syl * V.step_l + sxl];
        // each lane owns up to four of the 121 patch pixels
        int lv4[4], dy4[4], dx4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int p = lane + 32 * q;
            dy4[q] = p / 11 - win;
            dx4[q] = p - (p / 11) * 11 - win;
            lv4[q] = p < 121 ? (int)L[(size_t)(syl + dy4[q]) * V.step_l + sxl + dx4[q]] - lc : 0;
        }
        float best_corr = 4294967295.0f;  // UINT_MAX as float
        int best_off = 0;
        float c_prev = 0.f, c_best_m1 = 0.f, c_best_p1 = 0.f, c_best = 0.f;
        bool want_next = false;
        for (int off = -slide; off <= slide; ++off) {
            const int rc = R[(size_t)syl * V.step_r + sxr + off];
            int sum = 0;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                if (lane + 32 * q < 121) {
                    const int rv = (int)R[(size_t)(syl + dy4[q]) * V.step_r + sxr + off + dx4[q]] - rc;
                    sum += abs(lv4[q] - rv);
                }
            }
            sum = __reduce_add_sync(kFull, sum);
            const float c = (float)sum;
            if (want_next) {
                c_best_p1 = c;
                want_next = false;
            }
            if (c < best_corr) {
                best_corr = c;
                best_off = off;
                c_best = c;
                c_best_m1 = c_prev;
                want_next = true;
            }
            c_prev = c;
        }
        if (best_off == -slide || best_off == slide) continue;
        const float c1 = c_best_m1, c2 = c_best, c3 = c_best_p1;
        const float x_delta = (float)((double)(c1 - c3) / (2.0 * (double)(c1 + c3) - 4.0 * (double)c2));
        if ((double)x_delta < -1.0 || 1.0 < (double)x_delta) continue;
        float best_x_right = D.scale_factors[lvl] * ((float)(sxr + best_off) + x_delta);
        float best_disp = kl.x - best_x_right;
        if (best_disp < 0.0f || D.max_disp <= best_disp) continue;
        if (best_disp <= 0.0f) {
            best_disp = 0.01f;
            best_x_right = kl.x - best_disp;
        }
        if (lane == 0) {
            dp_out[il] = D.fxb / best_disp;
            xr_out[il] = best_x_right;
            s_corr[il] = (int)best_corr;
            atomicAdd(&s_nvalid, 1);
        }
    }
    __syncthreads();
    // median of the (correlation, index) pairs: the element of rank n/2 in ascending order (stereo.cc:124-131)
    const int nv = s_nvalid;
    if (nv == 0) return;
    const int k = nv / 2;
    for (int i = tid; i < nl; i += kThreads) {
        const int c = s_corr[i];
        if (c < 0) continue;
        int rank = 0;
        for (int j = 0; j < nl; ++j) {
            const int cj = s_corr[j];
            rank += (cj >= 0) && (cj < c || (cj == c && j < i));
        }
        if (rank == k) s_median = c;
    }
    __syncthreads();
    const float thr = (float)(2.0 * (double)(float)s_median);
    for (int i = tid; i < nl; i += kThreads) {
        const int c = s_corr[i];
        if (c >= 0 && thr < (float)c) {
            xr_out[i] = -1.0f;
            dp_out[i] = -1.0f;
        }
    }
}

size_t stereo_smem(int cap) { return (size_t)cap * (32 + 4 + 4 + 4 + 1) + 16; }

plp_status fill_levels(const plp_orb *left, const plp_orb *right, int batch, StereoDev &D) {
    for (int l = 0; l < D.num_levels; ++l) {
        plp_image_view a, a1, c, c1;
        PLP_TRY(plp_orb_get_pyramid(left, 0, l, &a));
        PLP_TRY(plp_orb_get_pyramid(right, 0, l, &c));
        StereoLevel &V = D.lv[l];
        V.left = a.data;
        V.right = c.data;
        V.step_l = a.step;
        V.step_r = c.step;
        V.w = a.cols;
        V.h = a.rows;
        V.stride_l = V.stride_r = 0;
        if (batch > 1) {
            PLP_TRY(plp_orb_get_pyramid(left, 1, l, &a1));
            PLP_TRY(plp_orb_get_pyramid(right, 1, l, &c1));
            V.stride_l = (size_t)(a1.data - a.data);
            V.stride_r = (size_t)(c1.data - c.data);
        }
        PLP_REQUIRE(a.rows == c.rows && a.cols == c.cols, "left / right pyramids differ in size");
    }
    return PLP_OK;
}

}  // namespace

extern "C" {

plp_status plp_stereo_compute_batch_dev(plp_ctx *ctx, const plp_orb *left, const plp_orb *right, int batch,
                                        const plp_keypoint *d_kp_l, const uint8_t *d_desc_l, const int32_t *d_n_l,
                                        const plp_keypoint *d_kp_r, const uint8_t *d_desc_r, const int32_t *d_n_r,
                                        float focal_x_baseline, float true_baseline, float *d_x_right_out,
                                        float *d_depth_out, int32_t *d_best_right_out) {
    PLP_REQUIRE(ctx && left && right && d_kp_l && d_desc_l && d_n_l && d_kp_r && d_desc_r && d_n_r && d_x_right_out &&
                    d_depth_out,
                "null pointer");
    PLP_REQUIRE(batch >= 1 && true_baseline > 0.f, "batch / baseline");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    StereoDev D;
    memset(&D, 0, sizeof(D));
    D.cap = plp_orb_capacity(left);
    PLP_REQUIRE(D.cap == plp_orb_capacity(right) && D.cap < 32768, "left / right extractors differ");
    uint32_t nk[kMaxLevels];
    float ls[kMaxLevels], ils[kMaxLevels];
    plp_image_view v0;
    int L = 0;
    while (L < kMaxLevels && plp_orb_get_pyramid(left, 0, L, &v0) == PLP_OK) ++L;
    PLP_REQUIRE(L >= 1, "no pyramid: run the extraction first");
    D.num_levels = L;
    PLP_TRY(plp_orb_get_tables(left, D.scale_factors, D.inv_scale_factors, ls, ils, nk));
    PLP_TRY(fill_levels(left, right, batch, D));
    D.rows = D.lv[0].h;
    D.fxb = focal_x_baseline;
    D.max_disp = focal_x_baseline / true_baseline;  // stereo.cc:42
    D.kp_l = d_kp_l;
    D.kp_r = d_kp_r;
    D.desc_l = d_desc_l;
    D.desc_r = d_desc_r;
    D.n_l = d_n_l;
    D.n_r = d_n_r;
    D.x_right = d_x_right_out;
    D.depth = d_depth_out;
    D.best_right = d_best_right_out;
    const size_t smem = stereo_smem(D.cap);
    PLP_SMEM_OPTIN(stereo_kernel, smem);
    PLP_LAUNCH(ctx, stereo_kernel, batch, kThreads, smem, D);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

plp_status plp_stereo_compute(plp_ctx *ctx, const plp_orb *left, const plp_orb *right, const plp_keypoint *kp_l,
                              const uint8_t *desc_l, int n_l, const plp_keypoint *kp_r, const uint8_t *desc_r, int n_r,
                              float focal_x_baseline, float true_baseline, float *x_right_out, float *depths_out,
                              int32_t *best_right_out) {
    PLP_REQUIRE(ctx && left && right && x_right_out && depths_out, "null pointer");
    PLP_REQUIRE(n_l >= 0 && n_r >= 0, "sizes");
    for (int i = 0; i < n_l; ++i) {
        x_right_out[i] = -1.0f;
        depths_out[i] = -1.0f;
        if (best_right_out) best_right_out[i] = -1;
    }
    if (n_l == 0 || n_r == 0) return PLP_OK;
    PLP_REQUIRE(kp_l && desc_l && kp_r && desc_r, "null pointer");
    const int cap = plp_orb_capacity(left);
    PLP_REQUIRE(n_l <= cap && n_r <= cap, "more keypoints than the extractor's capacity");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const int32_t n2[2] = {n_l, n_r};
    const plp_keypoint *dkl, *dkr;
    const uint8_t *ddl, *ddr;
    const int32_t *dn;
    float *dx, *dd;
    int32_t *db;
    lay.in(dkl, kp_l, n_l);
    lay.in(dkr, kp_r, n_r);
    lay.in(ddl, desc_l, (size_t)n_l * 32);
    lay.in(ddr, desc_r, (size_t)n_r * 32);
    lay.in(dn, n2, 2);
    lay.out(dx, n_l);
    lay.out(dd, n_l);
    lay.out(db, n_l);
    PLP_TRY(lay.upload(ctx, 3));
    PLP_TRY(plp_stereo_compute_batch_dev(ctx, left, right, 1, dkl, ddl, dn, dkr, ddr, dn + 1, focal_x_baseline,
                                         true_baseline, dx, dd, db));
    cudaStream_t s = ctx->stream;
    PLP_CUDA_TRY(cudaMemcpyAsync(x_right_out, dx, (size_t)n_l * 4, cudaMemcpyDeviceToHost, s));
    PLP_CUDA_TRY(cudaMemcpyAsync(depths_out, dd, (size_t)n_l * 4, cudaMemcpyDeviceToHost, s));
    if (best_right_out) PLP_CUDA_TRY(cudaMemcpyAsync(best_right_out, db, (size_t)n_l * 4, cudaMemcpyDeviceToHost, s));
    PLP_CUDA_TRY(cudaStreamSynchronize(s));
    return PLP_OK;
}

}  // extern "C"
