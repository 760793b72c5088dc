// fuse.cu -- match::fuse search kernels (sm_100a).
//
// Replaces the per-landmark search of match/fuse.cc:40-151 (detect_duplication), :153-300 (replace_duplication) and
// :304-503 (replace_duplication_line) of the reference.  Unlike the projection matchers, fuse.cc has no "skip keypoints
// claimed by an earlier landmark": every landmark's best keypoint depends only on the landmark and on the target
// keyframe's features, so a (target keyframe x landmark) batch is embarrassingly parallel -- grid = (landmark chunks,
// targets), one WARP per landmark.  Only the effects (add_observation / replace) are sequential; they stay in the adapter.
//
// Exactness: reprojection, the distance / viewing-angle gates and the chi-square gates are evaluated in the reference's
// double / float mix (this file is compiled with -fmad=false); predict_scale_level's logf becomes a comparison of the
// float ratio against thresholds derived on the host from the caller's own libm (see build_level_thresholds);
// candidates are visited in get_keypoints_in_cell order (cell-x, cell-y, insertion) via the same rank sort as match.cu,
// and "first strictly smaller distance wins" is min(distance << 32 | traversal position).
#include "common.cuh"
#include "pack.cuh"
#include "fuse_kernels.cuh"

#include <math.h>
#include <algorithm>
#include <cmath>
#include <mutex>

namespace plp {

namespace {

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// data/landmark.cc:349-361 as the reference evaluates it on the host
static int host_pred(float ratio, float lsf) {
    const float q = std::ceil(std::log(ratio) / lsf);
    if (!(q == q)) return INT32_MIN;  // NaN -> "negative" like the x86 conversion
    if (q >= 2147483648.0f || q < -2147483648.0f) return INT32_MIN;
    return (int)q;
}

// level_thr[k] (1 <= k < num_levels) = smallest positive float r with host_pred(r) >= k.  logf is monotone in every
// libm we know of; the neighbourhood of each threshold is checked and a violation is reported, never papered over.
struct ThresholdCacheEntry {
    float lsf;
    int num_levels;
    float thr[kMaxLevels];
};
static std::mutex g_thr_mutex;
static std::vector<ThresholdCacheEntry> g_thr_cache;  // a process sees a handful of (scale factor, levels) pairs

static plp_status build_level_thresholds_uncached(float lsf, int num_levels, float *thr);

// the table costs ~60 k logf evaluations (bisection + the monotonicity check): computed once per (lsf, num_levels)
static plp_status build_level_thresholds(float lsf, int num_levels, float *thr) {
    PLP_REQUIRE(lsf > 0.0f && num_levels >= 1 && num_levels <= kMaxLevels, "log_scale_factor / num_levels");
    std::lock_guard<std::mutex> lock(g_thr_mutex);
    for (const ThresholdCacheEntry &e : g_thr_cache)
        if (memcmp(&e.lsf, &lsf, 4) == 0 && e.num_levels == num_levels) {
            memcpy(thr, e.thr, sizeof(e.thr));
            return PLP_OK;
        }
    ThresholdCacheEntry e;
    e.lsf = lsf;
    e.num_levels = num_levels;
    PLP_TRY(build_level_thresholds_uncached(lsf, num_levels, e.thr));
    if (g_thr_cache.size() < 64) g_thr_cache.push_back(e);
    memcpy(thr, e.thr, sizeof(e.thr));
    return PLP_OK;
}

static plp_status build_level_thresholds_uncached(float lsf, int num_levels, float *thr) {
    for (int k = 0; k < kMaxLevels; ++k) thr[k] = INFINITY;
    for (int k = 1; k < num_levels; ++k) {
        uint32_t lo = 0x00000001u, hi = 0x7f7fffffu;  // predicate false at lo, true at hi
        float flo, fhi;
        memcpy(&flo, &lo, 4);
        memcpy(&fhi, &hi, 4);
        if (host_pred(flo, lsf) >= k || host_pred(fhi, lsf) < k) {
            set_error("predict_scale_level: no threshold for level %d (log_scale_factor %g)", k, (double)lsf);
            return PLP_ERR_INVALID;
        }
        while (hi - lo > 1) {
            const uint32_t mid = lo + (hi - lo) / 2;
            float f;
            memcpy(&f, &mid, 4);
            if (host_pred(f, lsf) >= k)
                hi = mid;
            else
                lo = mid;
        }
        for (uint32_t b = hi > 4096 ? hi - 4096 : 1; b < hi + 4096 && b <= 0x7f7fffffu; ++b) {
            float f;
            memcpy(&f, &b, 4);
            if ((host_pred(f, lsf) >= k) != (b >= hi)) {
                set_error("predict_scale_level: host logf is not monotone around level %d", k);
                return PLP_ERR_INVALID;
            }
        }
        memcpy(&thr[k], &hi, 4);
    }
    return PLP_OK;
}

static plp_status fill_params(FuseParams &P, const plp_camera *cam, const plp_grid *grid, const float *scale_factors,
                              const float *inv_level_sigma_sq, int num_levels, float log_scale_factor, float margin,
                              int mode) {
    memset(&P, 0, sizeof(P));
    P.cam = *cam;
    if (grid) P.grid = *grid;
    PLP_TRY(build_level_thresholds(log_scale_factor, num_levels, P.level_thr));
    for (int l = 0; l < num_levels; ++l) {
        P.scale_factors[l] = scale_factors[l];
        P.inv_sigma_sq[l] = inv_level_sigma_sq[l];
    }
    P.num_levels = num_levels;
    P.margin = margin;
    P.mode = mode;
    return PLP_OK;
}

static void add_landmarks(Layout &lay, const plp_fuse_landmarks &lms, int doubles_per_lm, FuseLandmarks &L) {
    const size_t m = (size_t)lms.m;
    L.m = lms.m;
    lay.in(L.pos_w, lms.pos_w, m * doubles_per_lm);
    lay.in(L.normal, lms.obs_mean_normal, m * 3);
    lay.in(L.min_d, lms.min_valid_dist, m);
    lay.in(L.max_d, lms.max_valid_dist, m);
    lay.in(L.max_raw, lms.max_valid_dist_raw, m);
    lay.in(L.desc, lms.desc, m * 32);
    lay.in(L.valid, lms.valid, m);
}

// landmarks per CTA so that (chunks x targets) fills the GPU about twice
static int chunk_size(const plp_ctx *ctx, int m, int num_targets) {
    const int want = std::max(1, (2 * std::max(ctx->sm_count, 1) + num_targets - 1) / num_targets);
    return std::max(32, div_up(m, want));
}

}  // namespace

}  // namespace plp

using namespace plp;

extern "C" {

plp_status plp_fuse_level_thresholds(float log_scale_factor, int num_levels, float *thr_out) {
    PLP_REQUIRE(thr_out, "null pointer");
    float thr[kMaxLevels];
    PLP_TRY(build_level_thresholds(log_scale_factor, num_levels, thr));
    thr_out[0] = 0.0f;
    for (int k = 1; k < num_levels; ++k) thr_out[k] = thr[k];
    return PLP_OK;
}

plp_status plp_fuse_search_points(plp_ctx *ctx, const plp_fuse_target_points *targets, int num_targets,
                                  const plp_grid *grid, const plp_camera *cam, const float *scale_factors,
                                  const float *inv_level_sigma_sq, int num_levels, float log_scale_factor,
                                  const plp_fuse_landmarks *lms, float margin, int mode, int32_t *best_idx_out,
                                  uint16_t *best_dist_out) {
    PLP_REQUIRE(ctx && grid && cam && scale_factors && inv_level_sigma_sq && lms && best_idx_out, "null pointer");
    PLP_REQUIRE(num_targets >= 0 && lms->m >= 0, "sizes");
    PLP_REQUIRE(mode == PLP_FUSE_DETECT || mode == PLP_FUSE_REPLACE, "mode");
    if (num_targets == 0 || lms->m == 0) return PLP_OK;
    PLP_REQUIRE(targets, "targets");
    PLP_REQUIRE(lms->pos_w && lms->obs_mean_normal && lms->min_valid_dist && lms->max_valid_dist &&
                    lms->max_valid_dist_raw && lms->desc,
                "landmark arrays");
    PLP_REQUIRE(grid->num_cols >= 1 && grid->num_rows >= 1 && (long long)grid->num_cols * grid->num_rows <= 16384,
                "grid size");
    const int m = lms->m;
    int max_n = 0;
    for (int t = 0; t < num_targets; ++t) {
        const plp_frame_points &f = targets[t].pts;
        PLP_REQUIRE(f.n >= 0, "target size");
        PLP_REQUIRE(f.n == 0 || (f.x && f.y && f.octave && f.desc), "target arrays");
        max_n = std::max(max_n, f.n);
    }
    if (max_n > kFuseMaxPoints) {
        set_error("fuse: %d keypoints exceed the per-keyframe capacity %d", max_n, kFuseMaxPoints);
        return PLP_ERR_CAPACITY;
    }
    FuseParams P;
    PLP_TRY(fill_params(P, cam, grid, scale_factors, inv_level_sigma_sq, num_levels, log_scale_factor, margin, mode));
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    FuseLandmarks L;
    add_landmarks(lay, *lms, 3, L);
    std::vector<FusePointTarget> dev_targets(num_targets);
    for (int t = 0; t < num_targets; ++t) {
        const plp_frame_points &f = targets[t].pts;
        const size_t n = (size_t)f.n;
        FusePointTarget &T = dev_targets[t];
        T.n = f.n;
        lay.in(T.x, f.x, n);
        lay.in(T.y, f.y, n);
        lay.in(T.xr, f.x_right, n);
        lay.in(T.octave, f.octave, n);
        lay.in(T.desc, f.desc, n * 32);
        lay.in(T.skip, targets[t].skip, m);
        memcpy(T.R, targets[t].rot_cw, sizeof(T.R));
        memcpy(T.t, targets[t].trans_cw, sizeof(T.t));
        memcpy(T.c, targets[t].cam_center, sizeof(T.c));
    }
    const FusePointTarget *d_targets;
    int32_t *d_idx;
    uint16_t *d_dist;
    lay.in(d_targets, dev_targets.data(), num_targets);
    lay.out(d_idx, (size_t)num_targets * m);
    lay.out(d_dist, (size_t)num_targets * m);
    PLP_TRY(lay.upload(ctx, 0));
    const int cap = max_n < 64 ? 64 : ((max_n + 63) / 64) * 64;
    const size_t smem = fuse_point_smem_bytes(cap, grid->num_cols * grid->num_rows);
    PLP_SMEM_OPTIN(fuse_points_kernel, smem);
    const int chunk = chunk_size(ctx, m, num_targets);
    dim3 g(div_up(m, chunk), num_targets);
    PLP_LAUNCH(ctx, fuse_points_kernel, g, kThreads, smem, d_targets, L, P, cap, chunk, d_idx, d_dist);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(best_idx_out, d_idx, (size_t)num_targets * m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (best_dist_out)
        PLP_CUDA_TRY(cudaMemcpyAsync(best_dist_out, d_dist, (size_t)num_targets * m * 2, cudaMemcpyDeviceToHost,
                                     ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

plp_status plp_fuse_search_lines(plp_ctx *ctx, const plp_fuse_target_lines *targets, int num_targets,
                                 const plp_camera *cam, const float *scale_factors_lsd,
                                 const float *inv_level_sigma_sq_lsd, int num_levels_lsd, float log_scale_factor_lsd,
                                 const plp_fuse_landmarks *lms, float margin, int32_t *best_idx_out,
                                 uint16_t *best_dist_out) {
    PLP_REQUIRE(ctx && cam && scale_factors_lsd && inv_level_sigma_sq_lsd && lms && best_idx_out, "null pointer");
    PLP_REQUIRE(num_targets >= 0 && lms->m >= 0, "sizes");
    if (num_targets == 0 || lms->m == 0) return PLP_OK;
    PLP_REQUIRE(targets, "targets");
    PLP_REQUIRE(lms->pos_w && lms->min_valid_dist && lms->max_valid_dist && lms->max_valid_dist_raw && lms->desc,
                "landmark arrays");
    const int m = lms->m;
    int max_n = 0;
    for (int t = 0; t < num_targets; ++t) {
        const plp_frame_lines &f = targets[t].lines;
        PLP_REQUIRE(f.n >= 0, "target size");
        PLP_REQUIRE(f.n == 0 || (f.sx && f.sy && f.ex && f.ey && f.octave && f.desc), "target arrays");
        max_n = std::max(max_n, f.n);
    }
    if (max_n > kFuseMaxLines) {
        set_error("fuse: %d keylines exceed the per-keyframe capacity %d", max_n, kFuseMaxLines);
        return PLP_ERR_CAPACITY;
    }
    FuseParams P;
    PLP_TRY(fill_params(P, cam, nullptr, scale_factors_lsd, inv_level_sigma_sq_lsd, num_levels_lsd, log_scale_factor_lsd,
                        margin, PLP_FUSE_REPLACE));
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    FuseLandmarks L;
    plp_fuse_landmarks lms_no_normal = *lms;
    lms_no_normal.obs_mean_normal = nullptr;
    add_landmarks(lay, lms_no_normal, 6, L);
    std::vector<FuseLineTarget> dev_targets(num_targets);
    for (int t = 0; t < num_targets; ++t) {
        const plp_frame_lines &f = targets[t].lines;
        const size_t n = (size_t)f.n;
        FuseLineTarget &T = dev_targets[t];
        T.n = f.n;
        lay.in(T.sx, f.sx, n);
        lay.in(T.sy, f.sy, n);
        lay.in(T.ex, f.ex, n);
        lay.in(T.ey, f.ey, n);
        lay.in(T.octave, f.octave, n);
        lay.in(T.desc, f.desc, n * 32);
        lay.in(T.skip, targets[t].skip, m);
        memcpy(T.R, targets[t].rot_cw, sizeof(T.R));
        memcpy(T.t, targets[t].trans_cw, sizeof(T.t));
        memcpy(T.c, targets[t].cam_center, sizeof(T.c));
    }
    const FuseLineTarget *d_targets;
    int32_t *d_idx;
    uint16_t *d_dist;
    lay.in(d_targets, dev_targets.data(), num_targets);
    lay.out(d_idx, (size_t)num_targets * m);
    lay.out(d_dist, (size_t)num_targets * m);
    PLP_TRY(lay.upload(ctx, 0));
    const int cap = max_n < 64 ? 64 : ((max_n + 63) / 64) * 64;
    const size_t smem = (size_t)cap * (32 + 5 * 4);
    PLP_SMEM_OPTIN(fuse_lines_kernel, smem);
    const int chunk = chunk_size(ctx, m, num_targets);
    dim3 g(div_up(m, chunk), num_targets);
    PLP_LAUNCH(ctx, fuse_lines_kernel, g, kThreads, smem, d_targets, L, P, cap, chunk, d_idx, d_dist);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(best_idx_out, d_idx, (size_t)num_targets * m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    if (best_dist_out)
        PLP_CUDA_TRY(cudaMemcpyAsync(best_dist_out, d_dist, (size_t)num_targets * m * 2, cudaMemcpyDeviceToHost,
                                     ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

}  // extern "C"
