// pose_opt.cu -- motion-only bundle adjustment on sm_100a.
//
// Replaces optimize::pose_optimizer::optimize (optimize/pose_optimizer.cc:53-229) and
// optimize::pose_optimizer_extended_line::optimize (optimize/pose_optimizer_extended_line.cc:62-305), i.e. the
// g2o graph {1 SE3 vertex, one unary edge per matched keypoint / keyline} solved with
// OptimizationAlgorithmLevenberg: 4 trials x <= 10 LM iterations with chi-square re-classification of ALL
// edges after each trial and removal of the Huber kernels at trial 2.
//
// One 128-thread CTA per frame runs the whole optimisation in a single launch (40 LM iterations x launch latency would
// otherwise dominate); device code and the work decomposition are in pose_opt_kernels.cuh.  The batch dimension is
// the grid.
//
// g2o semantics that are reproduced on purpose (see DESIGN.md "pose optimiser"):
//   - lambda_0 = 1e-5 * max diag(H) at the first iteration of every optimize() call, nu = 2
//   - rho = (chi_old - chi_new) / (dx^T (lambda dx + b) + 1e-3); accept iff rho > 0 and finite
//   - <= 10 retries per iteration; "terminate" when they are exhausted, rho == 0 or lambda overflows
//   - after a rejected last step the edge errors stay those of the rejected state (g2o does not recompute
//     them on pop()), and the reference thresholds these stale chi2 values for inlier edges
//   - line edges have no analytic Jacobian in the reference -> g2o central differences with delta = 1e-9
#include "common.cuh"
#include "pack.cuh"
#include "se3.cuh"
#include "pose_kernels.cuh"
#include "pose_opt_kernels.cuh"

namespace plp {

namespace {

__global__ void build_pose_jobs_kernel(PoseJob *jobs, int batch, const double *T_in, const plp_pt_obs *pts,
                                       const int32_t *pt_off, const plp_line_obs *lines, const int32_t *line_off,
                                       double *T_out, uint8_t *pt_outlier, uint8_t *line_outlier, int32_t *n_inl,
                                       int32_t *lm_iters) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= batch) return;
    PoseJob J;
    J.T_in = T_in + 16 * (size_t)b;
    J.pts = pts + pt_off[b];
    J.n_pts = pt_off[b + 1] - pt_off[b];
    const int l0 = line_off ? line_off[b] : 0, l1 = line_off ? line_off[b + 1] : 0;
    J.lines = lines ? lines + l0 : nullptr;
    J.n_lines = lines ? l1 - l0 : 0;
    J.T_out = T_out + 16 * (size_t)b;
    J.pt_outlier = pt_outlier + pt_off[b];
    J.line_outlier = line_outlier ? line_outlier + l0 : nullptr;
    J.n_inliers = n_inl + b;
    J.lm_iters = lm_iters ? lm_iters + b : nullptr;
    jobs[b] = J;
}

}  // namespace

plp_status launch_pose_opt(plp_ctx *ctx, const PoseJob *d_jobs, int batch, int max_edges, const plp_camera &cam,
                           const plp_pose_opt_cfg &cfg) {
    (void)max_edges;  // no per-frame shared-memory tables any more: the edge count is unbounded
    if (batch <= 0) return PLP_OK;
    using po::pose_opt_kernel;
    PLP_LAUNCH(ctx, pose_opt_kernel, batch, po::kThreads, 0, d_jobs, batch, cam, cfg);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

}  // namespace plp

using namespace plp;

extern "C" {

plp_status plp_pose_optimize_batch_dev(plp_ctx *ctx, const plp_camera *cam, int batch, const double *d_T_in,
                                       const plp_pt_obs *d_pts, const int32_t *d_pt_off, const plp_line_obs *d_lines,
                                       const int32_t *d_line_off, int max_edges_per_frame, const plp_pose_opt_cfg *cfg,
                                       double *d_T_out, uint8_t *d_pt_outlier, uint8_t *d_line_outlier,
                                       int32_t *d_n_inliers, int32_t *d_lm_iters) {
    PLP_REQUIRE(ctx && cam && cfg && d_T_in && d_pts && d_pt_off && d_T_out && d_pt_outlier && d_n_inliers,
                "null pointer");
    PLP_REQUIRE(batch >= 0 && cfg->num_trials >= 1 && cfg->num_each_iter >= 1, "batch / cfg");
    PLP_REQUIRE(!d_lines || (d_line_off && d_line_outlier), "line arrays");
    if (batch == 0) return PLP_OK;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    void *d_jobs = nullptr;
    PLP_TRY(ctx_scratch(ctx, 1, (size_t)batch * sizeof(PoseJob), &d_jobs));
    PLP_LAUNCH(ctx, build_pose_jobs_kernel, div_up(batch, 128), 128, 0, (PoseJob *)d_jobs, batch, d_T_in, d_pts,
               d_pt_off, d_lines, d_line_off, d_T_out, d_pt_outlier, d_line_outlier, d_n_inliers, d_lm_iters);
    PLP_CHECK_LAUNCH();
    return launch_pose_opt(ctx, (const PoseJob *)d_jobs, batch, max_edges_per_frame, *cam, *cfg);
}

plp_status plp_pose_optimize_batch(plp_ctx *ctx, const plp_camera *cam, int batch, const double *T_in,
                                   const plp_pt_obs *pts, const int32_t *pt_off, const plp_line_obs *lines,
                                   const int32_t *line_off, const plp_pose_opt_cfg *cfg, double *T_out,
                                   uint8_t *pt_outlier, uint8_t *line_outlier, int32_t *n_inliers) {
    PLP_REQUIRE(ctx && cam && cfg && T_in && pt_off && T_out && n_inliers, "null pointer");
    PLP_REQUIRE(batch >= 0, "batch");
    if (batch == 0) return PLP_OK;
    const int n_pts = pt_off[batch], n_lines = line_off ? line_off[batch] : 0;
    PLP_REQUIRE(n_pts >= 0 && n_lines >= 0 && pt_off[0] == 0 && (!line_off || line_off[0] == 0), "offsets");
    PLP_REQUIRE((n_pts == 0 || (pts && pt_outlier)) && (n_lines == 0 || (lines && line_outlier)), "null arrays");
    int max_edges = 0;
    for (int b = 0; b < batch; ++b) {
        const int e = (pt_off[b + 1] - pt_off[b]) + (line_off ? line_off[b + 1] - line_off[b] : 0);
        PLP_REQUIRE(pt_off[b + 1] >= pt_off[b] && (!line_off || line_off[b + 1] >= line_off[b]), "offsets not monotone");
        max_edges = e > max_edges ? e : max_edges;
    }
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    static const plp_pt_obs no_pts{};  // the batch entry point takes a non-null point array even without points
    const double *d_T;
    const plp_pt_obs *d_pts;
    const int32_t *d_po, *d_lo;
    const plp_line_obs *d_lines;
    double *d_To;
    uint8_t *d_pout, *d_lout = nullptr;
    int32_t *d_inl;
    lay.in(d_T, T_in, (size_t)batch * 16);
    lay.in(d_pts, n_pts ? pts : &no_pts, n_pts ? (size_t)n_pts : 1);
    lay.in(d_po, pt_off, (size_t)batch + 1);
    lay.in(d_lines, lines, n_lines);
    lay.in(d_lo, n_lines ? line_off : nullptr, (size_t)batch + 1);
    lay.out(d_To, (size_t)batch * 16);
    lay.out(d_pout, (size_t)n_pts + 8);
    if (n_lines) lay.out(d_lout, (size_t)n_lines + 8);
    lay.out(d_inl, batch);
    PLP_TRY(lay.upload(ctx, 0));
    PLP_TRY(plp_pose_optimize_batch_dev(ctx, cam, batch, d_T, d_pts, d_po, d_lines, d_lo, max_edges, cfg, d_To, d_pout,
                                        d_lout, d_inl, nullptr));
    PLP_CUDA_TRY(cudaMemcpyAsync(T_out, d_To, (size_t)batch * 128, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_pts) PLP_CUDA_TRY(cudaMemcpyAsync(pt_outlier, d_pout, (size_t)n_pts, cudaMemcpyDeviceToHost, ctx->stream));
    if (n_lines) PLP_CUDA_TRY(cudaMemcpyAsync(line_outlier, d_lout, (size_t)n_lines, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(n_inliers, d_inl, (size_t)batch * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

plp_status plp_pose_optimize(plp_ctx *ctx, const plp_camera *cam, const double *T_cw_in, const plp_pt_obs *pts,
                             int n_pts, const plp_line_obs *lines, int n_lines, const plp_pose_opt_cfg *cfg,
                             double *T_cw_out, uint8_t *pt_outlier, uint8_t *line_outlier, int32_t *n_inliers_out) {
    PLP_REQUIRE(n_pts >= 0 && n_lines >= 0, "sizes");
    const int32_t po[2] = {0, n_pts}, lo[2] = {0, n_lines};
    return plp_pose_optimize_batch(ctx, cam, 1, T_cw_in, pts, po, n_lines ? lines : nullptr, n_lines ? lo : nullptr, cfg,
                                   T_cw_out, pt_outlier, line_outlier, n_inliers_out);
}

}  // extern "C"
