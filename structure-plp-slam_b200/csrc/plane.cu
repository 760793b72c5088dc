// plane.cu -- Planar_Mapping_module plane RANSAC (planar_mapping_module.cc:412-771) (sm_100a).
//
// Same shape as essential.cu: hypotheses are independent given their index draws -> one CTA per hypothesis (thread 0
// fits the sample with planemath.h -- the text the oracle compiles, hence bit-identical --, all threads test the
// landmarks, thread 0 compacts the inliers in index order and refits), then a one-CTA kernel replays the reference's
// sequential bookkeeping over the per-hypothesis results and applies step [4].  FP64, compiled with -fmad=false.
#include "common.cuh"
#include "pack.cuh"
#include "plane_kernels.cuh"


using namespace plp;

extern "C" {

plp_status plp_plane_ransac(plp_ctx *ctx, const double *pos_w, const uint8_t *valid, int n, const int32_t *samples,
                            int num_iter, int sample_size, const plp_plane_ransac_cfg *cfg, double *eq_inout,
                            double *plane_error_inout, uint8_t *inlier_out, int32_t *status_out) {
    PLP_REQUIRE(ctx && cfg && status_out, "null pointer");
    PLP_REQUIRE(n >= 0 && num_iter >= 0 && sample_size >= 0, "sizes");
    PLP_REQUIRE(cfg->mode == 0 || cfg->mode == 1, "mode");
    PLP_REQUIRE(cfg->points_per_ransac >= 1, "points_per_ransac");
    *status_out = 0;
    if (n > 0) {
        PLP_REQUIRE(inlier_out, "inlier_out");
        memset(inlier_out, 0, (size_t)n);
    }
    if (n == 0) return PLP_OK;                 // planar_mapping_module.cc:423-426 / :597-600
    if (n < cfg->points_per_ransac) {          // :428-436 / :602-606 (update: plane->set_invalid())
        *status_out = cfg->mode == 1 ? 2 : 0;
        return PLP_OK;
    }
    PLP_REQUIRE(pos_w && eq_inout && plane_error_inout, "null pointer");
    if (num_iter == 0) return PLP_OK;          // no iteration: best_found stays false
    PLP_REQUIRE(samples && sample_size >= 1, "samples");
    for (long long i = 0; i < (long long)num_iter * sample_size; ++i)
        PLP_REQUIRE(samples[i] >= 0 && samples[i] < n, "sample index out of range");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const size_t N = (size_t)n, K = (size_t)num_iter;
    PlaneJob J;
    lay.in(J.pos, pos_w, N * 3);
    lay.in(J.valid, valid, N);
    lay.in(J.samples, samples, K * (size_t)sample_size);
    lay.in(J.eq, eq_inout, 4);
    lay.in(J.plane_err, plane_error_inout, 1);
    lay.out(J.eq_s, K * 4);
    lay.out(J.eq_r, K * 4);
    lay.out(J.res, K);
    lay.out(J.err, K);
    lay.out(J.elig, K);
    lay.out(J.cnt, K);
    lay.out(J.flag, K * N);
    lay.out(J.idx, K * N);
    lay.out(J.inlier, N);
    lay.out(J.status, 1);
    J.n = n;
    J.num_iter = num_iter;
    J.sample_size = sample_size;
    J.cfg = *cfg;
    PLP_TRY(lay.upload(ctx, 0));
    PLP_LAUNCH(ctx, plane_hypothesis_kernel, num_iter, kPlThreads, 0, J);
    PLP_CHECK_LAUNCH();
    PLP_LAUNCH(ctx, plane_select_kernel, 1, kPlThreads, 0, J);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(eq_inout, J.eq, 32, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(plane_error_inout, J.plane_err, 8, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(inlier_out, J.inlier, N, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(status_out, J.status, 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

}  // extern "C"
