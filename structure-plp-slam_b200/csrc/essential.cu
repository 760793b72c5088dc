// essential.cu -- solve::essential_solver::find_via_ransac (solve/essential_solver.cc:37-121) (sm_100a).
//
// RANSAC hypotheses are independent given their sample sets: grid = one CTA per hypothesis.  Thread 0 solves the
// eight-point system (9 x 9 cyclic Jacobi, essmath.h -- the same text the oracle compiles, hence bit-identical), all
// threads test the matches (two epipolar residuals each, the reference's double -> float mix), and the score is the
// reference's sequential float sum in match order (thread 0 walks the per-match residuals staged in shared memory /
// global scratch).  A one-CTA kernel then replays "if (best_score_ < score_in_sac)" over the hypotheses in order,
// copies the winner's inlier flags and optionally recomputes E from all inliers (:99-120).  FP64, compiled with
// -fmad=false.
#include "common.cuh"
#include "pack.cuh"
#include "essential_kernels.cuh"


using namespace plp;

extern "C" {

plp_status plp_essential_ransac(plp_ctx *ctx, const double *bearings_1, int n1, const double *bearings_2, int n2,
                                const int32_t *matches_12, int num_matches, const int32_t *samples, int num_iter,
                                int recompute, uint8_t *is_inlier_out, double *best_E_21_out, double *best_score_out,
                                int32_t *solution_is_valid_out) {
    PLP_REQUIRE(ctx && solution_is_valid_out, "null pointer");
    PLP_REQUIRE(n1 >= 0 && n2 >= 0 && num_matches >= 0 && num_iter >= 0, "sizes");
    *solution_is_valid_out = 0;
    if (num_matches < 8) return PLP_OK;  // essential_solver.cc:45-49: solution_is_valid_ = false, nothing else touched
    PLP_REQUIRE(bearings_1 && bearings_2 && matches_12 && is_inlier_out && best_E_21_out && best_score_out, "null pointer");
    PLP_REQUIRE(num_iter == 0 || samples, "samples");
    for (int i = 0; i < num_matches; ++i)
        PLP_REQUIRE(matches_12[2 * i] >= 0 && matches_12[2 * i] < n1 && matches_12[2 * i + 1] >= 0 && matches_12[2 * i + 1] < n2,
                    "match index out of range");
    for (int i = 0; i < num_iter * 8; ++i) PLP_REQUIRE(samples[i] >= 0 && samples[i] < num_matches, "sample index out of range");
    if (num_iter == 0) {  // best_score_ stays 0: invalid, all flags false
        memset(is_inlier_out, 0, (size_t)num_matches);
        for (int k = 0; k < 9; ++k) best_E_21_out[k] = 0.0;
        *best_score_out = 0.0;
        return PLP_OK;
    }
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    Layout lay;
    const size_t M = (size_t)num_matches, K = (size_t)num_iter;
    EssJob J;
    lay.in(J.b1, bearings_1, (size_t)n1 * 3);
    lay.in(J.b2, bearings_2, (size_t)n2 * 3);
    lay.in(J.matches, matches_12, M * 2);
    lay.in(J.samples, samples, K * 8);
    lay.out(J.E, K * 9);
    lay.out(J.score, K);
    lay.out(J.inlier, K * M);
    lay.out(J.res, K * M * 2);
    lay.out(J.best_inlier, M);
    lay.out(J.best_E, 9);
    lay.out(J.best_score, 1);
    lay.out(J.valid, 1);
    J.num_matches = num_matches;
    J.num_iter = num_iter;
    J.recompute = recompute;
    PLP_TRY(lay.upload(ctx, 0));
    PLP_LAUNCH(ctx, essential_hypothesis_kernel, num_iter, kEssThreads, 0, J);
    PLP_CHECK_LAUNCH();
    PLP_LAUNCH(ctx, essential_select_kernel, 1, kEssThreads, 0, J);
    PLP_CHECK_LAUNCH();
    PLP_CUDA_TRY(cudaMemcpyAsync(is_inlier_out, J.best_inlier, M, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(best_E_21_out, J.best_E, 72, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(best_score_out, J.best_score, 8, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(solution_is_valid_out, J.valid, 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

}  // extern "C"
