// match_kernels.cuh -- device job descriptors + launchers shared by match.cu (host-pointer C ABI)
// and pipeline.cu (device-resident batched tracking front-end).
#pragma once
#include "common.cuh"
#include "match_jobs.h"

namespace plp {

constexpr int kMatchMaxPoints = 3072;  // per-frame keypoint capacity of the window matcher (smem bound)
constexpr int kBruteMaxPoints = 4096;
constexpr int kLineMaxLines = 16384;   // per-frame keyline capacity of the keyline matcher (smem bound)

plp_status launch_point_match(plp_ctx *ctx, const PointMatchJob *d_jobs, int num_jobs, int max_n,
                              const plp_grid &grid, int ratio_test, float lowe_ratio,
                              int check_orientation);
plp_status launch_line_match(plp_ctx *ctx, const LineMatchJob *d_jobs, int num_jobs, int ratio_test,
                             float lowe_ratio, int rgbd_gate);
plp_status launch_brute_match(plp_ctx *ctx, const BruteJob *d_jobs, int num_jobs, int max_n_frm,
                              float lowe_ratio, int check_orientation);
plp_status launch_project_points(plp_ctx *ctx, const ProjectJob *d_jobs, int num_jobs, int max_n,
                                 const plp_camera &cam, const float *d_scale_factors, int num_levels,
                                 float margin);
plp_status launch_project_lines(plp_ctx *ctx, const ProjectJob *d_jobs, int num_jobs, int max_n,
                                const plp_camera &cam, const float *d_scale_factors, int num_levels,
                                float margin);

// host-side: projection.cc:220-238 forward/backward assumption
void motion_assumption(const plp_camera &cam, const double *pose_cw_curr, const double *pose_cw_last,
                       int *fwd, int *bwd);

}  // namespace plp
