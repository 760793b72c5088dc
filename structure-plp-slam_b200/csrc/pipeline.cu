// pipeline.cu -- device-resident, frame-batched tracking front-end:
//   frame_tracker::motion_based_track (module/frame_tracker.cc:52-124) =
//       projection::match_current_and_last_frames (margin, retry with 2*margin below 20 matches)
//     + pose_optimizer::optimize + discard_outliers (frame_tracker.cc:253-283)
// chained after orb_extractor::extract without leaving HBM.  This is the "extract + match + pose-opt" hot loop
// of BASELINE.json for a batch of independent (frame, last-frame-landmarks, predicted pose) triples -- SURVEY.md
// section 8(e): a live sequence is sequential, so the batch is made of independent tracking problems (offline /
// multi-sequence mode); each CTA handles one frame.
//
// The keypoints of the current frames are taken from the ORB handle's most recent extraction.  Undistortion is
// the identity here (zero-distortion camera; the host-pointer entry points take undistorted coordinates from
// the adapter instead).
#include "common.cuh"
#include "match_kernels.cuh"
#include "pack.cuh"
#include "pose_kernels.cuh"

namespace plp {

namespace {

constexpr int kNumMatchesThr = 20;  // frame_tracker::num_matches_thr_ (module/frame_tracker.h)

struct TrackDev {
    int batch, cap, num_levels;
    // current frames (ORB output)
    const plp_keypoint *kp;
    const uint8_t *desc;
    const int32_t *n_kp;
    // last frames
    const double *last_pos_w;
    const int32_t *last_octave;
    const float *last_angle;
    const uint8_t *last_desc;
    const uint8_t *last_valid;
    const int32_t *last_offsets;
    const double *pose_pred, *pose_last;
    // scratch (SoA copies of the current keypoints, queries, jobs)
    float *x, *y, *angle;
    int32_t *octave;
    float *qx, *qy, *qxr, *qradius;
    int32_t *qmin, *qmax;
    uint8_t *qvalid;
    int32_t *choice;
    uint32_t *num_matches;
    ProjectJob *pjobs;       // 2 x batch (first attempt, retry)
    PointMatchJob *mjobs;    // 2 x batch
    PoseJob *posejobs;       // batch
    plp_pt_obs *obs;         // batch x cap
    int32_t *obs_kp;         // batch x cap : keypoint index of each observation
    uint8_t *obs_outlier;    // batch x cap
    float inv_level_sigma_sq[16];
    // outputs
    int32_t *matched;        // batch x cap : last-frame index per keypoint (-1: none) after discard_outliers
    double *pose_out;        // batch x 16
    int32_t *num_valid;      // batch
    int32_t *n_inliers;      // batch (pose optimiser return value)
    int32_t *lm_iters;       // batch
    int max_last;
};

__global__ void track_prep_kernel(TrackDev T, float margin, int check_orientation) {
    const int b = blockIdx.x, tid = threadIdx.x;
    const int n = T.n_kp[b];
    const size_t base = (size_t)b * T.cap;
    for (int i = tid; i < n; i += blockDim.x) {
        const plp_keypoint k = T.kp[base + i];
        T.x[base + i] = k.x;
        T.y[base + i] = k.y;
        T.angle[base + i] = k.angle;
        T.octave[base + i] = k.octave;
    }
    if (tid == 0) {
        const int l0 = T.last_offsets[b], m = T.last_offsets[b + 1] - l0;
        for (int attempt = 0; attempt < 2; ++attempt) {
            ProjectJob P;
            P.n_last = m;
            P.pos_w = T.last_pos_w + 3 * (size_t)l0;
            P.octave = T.last_octave + l0;
            P.valid = T.last_valid ? T.last_valid + l0 : nullptr;
            for (int k = 0; k < 12; ++k) P.pose_cw[k] = T.pose_pred[16 * (size_t)b + k];
            P.assume_forward = 0;  // monocular (projection.cc:231-238)
            P.assume_backward = 0;
            const size_t qb = (size_t)b * T.max_last;
            P.qx = T.qx + qb;
            P.qy = T.qy + qb;
            P.qxr = T.qxr + qb;
            P.qx2 = P.qy2 = P.qxr2 = nullptr;
            P.qradius = T.qradius + qb;
            P.qmin = T.qmin + qb;
            P.qmax = T.qmax + qb;
            P.qvalid = T.qvalid + qb;
            PointMatchJob J;
            J.n = n;
            J.x = T.x + base;
            J.y = T.y + base;
            J.octave = T.octave + base;
            J.angle = T.angle + base;
            J.x_right = nullptr;
            J.desc = T.desc + base * 32;
            J.claimed = nullptr;  // curr_frm.landmarks_ was just cleared (frame_tracker.cc:61)
            J.hamm_thr_p1 = 0;
            J.m = m;
            J.qx = P.qx;
            J.qy = P.qy;
            J.qxr = P.qxr;
            J.qradius = P.qradius;
            J.qmin = P.qmin;
            J.qmax = P.qmax;
            J.qangle = T.last_angle + l0;
            J.qdesc = T.last_desc + (size_t)l0 * 32;
            J.qvalid = P.qvalid;
            J.choice = T.choice + qb;
            J.best_idx_out = nullptr;
            J.matched_out = T.matched + base;
            J.num_matches = T.num_matches + b;
            T.pjobs[attempt * T.batch + b] = P;
            T.mjobs[attempt * T.batch + b] = J;
        }
    }
}

// disable the widened-margin retry for frames whose first attempt reached the threshold (frame_tracker.cc:66-71)
__global__ void track_retry_gate_kernel(TrackDev T) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= T.batch) return;
    if (T.num_matches[b] >= (uint32_t)kNumMatchesThr) {
        T.pjobs[T.batch + b].n_last = -1;
        T.mjobs[T.batch + b].m = -1;
    }
}

// 2D-3D observations of the matched keypoints, in keypoint order (pose_optimizer.cc:126-151)
__global__ void track_gather_kernel(TrackDev T) {
    __shared__ int warp_sums[8];
    __shared__ int s_base;
    const int b = blockIdx.x, tid = threadIdx.x;
    const int n = T.n_kp[b];
    const size_t base = (size_t)b * T.cap;
    const int l0 = T.last_offsets[b];
    const bool enough = T.num_matches[b] >= (uint32_t)kNumMatchesThr;  // frame_tracker.cc:73-77
    if (tid == 0) s_base = 0;
    __syncthreads();
    for (int start = 0; start < n; start += 256) {
        const int i = start + tid;
        int q = -1;
        if (i < n && enough) q = T.matched[base + i];
        const int flag = q >= 0;
        // ordered compaction
        const unsigned bal = __ballot_sync(0xffffffffu, flag);
        const int lane = tid & 31, warp = tid >> 5;
        if (lane == 0) warp_sums[warp] = __popc(bal);
        __syncthreads();
        int off = s_base;
        for (int w = 0; w < warp; ++w) off += warp_sums[w];
        off += __popc(bal & ((1u << lane) - 1));
        if (flag) {
            plp_pt_obs o;
            const double *X = T.last_pos_w + 3 * (size_t)(l0 + q);
            o.pos_w[0] = X[0];
            o.pos_w[1] = X[1];
            o.pos_w[2] = X[2];
            o.obs_x = T.x[base + i];
            o.obs_y = T.y[base + i];
            o.x_right = -1.0f;
            o.inv_sigma_sq = T.inv_level_sigma_sq[T.octave[base + i]];
            T.obs[base + off] = o;
            T.obs_kp[base + off] = i;
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int w = 0; w < 8; ++w) tot += warp_sums[w];
            s_base += tot;
        }
        __syncthreads();
    }
    if (tid == 0) {
        PoseJob J;
        J.T_in = T.pose_pred + 16 * (size_t)b;
        J.pts = T.obs + base;
        J.n_pts = s_base;
        J.lines = nullptr;
        J.n_lines = 0;
        J.T_out = T.pose_out + 16 * (size_t)b;
        J.pt_outlier = T.obs_outlier + base;
        J.line_outlier = nullptr;
        J.n_inliers = T.n_inliers + b;
        J.lm_iters = T.lm_iters + b;
        T.posejobs[b] = J;
    }
}

// frame_tracker::discard_outliers (frame_tracker.cc:253-283)
__global__ void track_finish_kernel(TrackDev T) {
    __shared__ int s_cnt;
    const int b = blockIdx.x, tid = threadIdx.x;
    const size_t base = (size_t)b * T.cap;
    const int n_obs = T.posejobs[b].n_pts;
    const bool enough = T.num_matches[b] >= (uint32_t)kNumMatchesThr;
    if (tid == 0) s_cnt = 0;
    __syncthreads();
    int valid = 0;
    if (enough) {
        for (int k = tid; k < n_obs; k += blockDim.x) {
            if (T.obs_outlier[base + k])
                T.matched[base + T.obs_kp[base + k]] = -1;
            else
                ++valid;
        }
    } else {
        const int n = T.n_kp[b];
        for (int i = tid; i < n; i += blockDim.x) T.matched[base + i] = -1;
    }
    atomicAdd(&s_cnt, valid);
    __syncthreads();
    if (tid == 0) T.num_valid[b] = s_cnt;
}

}  // namespace

}  // namespace plp

using namespace plp;

struct plp_tracker {
    plp_ctx *ctx = nullptr;
    int max_batch = 0, cap = 0, max_last = 0, num_levels = 0;
    plp_camera cam;
    plp_grid grid;
    float scale_factors[16];
    float inv_level_sigma_sq[16];
    float *d_scale_factors = nullptr;
    uint8_t *d_block = nullptr;  // one allocation carved into the scratch arrays
    TrackDev dev;
};

extern "C" {

plp_status plp_tracker_create(plp_ctx *ctx, const plp_camera *cam, const plp_grid *grid, const float *scale_factors,
                              const float *inv_level_sigma_sq, int num_levels, int max_batch, int kp_capacity,
                              int max_last_points, plp_tracker **out) {
    PLP_REQUIRE(ctx && cam && grid && scale_factors && inv_level_sigma_sq && out, "null pointer");
    PLP_REQUIRE(num_levels >= 1 && num_levels <= 16 && max_batch >= 1 && kp_capacity >= 1 && max_last_points >= 1, "sizes");
    PLP_REQUIRE(cam->setup_type == 0, "the batched tracker implements the monocular path");
    *out = nullptr;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    plp_tracker *t = new plp_tracker();
    t->ctx = ctx;
    t->max_batch = max_batch;
    t->cap = kp_capacity;
    t->max_last = max_last_points;
    t->num_levels = num_levels;
    t->cam = *cam;
    t->grid = *grid;
    for (int l = 0; l < num_levels; ++l) {
        t->scale_factors[l] = scale_factors[l];
        t->inv_level_sigma_sq[l] = inv_level_sigma_sq[l];
    }
    const size_t B = max_batch, C = kp_capacity, M = max_last_points;
    TrackDev &T = t->dev;
    memset(&T, 0, sizeof(T));
    Layout lay;
    lay.out(t->d_scale_factors, 16);
    lay.out(T.x, B * C);
    lay.out(T.y, B * C);
    lay.out(T.angle, B * C);
    lay.out(T.octave, B * C);
    lay.out(T.qx, B * M);
    lay.out(T.qy, B * M);
    lay.out(T.qxr, B * M);
    lay.out(T.qradius, B * M);
    lay.out(T.qmin, B * M);
    lay.out(T.qmax, B * M);
    lay.out(T.qvalid, B * M);
    lay.out(T.choice, B * M);
    lay.out(T.num_matches, B);
    lay.out(T.pjobs, 2 * B);
    lay.out(T.mjobs, 2 * B);
    lay.out(T.posejobs, B);
    lay.out(T.obs, B * C);
    lay.out(T.obs_kp, B * C);
    lay.out(T.obs_outlier, B * C);
    if (cudaMalloc((void **)&t->d_block, lay.bytes()) != cudaSuccess) {
        set_error("tracker: cudaMalloc(%zu) failed", lay.bytes());
        delete t;
        return PLP_ERR_CUDA;
    }
    lay.bind(t->d_block);
    cudaMemcpy(t->d_scale_factors, t->scale_factors, num_levels * 4, cudaMemcpyHostToDevice);
    T.cap = kp_capacity;
    T.num_levels = num_levels;
    T.max_last = max_last_points;
    for (int l = 0; l < 16; ++l) T.inv_level_sigma_sq[l] = l < num_levels ? inv_level_sigma_sq[l] : 1.0f;
    *out = t;
    return PLP_OK;
}

void plp_tracker_destroy(plp_tracker *t) {
    if (!t) return;
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    if (t->d_block) cudaFree(t->d_block);
    delete t;
}

plp_status plp_tracker_motion_track_batch_dev(plp_tracker *t, int batch, const plp_keypoint *d_kp, const uint8_t *d_desc,
                                              const int32_t *d_n_kp, const plp_track_last *last, float margin,
                                              int32_t *d_matched_out, double *d_pose_out, int32_t *d_num_valid_out,
                                              int32_t *d_n_inliers_out, int32_t *d_lm_iters_out) {
    PLP_REQUIRE(t && d_kp && d_desc && d_n_kp && last && d_matched_out && d_pose_out && d_num_valid_out &&
                    d_n_inliers_out && d_lm_iters_out,
                "null pointer");
    PLP_REQUIRE(batch >= 1 && batch <= t->max_batch, "batch exceeds the tracker's max_batch");
    PLP_REQUIRE(last->pos_w && last->octave && last->angle && last->desc && last->offsets && last->pose_pred &&
                    last->pose_last,
                "last-frame arrays");
    plp_ctx *ctx = t->ctx;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    TrackDev T = t->dev;
    T.batch = batch;
    T.kp = d_kp;
    T.desc = d_desc;
    T.n_kp = d_n_kp;
    T.last_pos_w = last->pos_w;
    T.last_octave = last->octave;
    T.last_angle = last->angle;
    T.last_desc = last->desc;
    T.last_valid = last->valid;
    T.last_offsets = last->offsets;
    T.pose_pred = last->pose_pred;
    T.pose_last = last->pose_last;
    T.matched = d_matched_out;
    T.pose_out = d_pose_out;
    T.num_valid = d_num_valid_out;
    T.n_inliers = d_n_inliers_out;
    T.lm_iters = d_lm_iters_out;
    PLP_LAUNCH(ctx, track_prep_kernel, batch, 256, 0, T, margin, 1);
    PLP_CHECK_LAUNCH();
    // first attempt (projection.cc:214-358 with `margin`)
    PLP_TRY(launch_project_points(ctx, T.pjobs, batch, t->max_last, t->cam, t->d_scale_factors, t->num_levels, margin));
    PLP_TRY(launch_point_match(ctx, T.mjobs, batch, t->cap > kMatchMaxPoints ? kMatchMaxPoints : t->cap, t->grid, 0, 0.0f, 1));
    // widened retry for the frames that found fewer than 20 matches (frame_tracker.cc:66-71)
    PLP_LAUNCH(ctx, track_retry_gate_kernel, div_up(batch, 128), 128, 0, T);
    PLP_CHECK_LAUNCH();
    PLP_TRY(launch_project_points(ctx, T.pjobs + batch, batch, t->max_last, t->cam, t->d_scale_factors, t->num_levels,
                                  2 * margin));
    PLP_TRY(launch_point_match(ctx, T.mjobs + batch, batch, t->cap > kMatchMaxPoints ? kMatchMaxPoints : t->cap, t->grid,
                               0, 0.0f, 1));
    PLP_LAUNCH(ctx, track_gather_kernel, batch, 256, 0, T);
    PLP_CHECK_LAUNCH();
    plp_pose_opt_cfg cfg{4, 10};
    PLP_TRY(launch_pose_opt(ctx, T.posejobs, batch, t->cap > 6144 ? 6144 : t->cap, t->cam, cfg));
    PLP_LAUNCH(ctx, track_finish_kernel, batch, 256, 0, T);
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

}  // extern "C"
