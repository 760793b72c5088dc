// ba_host.cu -- C ABI and Levenberg-Marquardt driver of the local bundle adjuster (kernels: local_ba.cu).
//
// The host only (1) uploads the gathered graph, (2) enqueues chunks of LM "tries" (each try = a fixed sequence of
// kernels whose accept/reject logic runs on the device), (3) polls the device state once per chunk to learn
// whether optimize(n) finished, (4) runs the outlier classification between the two optimize() calls and
// downloads the result.  See optimize/local_bundle_adjuster.cc:276-372 for the control flow that is mirrored.
#include <algorithm>

#include "ba_kernels.cuh"
#include "pack.cuh"

using namespace plp;

struct plp_ba_comm;
namespace plp {
BaCollective *ba_comm_collective(plp_ba_comm *c);
int ba_comm_rank(plp_ba_comm *c);
int ba_comm_world(plp_ba_comm *c);
}  // namespace plp

struct plp_ba {
    plp_ctx *ctx = nullptr;
    plp_ba_cfg cfg;
    BaDev dev;
    uint8_t *d_block = nullptr;
    size_t block_bytes = 0;
    // initial state kept on the device so that a solve can be repeated (benchmarks)
    double *d_T_in = nullptr, *d_pts_in = nullptr, *d_lines_in = nullptr;
    double *d_T_out = nullptr, *d_pts_out = nullptr, *d_lines_out = nullptr;
    BaState *h_state = nullptr;  // pinned
    double *d_stop = nullptr;    // multi-GPU: the force-stop word every rank agrees on (sum over ranks)
    double *h_stop = nullptr;    // pinned, 2 doubles: [0] upload, [1] reduced value
    plp_ba_comm *comm = nullptr;
    int n_kf = 0, n_pts = 0, n_lines = 0, n_pe = 0, n_le = 0;
    cudaGraphExec_t try_graph = nullptr;  // one LM try captured as a CUDA graph
    int try_graph_launches = 0;
};

namespace {

// One LM try = a fixed sequence of 7 launches whose arguments never change (all state lives in device memory),
// so it is captured once into a CUDA graph and replayed: ~7 x 4 us of launch overhead -> one graph launch.
plp_status launch_try(plp_ba *b) {
    plp_ctx *ctx = b->ctx;
    BaCollective *coll = b->comm ? ba_comm_collective(b->comm) : nullptr;
    // events / NCCL: plain launches; the NVLink peer all-reduce is an ordinary kernel whose call counter lives in device
    // memory, so a try that uses it is captured like a single-GPU try
    if (ctx->timing || (coll && !coll->graph_safe(b->dev.packed_sum_len + b->dev.world))) return ba_launch_try(ctx, b->dev, coll);
    if (!b->try_graph) {
        cudaGraph_t g = nullptr;
        const uint64_t l0 = ctx->launches;
        PLP_CUDA_TRY(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
        const plp_status s = ba_launch_try(ctx, b->dev, coll);
        const cudaError_t e = cudaStreamEndCapture(ctx->stream, &g);
        b->try_graph_launches = (int)(ctx->launches - l0);
        ctx->launches = l0;
        if (s != PLP_OK) return s;
        if (e != cudaSuccess) {
            set_error("cudaStreamEndCapture failed: %s", cudaGetErrorString(e));
            return PLP_ERR_CUDA;
        }
        PLP_CUDA_TRY(cudaGraphInstantiate(&b->try_graph, g, 0));
        cudaGraphDestroy(g);
    }
    PLP_CUDA_TRY(cudaGraphLaunch(b->try_graph, ctx->stream));
    ctx->launches += b->try_graph_launches;
    if (coll) coll->add_calls(2);  // packed system + trial sums
    return PLP_OK;
}

plp_status read_state(plp_ba *b) {
    PLP_CUDA_TRY(cudaMemcpyAsync(b->h_state, b->dev.state, sizeof(BaState), cudaMemcpyDeviceToHost, b->ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(b->ctx->stream));
    if (b->comm) PLP_TRY(ba_comm_collective(b->comm)->check());  // a peer all-reduce that timed out is an error, not a result
    return PLP_OK;
}

// The force-stop flag is written asynchronously by another host thread (mapping_module.cc:159-164), so two ranks may
// read different values at the "same" point.  With a communicator every rank issues the same sequence of collectives
// only if the stop decision itself is collective: the local flag is summed over the ranks (one 8-byte all-reduce per
// chunk of LM tries, outside the per-try path) and every rank acts on the reduced value.
plp_status stop_requested(plp_ba *b, volatile const uint8_t *force_stop, bool *stop) {
    const bool local = force_stop && *force_stop;
    BaCollective *coll = b->comm ? ba_comm_collective(b->comm) : nullptr;
    if (!coll) {
        *stop = local;
        return PLP_OK;
    }
    plp_ctx *ctx = b->ctx;
    b->h_stop[0] = local ? 1.0 : 0.0;
    PLP_CUDA_TRY(cudaMemcpyAsync(b->d_stop, b->h_stop, 8, cudaMemcpyHostToDevice, ctx->stream));
    PLP_TRY(coll->all_reduce(b->d_stop, 1));
    PLP_CUDA_TRY(cudaMemcpyAsync(b->h_stop + 1, b->d_stop, 8, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    *stop = b->h_stop[1] != 0.0;
    return PLP_OK;
}

// SparseOptimizer::optimize(n): enqueue tries in chunks until the device state machine reports completion
plp_status run_optimize(plp_ba *b, int n, int robust, bool first, volatile const uint8_t *force_stop, int *iters_done,
                        bool *stopped) {
    plp_ctx *ctx = b->ctx;
    PLP_TRY(ba_launch_set_state(ctx, b->dev, n, robust, first ? 1 : 0));
    int launched = 0;
    const int hard_cap = n * 10 + 4;
    int chunk = n + 2;  // 1 lambda-init try + n iterations + 1 spare (typical runs finish in the first chunk)
    while (true) {
        for (int t = 0; t < chunk; ++t) PLP_TRY(launch_try(b));
        PLP_TRY(ba_launch_decide(ctx, b->dev));
        launched += chunk;
        PLP_TRY(read_state(b));
        if (b->h_state->phase == kBaDone || launched >= hard_cap) break;  // identical on every rank (replicated state)
        if (force_stop || b->comm) {  // g2o polls the force-stop flag between iterations
            PLP_TRY(stop_requested(b, force_stop, stopped));
            if (*stopped) break;
        }
        chunk = 2;
    }
    *iters_done = b->h_state->it;
    return PLP_OK;
}

}  // namespace

extern "C" {

void plp_ba_destroy(plp_ba *b) {
    if (!b) return;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    if (b->d_block) cudaFree(b->d_block);
    if (b->h_state) cudaFreeHost(b->h_state);
    if (b->h_stop) cudaFreeHost(b->h_stop);
    if (b->try_graph) cudaGraphExecDestroy(b->try_graph);
    delete b;
}

plp_status plp_ba_create(plp_ctx *ctx, const plp_ba_problem *p, const plp_ba_cfg *cfg, plp_ba_comm *comm, plp_ba **out) {
    PLP_REQUIRE(ctx && p && cfg && out, "null pointer");
    *out = nullptr;
    PLP_REQUIRE(p->n_kf >= 1, "n_kf >= 1");  // fixed keyframes are unbounded: every array is sized by n_kf
    PLP_REQUIRE(p->n_pts >= 0 && p->n_lines >= 0 && p->n_pt_edges >= 0 && p->n_line_edges >= 0 && p->n_plane_edges >= 0, "sizes");
    PLP_REQUIRE(p->kf_pose_cw && p->kf_fixed, "keyframe arrays");
    PLP_REQUIRE(p->n_pts == 0 || p->pt_pos_w, "pt_pos_w");
    PLP_REQUIRE(p->n_pt_edges == 0 || (p->pt_edge_kf && p->pt_edge_lm && p->pt_edge_obs && p->pt_edge_inv_sigma_sq), "point edges");
    PLP_REQUIRE(p->n_lines == 0 || p->line_plucker, "line_plucker");
    PLP_REQUIRE(p->n_line_edges == 0 || (p->line_edge_kf && p->line_edge_lm && p->line_edge_obs && p->line_edge_inv_sigma_sq), "line edges");
    PLP_REQUIRE(p->n_plane_edges == 0 || (p->plane_edge_lm && p->plane_edge_fn), "plane edges");
    const int n_kf = p->n_kf, n_pts = p->n_pts, n_lines = p->n_lines, n_pe = p->n_pt_edges, n_le = p->n_line_edges;
    std::vector<int> hidx(n_kf, -1);
    int n_free = 0;
    for (int k = 0; k < n_kf; ++k)
        if (!p->kf_fixed[k]) hidx[k] = n_free++;
    const bool large = n_free > kBaMaxFree;  // reduced camera system dense in HBM + blocked Cholesky (ba_chol.cu)
    PLP_REQUIRE(n_free >= 1, "at least one non-fixed keyframe");
    // CSR offsets (edges must be grouped by ascending landmark index, as the reference creates them)
    std::vector<int> pt_off(n_pts + 1, 0), ln_off(n_lines + 1, 0);
    for (int e = 0; e < n_pe; ++e) {
        const int l = p->pt_edge_lm[e], k = p->pt_edge_kf[e];
        PLP_REQUIRE(l >= 0 && l < n_pts && k >= 0 && k < n_kf, "point edge index out of range");
        PLP_REQUIRE(e == 0 || p->pt_edge_lm[e - 1] <= l, "point edges must be grouped by ascending landmark index");
        pt_off[l + 1]++;
    }
    for (int l = 0; l < n_pts; ++l) pt_off[l + 1] += pt_off[l];
    for (int e = 0; e < n_le; ++e) {
        const int l = p->line_edge_lm[e], k = p->line_edge_kf[e];
        PLP_REQUIRE(l >= 0 && l < n_lines && k >= 0 && k < n_kf, "line edge index out of range");
        PLP_REQUIRE(e == 0 || p->line_edge_lm[e - 1] <= l, "line edges must be grouped by ascending landmark index");
        ln_off[l + 1]++;
    }
    for (int l = 0; l < n_lines; ++l) ln_off[l + 1] += ln_off[l];
    std::vector<int> pt_plane(std::max(n_pts, 1), -1);
    for (int i = 0; i < p->n_plane_edges; ++i) {
        const int l = p->plane_edge_lm[i];
        PLP_REQUIRE(l >= 0 && l < n_pts, "plane edge landmark out of range");
        PLP_REQUIRE(pt_plane[l] < 0, "at most one plane edge per landmark (landmark::get_Owning_Plane)");
        pt_plane[l] = i;
    }
    // free degree per landmark -> landmarks per batch; CTA ranges balanced by the cost model of ba_linearize_kernel: a
    // warp owns a landmark, a point landmark costs one round over its (<= 32) edges, a line landmark one round per edge
    // (numeric Jacobians: 21 evaluations spread over the lanes) plus the same per-landmark tail
    const int n_lm = n_pts + n_lines;
    int w_point = 4, w_line0 = 8;
    if (const char *wenv = getenv("PLP_BA_COST_WEIGHTS")) sscanf(wenv, "%d,%d", &w_point, &w_line0);  // tuning aid
    int max_deg = 1;
    std::vector<int> deg_e(n_lm + 1, 0);
    for (int l = 0; l < n_pts; ++l) {
        int d = 0;
        for (int e = pt_off[l]; e < pt_off[l + 1]; ++e) d += hidx[p->pt_edge_kf[e]] >= 0;
        max_deg = std::max(max_deg, d);
        deg_e[l + 1] = deg_e[l] + w_point * (1 + (pt_off[l + 1] - pt_off[l] - 1) / 32);  // lane = edge: one round per 32 edges
    }
    for (int l = 0; l < n_lines; ++l) {
        int d = 0;
        for (int e = ln_off[l]; e < ln_off[l + 1]; ++e) d += hidx[p->line_edge_kf[e]] >= 0;
        max_deg = std::max(max_deg, d);
        deg_e[n_pts + l + 1] = deg_e[n_pts + l] + w_line0 + (ln_off[l + 1] - ln_off[l]);  // one warp round per line edge
    }
    PLP_REQUIRE(max_deg <= n_free, "a landmark is observed twice by the same keyframe");
    const int pool_cap = ba_pool_capacity(n_free, n_free * (n_free + 1) / 2, max_deg);
    const int LB = std::max(1, std::min(16, pool_cap / max_deg));
    // one batch of LB landmarks per CTA until every SM has one (a rank of an 8-GPU run owns 1/8 of the landmarks: its
    // linearisation then takes one batch time instead of two)
    int G = cfg->num_ctas > 0 ? cfg->num_ctas : std::max(1, std::min(ctx->sm_count, (n_lm + LB - 1) / LB));
    G = std::max(1, std::min(G, std::max(1, n_lm)));
    std::vector<int> ranges(G + 1, n_lm);
    ranges[0] = 0;
    {
        const long total = deg_e[n_lm];
        int l = 0;
        for (int g = 1; g < G; ++g) {
            const long target = total * g / G;
            while (l < n_lm && deg_e[l] < target) ++l;
            ranges[g] = l;
        }
        ranges[G] = n_lm;
    }
    const int n_pairs = n_free * (n_free + 1) / 2;
    std::vector<int> pair_bi(n_pairs), pair_bj(n_pairs);
    {
        int q = 0;
        for (int i = 0; i < n_free; ++i)
            for (int j = i; j < n_free; ++j) {
                pair_bi[q] = i;
                pair_bj[q] = j;
                ++q;
            }
    }
    const int world = comm ? ba_comm_world(comm) : 1, rank = comm ? ba_comm_rank(comm) : 0;
    const int packed_sum_len = n_pairs * 36 + 12 * n_free + 1;
    const int packed_len = (packed_sum_len + 1 + 31) & ~31;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    PLP_TRY(ba_prepare_kernels(n_free, n_pairs, pool_cap));
    plp_ba *b = new plp_ba();
    b->ctx = ctx;
    b->cfg = *cfg;
    b->comm = comm;
    b->n_kf = n_kf;
    b->n_pts = n_pts;
    b->n_lines = n_lines;
    b->n_pe = n_pe;
    b->n_le = n_le;
    // ---- lay out one device block
    BaDev &D = b->dev;
    memset(&D, 0, sizeof(D));
    Layout lay;
    const size_t P1 = std::max(n_pts, 1), L1 = std::max(n_lines, 1), E1 = std::max(n_pe, 1), F1 = std::max(n_le, 1);
    const size_t PL1 = std::max(p->n_plane_edges, 1);
    lay.out(D.kf_hidx, n_kf);
    lay.out(D.poses[0], n_kf);
    lay.out(D.poses[1], n_kf);
    lay.out(D.pert_pose, (size_t)n_kf * 12);
    lay.out(D.pair_bi, n_pairs);
    lay.out(D.pair_bj, n_pairs);
    lay.out(D.pts[0], P1 * 3);
    lay.out(D.pts[1], P1 * 3);
    lay.out(D.lines[0], L1 * 6);
    lay.out(D.lines[1], L1 * 6);
    lay.out(D.pt_off, P1 + 1);
    lay.out(D.pt_kf, E1);
    lay.out(D.pt_lm, E1);
    lay.out(D.pt_obs, E1 * 3);
    lay.out(D.pt_info, E1);
    lay.out(D.pt_level, E1);
    lay.out(D.pt_outlier, E1);
    lay.out(D.pt_chi2, E1);
    lay.out(D.pt_W, E1 * 24);
    lay.out(D.pt_Dinv, P1 * 16);
    lay.out(D.pt_bl, P1 * 4);
    lay.out(D.pt_active, P1);
    lay.out(D.pt_plane, P1);
    lay.out(D.pl_fn, PL1 * 4);
    lay.out(D.pl_err, PL1);
    lay.out(D.ln_off, L1 + 1);
    lay.out(D.ln_kf, F1);
    lay.out(D.ln_lm, F1);
    lay.out(D.ln_obs, F1 * 4);
    lay.out(D.ln_info, F1);
    lay.out(D.ln_level, F1);
    lay.out(D.ln_outlier, F1);
    lay.out(D.ln_chi2, F1);
    lay.out(D.ln_W, F1 * 24);
    lay.out(D.ln_Dinv, L1 * 16);
    lay.out(D.ln_bl, L1 * 4);
    lay.out(D.ln_active, L1);
    lay.out(D.cta_ranges, (size_t)G + 1);
    lay.out(D.partial, large ? 8 : (size_t)G * packed_len);
    lay.out(D.dense, large ? ba_dense_bytes(n_free) / 8 : 8);
    lay.out(D.packed, (size_t)packed_sum_len + world + 8);
    lay.out(D.dp, (size_t)6 * std::max(n_free, kBaMaxFree));
    lay.out(D.trial_partial, (size_t)G * 2);
    lay.out(D.trial_sum, 8);
    lay.out(D.state, 1);
    lay.out(b->d_T_in, (size_t)n_kf * 16);
    lay.out(b->d_pts_in, P1 * 3);
    lay.out(b->d_lines_in, L1 * 6);
    lay.out(b->d_T_out, (size_t)n_kf * 16);
    lay.out(b->d_pts_out, P1 * 3);
    lay.out(b->d_lines_out, L1 * 6);
    lay.out(b->d_stop, 8);
    if (cudaMalloc((void **)&b->d_block, lay.bytes()) != cudaSuccess) {
        set_error("local BA: cudaMalloc(%zu) failed", lay.bytes());
        delete b;
        return PLP_ERR_CUDA;
    }
    b->block_bytes = lay.bytes();
    lay.bind(b->d_block);
    if (cudaMallocHost((void **)&b->h_state, sizeof(BaState)) != cudaSuccess ||
        cudaMallocHost((void **)&b->h_stop, 16) != cudaSuccess) {
        set_error("local BA: cudaMallocHost failed");
        plp_ba_destroy(b);
        return PLP_ERR_CUDA;
    }
    cudaError_t up_err = cudaMemsetAsync(b->d_block, 0, lay.bytes(), ctx->stream);
    auto up = [&](const auto *dst, const auto *src, size_t n) {
        static_assert(std::is_same<std::decay_t<decltype(*dst)>, std::decay_t<decltype(*src)>>::value, "types differ");
        if (n && up_err == cudaSuccess)
            up_err = cudaMemcpyAsync((void *)dst, src, n * sizeof(*src), cudaMemcpyHostToDevice, ctx->stream);
    };
    up(D.kf_hidx, hidx.data(), n_kf);
    up(D.pair_bi, pair_bi.data(), n_pairs);
    up(D.pair_bj, pair_bj.data(), n_pairs);
    up(D.pt_off, pt_off.data(), (size_t)n_pts + 1);
    up(D.pt_kf, p->pt_edge_kf, n_pe);
    up(D.pt_lm, p->pt_edge_lm, n_pe);
    up(D.pt_obs, p->pt_edge_obs, (size_t)n_pe * 3);
    up(D.pt_info, p->pt_edge_inv_sigma_sq, n_pe);
    up(D.pt_plane, pt_plane.data(), n_pts);
    up(D.pl_fn, p->plane_edge_fn, (size_t)p->n_plane_edges * 4);
    up(D.ln_off, ln_off.data(), (size_t)n_lines + 1);
    up(D.ln_kf, p->line_edge_kf, n_le);
    up(D.ln_lm, p->line_edge_lm, n_le);
    up(D.ln_obs, p->line_edge_obs, (size_t)n_le * 4);
    up(D.ln_info, p->line_edge_inv_sigma_sq, n_le);
    up(D.cta_ranges, ranges.data(), (size_t)G + 1);
    up(b->d_T_in, p->kf_pose_cw, (size_t)n_kf * 16);
    up(b->d_pts_in, p->pt_pos_w, (size_t)n_pts * 3);
    up(b->d_lines_in, p->line_plucker, (size_t)n_lines * 6);
    if (up_err == cudaSuccess) up_err = cudaStreamSynchronize(ctx->stream);
    if (up_err != cudaSuccess) {
        set_error("local BA: upload failed: %s", cudaGetErrorString(up_err));
        plp_ba_destroy(b);
        return PLP_ERR_CUDA;
    }
    if (!p->n_plane_edges) D.pt_plane = nullptr;
    D.fx = p->fx;
    D.fy = p->fy;
    D.cx = p->cx;
    D.cy = p->cy;
    D.bf = p->focal_x_baseline;
    D.delta_pt = p->setup_type == 0 ? (double)sqrtf(5.99146f) : (double)sqrtf(7.81473f);
    D.delta_ln = (double)sqrtf(5.99146f);
    D.n_kf = n_kf;
    D.n_free = n_free;
    D.n_pairs = n_pairs;
    D.n_pts = n_pts;
    D.n_lines = n_lines;
    D.n_pt_edges = n_pe;
    D.n_ln_edges = n_le;
    D.n_pl_edges = p->n_plane_edges;
    D.num_ctas = G;
    D.batch_landmarks = LB;
    D.pool_cap = pool_cap;
    D.packed_len = packed_len;
    D.packed_sum_len = packed_sum_len;
    D.rank = rank;
    D.world = world;
    D.large = large ? 1 : 0;
    D.phase_init_grid = 64;
    *out = b;
    return PLP_OK;
}

// mode 0: local BA (optimize(first) with Huber, outlier classification, optimize(second) without);
// mode 1 / 2: global BA = one optimize(first) with (1) / without (2) the Huber kernel, no outlier rounds
static plp_status ba_solve_impl(plp_ba *b, volatile const uint8_t *force_stop, plp_ba_result *r, int mode);

plp_status plp_ba_solve(plp_ba *b, volatile const uint8_t *force_stop, plp_ba_result *r) {
    return ba_solve_impl(b, force_stop, r, 0);
}

static plp_status ba_solve_impl(plp_ba *b, volatile const uint8_t *force_stop, plp_ba_result *r, int mode) {
    PLP_REQUIRE(b && r, "null pointer");
    plp_ctx *ctx = b->ctx;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const BaDev &D = b->dev;
    // (re)initialise the estimate and the edge levels
    PLP_TRY(ba_launch_init_poses(ctx, D, b->d_T_in));
    if (b->n_pts) PLP_CUDA_TRY(cudaMemcpyAsync(D.pts[0], b->d_pts_in, (size_t)b->n_pts * 24, cudaMemcpyDeviceToDevice, ctx->stream));
    if (b->n_lines)
        PLP_CUDA_TRY(cudaMemcpyAsync(D.lines[0], b->d_lines_in, (size_t)b->n_lines * 48, cudaMemcpyDeviceToDevice, ctx->stream));
    if (b->n_pe) PLP_CUDA_TRY(cudaMemsetAsync(D.pt_level, 0, b->n_pe, ctx->stream));
    if (b->n_le) PLP_CUDA_TRY(cudaMemsetAsync(D.ln_level, 0, b->n_le, ctx->stream));
    if (b->n_pe) PLP_CUDA_TRY(cudaMemsetAsync(D.pt_outlier, 0, b->n_pe, ctx->stream));
    if (b->n_le) PLP_CUDA_TRY(cudaMemsetAsync(D.ln_outlier, 0, b->n_le, ctx->stream));
    r->iters_first = r->iters_second = r->lm_tries = 0;
    r->final_chi2 = 0;
    bool stop0 = false;  // local_bundle_adjuster.cc:276-282
    if (force_stop || b->comm) PLP_TRY(stop_requested(b, force_stop, &stop0));
    if (!stop0) {
        int it1 = 0, it2 = 0;
        bool stopped = false;
        PLP_TRY(run_optimize(b, b->cfg.num_first_iter, mode == 2 ? 0 : 1, true, force_stop, &it1, &stopped));
        r->iters_first = it1;
        if (!stopped && mode == 0 && (force_stop || b->comm)) PLP_TRY(stop_requested(b, force_stop, &stopped));
        if (mode != 0) {
            // global_bundle_adjuster.cc:247-253: a single optimize(num_iter); edges keep level 0
        } else if (!stopped) {  // :289-337
            PLP_TRY(ba_launch_classify(ctx, D, 1));
            PLP_TRY(run_optimize(b, b->cfg.num_second_iter, 0, false, force_stop, &it2, &stopped));
            r->iters_second = it2;
        }
        if (mode == 0) PLP_TRY(ba_launch_classify(ctx, D, 0));
        r->lm_tries = b->h_state->tries;
        r->final_chi2 = b->h_state->current_chi;
    } else {
        PLP_TRY(ba_launch_set_state(ctx, D, 0, 1, 1));
    }
    // export the current estimate and download
    PLP_TRY(ba_launch_export(ctx, D, b->d_T_out, b->d_pts_out, b->d_lines_out));
    if (r->kf_pose_cw) PLP_CUDA_TRY(cudaMemcpyAsync(r->kf_pose_cw, b->d_T_out, (size_t)b->n_kf * 128, cudaMemcpyDeviceToHost, ctx->stream));
    if (r->pt_pos_w && b->n_pts)
        PLP_CUDA_TRY(cudaMemcpyAsync(r->pt_pos_w, b->d_pts_out, (size_t)b->n_pts * 24, cudaMemcpyDeviceToHost, ctx->stream));
    if (r->line_plucker && b->n_lines)
        PLP_CUDA_TRY(cudaMemcpyAsync(r->line_plucker, b->d_lines_out, (size_t)b->n_lines * 48, cudaMemcpyDeviceToHost, ctx->stream));
    if (r->pt_edge_outlier && b->n_pe)
        PLP_CUDA_TRY(cudaMemcpyAsync(r->pt_edge_outlier, D.pt_outlier, (size_t)b->n_pe, cudaMemcpyDeviceToHost, ctx->stream));
    if (r->line_edge_outlier && b->n_le)
        PLP_CUDA_TRY(cudaMemcpyAsync(r->line_edge_outlier, D.ln_outlier, (size_t)b->n_le, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return PLP_OK;
}

/* LM tries only (no download): `tries` tries of the first optimize() phase on the current state.  Used by the
 * throughput benchmark (LM iterations per second) -- each try is one full linearise + Schur + solve + update. */
plp_status plp_ba_bench_tries(plp_ba *b, int tries, int32_t *iters_done, int32_t *tries_done) {
    PLP_REQUIRE(b && tries >= 1, "args");
    plp_ctx *ctx = b->ctx;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    BaCollective *coll = b->comm ? ba_comm_collective(b->comm) : nullptr;
    const BaDev &D = b->dev;
    PLP_TRY(ba_launch_init_poses(ctx, D, b->d_T_in));
    if (b->n_pts) PLP_CUDA_TRY(cudaMemcpyAsync(D.pts[0], b->d_pts_in, (size_t)b->n_pts * 24, cudaMemcpyDeviceToDevice, ctx->stream));
    if (b->n_lines)
        PLP_CUDA_TRY(cudaMemcpyAsync(D.lines[0], b->d_lines_in, (size_t)b->n_lines * 48, cudaMemcpyDeviceToDevice, ctx->stream));
    if (b->n_pe) PLP_CUDA_TRY(cudaMemsetAsync(D.pt_level, 0, b->n_pe, ctx->stream));
    if (b->n_le) PLP_CUDA_TRY(cudaMemsetAsync(D.ln_level, 0, b->n_le, ctx->stream));
    PLP_TRY(ba_launch_set_state(ctx, D, 1 << 28, 1, 1));
    (void)coll;
    for (int t = 0; t < tries + 1; ++t) PLP_TRY(launch_try(b));  // +1: the lambda-init try
    PLP_TRY(ba_launch_decide(ctx, D));
    PLP_TRY(read_state(b));
    if (iters_done) *iters_done = b->h_state->it;
    if (tries_done) *tries_done = b->h_state->tries;
    return PLP_OK;
}

plp_status plp_global_ba(plp_ctx *ctx, const plp_ba_problem *p, int num_iter, int use_huber_kernel,
                         volatile const uint8_t *force_stop, plp_ba_result *r) {
    PLP_REQUIRE(num_iter >= 0, "num_iter");
    const plp_ba_cfg cfg{num_iter, 0, 0};
    plp_ba *b = nullptr;
    PLP_TRY(plp_ba_create(ctx, p, &cfg, nullptr, &b));
    const plp_status s = ba_solve_impl(b, force_stop, r, use_huber_kernel ? 1 : 2);
    plp_ba_destroy(b);
    return s;
}

plp_status plp_local_ba(plp_ctx *ctx, const plp_ba_problem *p, const plp_ba_cfg *cfg, volatile const uint8_t *force_stop,
                        plp_ba_result *r) {
    plp_ba *b = nullptr;
    PLP_TRY(plp_ba_create(ctx, p, cfg, nullptr, &b));
    const plp_status s = plp_ba_solve(b, force_stop, r);
    plp_ba_destroy(b);
    return s;
}

}  // extern "C"
