// quadtree_emu.cc -- csrc/orb_quadtree.cuh (the ORB extractor's quadtree keypoint distribution) executed on the host:
// one (level, frame) job through each kernel instance orb.cu launches, on candidates given as cell lists.
#include "cta_emu.h"

#include <string.h>

struct short4 {
    short x, y, z, w;
};

#include "orb_quadtree.cuh"

using namespace plp::qt;

template <int kThreads, int NC, int CC, int kMinBlocks>
static void run(QtDev P) {
    emu_launch2(quadtree_kernel<kThreads, NC, CC, kMinBlocks>, 1u, 1u, (unsigned)kThreads, qt_smem_bytes<kThreads, NC, CC>(), P);
}

// instance: 0 = <512, 2048, 8192> (any configuration), 1 = <256, 1024, 1664> (large levels), 2 = <256, 512, 2048> (small
// levels) -- the shapes of QtLarge, QtWide and QtNarrow in orb.cu.  cell_buf holds num_cells lists of kCellCap packed
// candidates (x:11 | y:10 | score:11, relative to the 19-px border).  Returns the number of keypoints written.
extern "C" int emu_quadtree(int instance, int w, int h, int budget, int slot_cap, int num_cells, const int *cell_cnt,
                            const uint32_t *cell_buf, short *out_x, short *out_y, int *out_resp, int *status) {
    std::vector<LevelKp> out((size_t)slot_cap);
    const size_t per_job = (size_t)(kMaxCands + 1) * kBytesPerCand + 256;
    std::vector<unsigned long long> scratch(per_job / 8 + 1);
    int lvl_cnt = -1;
    *status = 0;
    QtDev P;
    memset(&P, 0, sizeof(P));
    P.num_levels = 1;
    P.num_cells = num_cells;
    P.total_slots = slot_cap;
    P.lv[0] = QtLevel{w, h, 0, num_cells, budget, 0, slot_cap};
    P.cell_buf = cell_buf;
    P.cell_cnt = cell_cnt;
    P.lvl_kp = out.data();
    P.lvl_cnt = &lvl_cnt;
    P.scratch = reinterpret_cast<uint8_t *>(scratch.data());
    P.scratch_per_job = per_job;
    P.status = status;
    switch (instance) {
        case 0: run<512, 2048, 8192, 1>(P); break;
        case 1: run<256, 1024, 1664, 3>(P); break;
        case 2: run<256, 512, 2048, 4>(P); break;
        default: return -1;
    }
    for (int i = 0; i < lvl_cnt; ++i) {
        out_x[i] = out[i].x;
        out_y[i] = out[i].y;
        out_resp[i] = out[i].response;
    }
    return lvl_cnt;
}
