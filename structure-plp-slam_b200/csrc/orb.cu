// orb.cu -- ORB extraction on sm_100a: pyramid -> per-cell FAST -> quadtree selection -> orientation ->
// 7x7 Gaussian -> steered BRIEF.  Replaces feature::orb_extractor::extract (feature/orb_extractor.cc:73-160
// and the helpers it calls, orb_extractor_node.cc:31-80, util/trigonometric.h:42-78) bit-exactly.
//
// Batched from day one: every kernel has the frame index as its outermost grid dimension, so one launch
// covers `batch` frames.  11 launches per batch (10 when one quadtree instance serves every level):
//   7 x pyr_resize_kernel     level l from level l-1 (chained like orb_extractor.cc:315-326), OpenCV's
//                             11-bit fixed-point bilinear
//   1 x fast_cells_kernel     one CTA per 64-px cell (6-px overlap, orb_extractor.cc:338-437): tile -> smem,
//                             FAST-9/16 score, 3x3 NMS at the initial threshold, fallback to the minimum
//                             threshold if the cell is empty, ordered compaction (row-major inside the cell)
//   2 x quadtree_kernel       one CTA per (level, frame): data-parallel formulation of
//                             distribute_keypoints_via_tree (see tools/quadtree_parallel_model.py), in
//                             orb_quadtree.cuh; one launch for the large levels, one for the small ones
//   1 x describe_kernel       one warp per keypoint: intensity-centroid angle, 45x45 patch -> separable Q8
//                             Gaussian in smem -> 256 steered comparisons, one descriptor byte per lane
// Compiled with -fmad=false: the f32 steering must round exactly like the oracle (no FMA).
#include "common.cuh"
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched with cudaGetDriverEntryPoint, no libcuda link)
#include <stdlib.h>
#include "brief_pattern.inc"
#include "orb_quadtree.cuh"

namespace plp {

namespace {

constexpr int kMaxLevels = qt::kMaxLevels;
constexpr int kPatchRadius = qt::kPatchRadius;  // orb_extractor.h:161 orb_patch_radius_
constexpr int kHalfPatch = 15;     // orb_extractor.h:158 fast_half_patch_size_
constexpr int kCellSize = 64;      // orb_extractor.cc:339
constexpr int kOverlap = 6;        // orb_extractor.cc:338
constexpr int kCellCap = qt::kCellCap;  // max NMS survivors of a 64x64 tested area
constexpr int kTilePitch = 80;
constexpr int kTileRows = 70;

struct LevelInfo {
    int w, h, pitch;
    size_t offset;        // byte offset of the level inside one frame's pyramid block (levels >= 1)
    size_t blur_offset;   // byte offset of the level inside one frame's blurred-pyramid block (all levels)
    int cells_x, cells_y; // number of cell columns/rows visited (orb_extractor.cc:356-357)
    int cell_base;        // index of this level's first cell in the per-frame cell list
    int num_cells;
    int budget;           // num_keypts_per_level_
    int slot_base;        // first output slot of this level (per-level keypoint lists)
    int slot_cap;
    float scale_factor;
    float size;           // keypoint size = (unsigned)(31 * scale)
};

struct CellDesc {
    short level, i, j, pad;
    short min_x, min_y, max_x, max_y;
};

struct BlurTile {  // one 64 x 32 output tile of the Gaussian-blurred pyramid
    short level, x0, y0, pad;
};

using qt::LevelKp;  // quadtree output, level coordinates (border already added)

struct OrbDev {
    int num_levels, rows, cols;
    int num_cells;       // per frame
    int total_slots;     // per frame
    int out_cap;         // per frame capacity of the final kp/desc arrays
    int ini_thr, min_thr;
    LevelInfo lv[kMaxLevels];
    int u_max[16];
    // per-batch inputs
    const uint8_t *img0;  // level 0 = the caller's images
    size_t img0_step, img0_frame_stride;
    const uint8_t *mask;  // optional, level-0 resolution, shared by the batch
    size_t mask_step;
    // device work areas
    uint8_t *pyr;  // batch x pyr_frame_bytes (levels >= 1)
    size_t pyr_frame_bytes;
    uint8_t *blur;  // batch x blur_frame_bytes: GaussianBlur(7x7, sigma 2) of every level (orb_extractor.cc:148-149)
    size_t blur_frame_bytes;
    const BlurTile *blur_tiles;
    int num_blur_tiles;
    const CellDesc *cells;
    uint32_t *cell_buf;   // batch x num_cells x kCellCap packed (x:11 | y:10 | score:8)
    int *cell_cnt;        // batch x num_cells
    LevelKp *lvl_kp;      // batch x total_slots
    int *lvl_cnt;         // batch x num_levels
    uint8_t *qt_scratch;  // global fallback work area of the quadtree kernel
    int *status;          // batch: != 0 on capacity overflow
};

__device__ __forceinline__ const uint8_t *level_ptr(const OrbDev &P, int b, int l) {
    return l == 0 ? P.img0 + (size_t)b * P.img0_frame_stride : P.pyr + (size_t)b * P.pyr_frame_bytes + P.lv[l].offset;
}
__device__ __forceinline__ int level_pitch(const OrbDev &P, int l) { return l == 0 ? (int)P.img0_step : P.lv[l].pitch; }

// =====================================================================================================
// 1. pyramid: cv::resize(INTER_LINEAR) fixed-point model (SURVEY.md Appendix A.1)
// =====================================================================================================
// tables: per destination column {sx0, sx1, a0, a1}, per destination row {sy0, sy1, b0, b1}
// A thread owns four destination columns of kResizeRows consecutive rows: the column taps and weights are row-independent,
// so they are unpacked once per strip (round 1 redid the table loads, the unpacking and the 64-bit address arithmetic for
// every row: 58 instructions per pixel).
constexpr int kResizeRows = 8;
__global__ void __launch_bounds__(256) pyr_resize_kernel(OrbDev P, int l, const short4 *__restrict__ xtab,
                                                         const short4 *__restrict__ ytab) {
    const int b = blockIdx.y;
    const int dw = P.lv[l].w, dh = P.lv[l].h, dpitch = P.lv[l].pitch;
    const int quads = (dw + 3) >> 2, strips = (dh + kResizeRows - 1) / kResizeRows;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= quads * strips) return;
    const int strip = q / quads, x0 = (q - strip * quads) * 4;
    const uint8_t *src = level_ptr(P, b, l - 1);
    const int spitch = level_pitch(P, l - 1);
    uint8_t *dst = const_cast<uint8_t *>(level_ptr(P, b, l));
    int sx0[4], sx1[4], a0[4], a1[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const short4 xt = xtab[min(x0 + k, dw - 1)];  // columns past dw are row padding: any value may be stored there
        sx0[k] = xt.x;
        sx1[k] = xt.y;
        a0[k] = xt.z;
        a1[k] = xt.w;
    }
    const int y_end = min(dh, (strip + 1) * kResizeRows);
    for (int y = strip * kResizeRows; y < y_end; ++y) {
        const short4 yt = ytab[y];
        const uint8_t *S0 = src + (size_t)yt.x * spitch, *S1 = src + (size_t)yt.y * spitch;
        const int b0 = yt.z, b1 = yt.w;
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int r0 = S0[sx0[k]] * a0[k] + S0[sx1[k]] * a1[k];
            const int r1 = S1[sx0[k]] * a0[k] + S1[sx1[k]] * a1[k];
            const int v = (((b0 * (r0 >> 4)) >> 16) + ((b1 * (r1 >> 4)) >> 16) + 2) >> 2;
            packed |= (uint32_t)(v & 0xff) << (8 * k);
        }
        // pitch is a multiple of 64 so the 4-byte store is aligned; pad bytes past dw are never read
        *reinterpret_cast<uint32_t *>(dst + (size_t)y * dpitch + x0) = packed;
    }
}

// =====================================================================================================
// 2. FAST-9/16 per cell
// =====================================================================================================
// FAST-9/16 ring (SURVEY.md Appendix A.2): offsets (dx, dy) of ring pixel k = 0 .. 15, starting below the centre, counter-clockwise:
//   (0,3) (1,3) (2,2) (3,1) (3,0) (3,-1) (2,-2) (1,-3) (0,-3) (-1,-3) (-2,-2) (-3,-1) (-3,0) (-3,1) (-2,2) (-1,3)
// m = max over the sixteen 9-arcs of min(arc differences), both polarities (d = v - ring for dark arcs, e = ring - v for bright
// ones); the sliding minimum of length 9 over the circular ring is built by doubling (2, 4, 4 + 4 + 1).  Written with minima
// and a bias instead of negations: ptxas 12.9 for sm_100a miscompiles max(a, -max(...)) (drops the negation when fusing
// into VIMNMX3), see DESIGN.md.
// The score of TWO pixels at once on packed 16-bit halves (DPX min / max, VIMNMX3.S16x2): every difference is biased
// by +256 so that both halves stay in [1, 511] -- plain 32-bit subtraction then never borrows across the halves and no
// negation is needed (e' = 512 - d').  Returns (m_a + 256) | (m_b + 256) << 16 with m = max over the sixteen 9-arcs of
// min(arc differences), both polarities; the pixel is a corner at threshold t  <=>  m > t  (a 9-arc whose pixels all
// differ by more than t has a minimum above t and vice versa), which is the FAST-9 arc test.
__device__ __forceinline__ uint32_t fast_m_pair(const uint8_t *pa, const uint8_t *pb) {
    const uint32_t v2 = ((uint32_t)pa[0] + 256u) | (((uint32_t)pb[0] + 256u) << 16);
    uint32_t d[16];
#define PLP_RING(k, off) d[k] = v2 - ((uint32_t)pa[off] | ((uint32_t)pb[off] << 16))
    PLP_RING(0, 3 * kTilePitch);
    PLP_RING(1, 3 * kTilePitch + 1);
    PLP_RING(2, 2 * kTilePitch + 2);
    PLP_RING(3, 1 * kTilePitch + 3);
    PLP_RING(4, 3);
    PLP_RING(5, -1 * kTilePitch + 3);
    PLP_RING(6, -2 * kTilePitch + 2);
    PLP_RING(7, -3 * kTilePitch + 1);
    PLP_RING(8, -3 * kTilePitch);
    PLP_RING(9, -3 * kTilePitch - 1);
    PLP_RING(10, -2 * kTilePitch - 2);
    PLP_RING(11, -1 * kTilePitch - 3);
    PLP_RING(12, -3);
    PLP_RING(13, 1 * kTilePitch - 3);
    PLP_RING(14, 2 * kTilePitch - 2);
    PLP_RING(15, 3 * kTilePitch - 1);
#undef PLP_RING
    uint32_t e[16], d2[16], e2[16], d4[16], e4[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) e[k] = 0x02000200u - d[k];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        d2[k] = __vimin3_s16x2(d[k], d[(k + 1) & 15], d[(k + 1) & 15]);
        e2[k] = __vimin3_s16x2(e[k], e[(k + 1) & 15], e[(k + 1) & 15]);
    }
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        d4[k] = __vimin3_s16x2(d2[k], d2[(k + 2) & 15], d2[(k + 2) & 15]);
        e4[k] = __vimin3_s16x2(e2[k], e2[(k + 2) & 15], e2[(k + 2) & 15]);
    }
    uint32_t best = 0u;
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const uint32_t d9 = __vimin3_s16x2(d4[k], d4[(k + 4) & 15], d[(k + 8) & 15]);
        const uint32_t e9 = __vimin3_s16x2(e4[k], e4[(k + 4) & 15], e[(k + 8) & 15]);
        best = __vimax3_s16x2(best, d9, e9);
    }
    return best;
}

__device__ __forceinline__ bool masked(const OrbDev &P, unsigned y, unsigned x, float scale) {
    // orb_extractor.cc:333-336 is_in_mask
    return P.mask[(size_t)(int)(y * scale) * P.mask_step + (int)(x * scale)] == 0;
}


// ---------------------------------------------------------------------------------------------------------------
// fast_cells_kernel_v2: same cell semantics, fewer instructions per pixel.
//   phase A  four pixels per lane on aligned 32-bit shared-memory words; the pretest is the sign-agnostic compass
//            condition "two ADJACENT compass pixels differ from the centre by more than t" evaluated with the native
//            VABSDIFF4 byte SIMD -- a necessary condition for a FAST-9 corner (a 9-arc covers two adjacent compass
//            pixels, all darker or all brighter), phase B decides exactly;
//   NMS      only over the corners found (they set bits in the per-(row, half) masks with atomicOr -- a bit mask is
//            order independent, so the row-major output order is unchanged);
//   output   one thread per mask word walks its set bits.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t compass4(const uint32_t *T32, int y, int g, uint32_t t4) {
    constexpr int kPitchW = kTilePitch / 4;
    const uint32_t *row = T32 + y * kPitchW;
    const uint32_t c = row[g], up = row[g - 3 * kPitchW], dn = row[g + 3 * kPitchW];
    const uint32_t wl = g > 0 ? row[g - 1] : 0u, wr = row[g + 1];
    const uint32_t lf = __funnelshift_r(wl, c, 8);   // bytes x-3 .. x   of the four pixels x = 4g .. 4g+3
    const uint32_t rt = __funnelshift_r(c, wr, 24);  // bytes x+3 .. x+6
    const uint32_t a0 = __vcmpgtu4(__vabsdiffu4(c, dn), t4), a4 = __vcmpgtu4(__vabsdiffu4(c, rt), t4);
    const uint32_t a8 = __vcmpgtu4(__vabsdiffu4(c, up), t4), a12 = __vcmpgtu4(__vabsdiffu4(c, lf), t4);
    const uint32_t sv = (a4 | a12) & (a0 | a8);  // the four adjacent pairs (0,4) (4,8) (8,12) (12,0)
    const uint32_t m = sv & 0x01010101u;
    return (m | (m >> 7) | (m >> 14) | (m >> 21)) & 0xfu;
}

// Stronger byte-SIMD pretest (thresholds < 128): a 9-arc covers at least FOUR CONSECUTIVE of the eight even ring pixels
// (0, 2, .., 14), which must then all differ from the centre by more than t -- a necessary condition for a FAST-9 corner
// that rejects about three times as many pixels as the compass pair, so that the scalar arc test (250 instructions)
// runs on few of them.  |ring - c| with the native VABSDIFF4; "byte > t" as ((x & 0x7f) + (0x7f - t) | x) & 0x80.
__device__ __forceinline__ uint32_t even8_4(const uint32_t *T32, int y, int g, uint32_t k7) {
    constexpr int kPitchW = kTilePitch / 4;
    const uint32_t *row = T32 + y * kPitchW + g;
    const uint32_t c = row[0];
    const uint32_t wl = g > 0 ? row[-1] : 0u, wr = row[1];
    const uint32_t *rp2 = row + 2 * kPitchW, *rm2 = row - 2 * kPitchW;
    const uint32_t p2l = g > 0 ? rp2[-1] : 0u, m2l = g > 0 ? rm2[-1] : 0u;
    auto gt = [&](uint32_t ring) -> uint32_t {
        const uint32_t d = __vabsdiffu4(c, ring);
        return (((d & 0x7f7f7f7fu) + k7) | d) & 0x80808080u;
    };
    const uint32_t e0 = gt(row[3 * kPitchW]);                      // ( 0, +3)
    const uint32_t e2 = gt(__funnelshift_r(rp2[0], rp2[1], 16));   // (+2, +2)
    const uint32_t e4 = gt(__funnelshift_r(c, wr, 24));            // (+3,  0)
    const uint32_t e6 = gt(__funnelshift_r(rm2[0], rm2[1], 16));   // (+2, -2)
    const uint32_t e8 = gt(row[-3 * kPitchW]);                     // ( 0, -3)
    const uint32_t e10 = gt(__funnelshift_r(m2l, rm2[0], 16));     // (-2, -2)
    const uint32_t e12 = gt(__funnelshift_r(wl, c, 8));            // (-3,  0)
    const uint32_t e14 = gt(__funnelshift_r(p2l, rp2[0], 16));     // (-2, +2)
    const uint32_t p0 = e0 & e2, p2 = e2 & e4, p4 = e4 & e6, p6 = e6 & e8, p8 = e8 & e10, p10 = e10 & e12, p12 = e12 & e14,
                   p14 = e14 & e0;
    const uint32_t r = (p0 & p4) | (p2 & p6) | (p4 & p8) | (p6 & p10) | (p8 & p12) | (p10 & p14) | (p12 & p0) | (p14 & p2);
    return ((r >> 7) | (r >> 14) | (r >> 21) | (r >> 28)) & 0xfu;
}

__global__ void __launch_bounds__(256, 4) fast_cells_kernel_v2(OrbDev P) {
    __shared__ __align__(16) uint8_t tile[kTileRows * kTilePitch];
    __shared__ __align__(16) uint8_t score[kTileRows * kTilePitch];
    __shared__ int s_total[2];
    __shared__ unsigned short s_list[4096 + 8];  // tile offsets of the pixels that survive the pretest
    __shared__ int s_nsurv;
    __shared__ unsigned s_rowbits[128];  // NMS survivors: one 32-bit mask per (tested row, 32-column half)
    __shared__ int s_rowbase[128];
    const int b = blockIdx.y, ci = blockIdx.x, tid = threadIdx.x;
    const CellDesc cell = P.cells[ci];
    const int l = cell.level;
    const int w = cell.max_x - cell.min_x, h = cell.max_y - cell.min_y;
    int *cnt_out = P.cell_cnt + (size_t)b * P.num_cells + ci;
    uint32_t *buf = P.cell_buf + ((size_t)b * P.num_cells + ci) * kCellCap;
    const float scale = P.lv[l].scale_factor;
    bool skip = (w < 7 || h < 7);
    if (!skip && P.mask) {  // orb_extractor.cc:395-401
        skip = masked(P, cell.min_y, cell.min_x, scale) || masked(P, cell.max_y, cell.min_x, scale) ||
               masked(P, cell.min_y, cell.max_x, scale) || masked(P, cell.max_y, cell.max_x, scale);
    }
    if (skip) {
        if (tid == 0) *cnt_out = 0;
        return;
    }
    const uint8_t *img = level_ptr(P, b, l);
    const int pitch = level_pitch(P, l);
    const int lane = tid & 31, warp = tid >> 5;
    // tile load.  Level pitches are 64-byte multiples and cells start at x = 19 + 64 j, so a tile row is fetched as
    // aligned 16-byte chunks starting xo = min_x & 15 (= 3) bytes to the left of the cell; the tile keeps that offset
    // (tile column = cell column + xo).  The chunks read [min_x - xo, min_x + w + 15) at most: left of it lie >= 16 border
    // pixels, and max_x + 15 <= cols - 4, so no read leaves the image row.  Unaligned caller buffers take the byte path.
    const bool vec = (((uintptr_t)img | (uintptr_t)pitch) & 15) == 0 && (cell.min_x & 15) + w <= kTilePitch;
    const int xo = vec ? (cell.min_x & 15) : 0;
    if (vec) {
        const int nchunks = (xo + w + 15) >> 4;  // <= 5 (xo + w <= 73 <= kTilePitch)
        for (int idx = tid; idx < h * nchunks; idx += 256) {
            const int y = idx / nchunks, c = idx - y * nchunks;
            const uint4 v = __ldg(reinterpret_cast<const uint4 *>(img + (size_t)(cell.min_y + y) * pitch + (cell.min_x - xo)) + c);
            *reinterpret_cast<uint4 *>(tile + y * kTilePitch + 16 * c) = v;
        }
    } else {
        for (int y = warp; y < h; y += 8) {
            const uint8_t *src = img + (size_t)(cell.min_y + y) * pitch + cell.min_x;
            for (int x = lane; x < w; x += 32) tile[y * kTilePitch + x] = src[x];
        }
    }
    for (int idx = tid; idx < kTileRows * kTilePitch / 4; idx += 256) reinterpret_cast<uint32_t *>(score)[idx] = 0;
    const int tw = w - 6, th = h - 6;  // tested area: rows 3 .. h-4, columns 3 .. w-4 (<= 64 x 64)
    const int halves = tw > 32 ? 2 : 1;
    const int x_lo = 3 + xo, x_hi = 3 + xo + tw;  // tested tile columns
    const uint32_t *T32 = reinterpret_cast<const uint32_t *>(tile);
    // append the pixels of `nib` (bits = pixels 4g .. 4g+3 of row y) to the survivor list.  The order of the list is
    // irrelevant (scores and NMS bits are per pixel, the output order comes from the row masks), so a lane with survivors
    // simply reserves its slots with one shared-memory atomic
    auto append = [&](uint32_t nib, int y, int g) {
        if (!nib) return;
        int pos = atomicAdd(&s_nsurv, __popc(nib));
        while (nib) {
            const int bit = __ffs(nib) - 1;
            nib &= nib - 1;
            s_list[pos++] = (unsigned short)(y * kTilePitch + 4 * g + bit);
        }
    };
    auto valid_nibble = [&](int g) -> uint32_t {
        const int lo = max(0, x_lo - 4 * g), hi = min(4, x_hi - 4 * g);
        return hi > lo ? (((1u << hi) - 1u) & ~((1u << lo) - 1u)) : 0u;
    };
    for (int pass = 0; pass < 2; ++pass) {
        const int thr = pass == 0 ? P.ini_thr : P.min_thr;
        const uint32_t t4 = (uint32_t)min(thr, 255) * 0x01010101u;
        const bool strong = thr < 128;  // the SWAR "byte > t" of even8_4 needs t < 128
        const uint32_t k7 = (uint32_t)(0x7f - min(thr, 127)) * 0x01010101u;
        if (tid < 128) s_rowbits[tid] = 0u;
        if (tid == 0) s_nsurv = 0;
        if (pass == 1)  // scores of the first pass must not leak into the second (cv::FAST runs from scratch)
            for (int idx = tid; idx < kTileRows * kTilePitch / 4; idx += 256) reinterpret_cast<uint32_t *>(score)[idx] = 0;
        __syncthreads();
        // phase A: a warp takes two rows, a lane four pixels (word groups 0 .. 15 = columns 0 .. 63)
        for (int rp = warp; rp < (th + 1) / 2; rp += 8) {
            const int ry = 2 * rp + (lane >> 4), g = lane & 15;
            uint32_t nib = 0;
            if (ry < th) nib = (strong ? even8_4(T32, 3 + ry, g, k7) : compass4(T32, 3 + ry, g, t4)) & valid_nibble(g);
            append(nib, 3 + ry, g);
        }
        for (int g = 16; 4 * g < x_hi; ++g) {  // word groups 16, 17 (tile columns 64 .. 71), one thread per row
            for (int base = 0; base < th; base += 256) {
                const int ry = base + tid;
                uint32_t nib = 0;
                if (ry < th) nib = (strong ? even8_4(T32, 3 + ry, g, k7) : compass4(T32, 3 + ry, g, t4)) & valid_nibble(g);
                append(nib, 3 + ry, g);
            }
        }
        __syncthreads();
        // phase B: exact arc test / score for the survivors
        const int nsurv = s_nsurv;
        {  // a thread scores two survivors at once (packed 16-bit halves)
            const int half = (nsurv + 1) >> 1;
            for (int i = tid; i < half; i += 256) {
                const int off_a = s_list[i];
                const bool has_b = i + half < nsurv;
                const int off_b = has_b ? s_list[i + half] : off_a;
                const uint32_t m2 = fast_m_pair(tile + off_a, tile + off_b);
                const int m_a = (int)(m2 & 0xffffu) - 256, m_b = (int)(m2 >> 16) - 256;
                if (m_a > thr) score[off_a] = (uint8_t)(m_a - 1);
                if (has_b && m_b > thr) score[off_b] = (uint8_t)(m_b - 1);
            }
        }
        __syncthreads();
        // 3x3 non-maximum suppression over the corners only
        bool any_local = false;
        for (int i = tid; i < nsurv; i += 256) {
            const int off = s_list[i];
            const uint8_t *sp = score + off;
            const int sc = sp[0];
            if (sc == 0) continue;
            bool keep = true;
#pragma unroll
            for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
                for (int dx = -1; dx <= 1; ++dx) {
                    if (dx == 0 && dy == 0) continue;
                    keep = keep && (sc > (int)sp[dy * kTilePitch + dx]);
                }
            if (keep) {
                const int y = off / kTilePitch, xx = off - y * kTilePitch - 3 - xo;
                atomicOr(&s_rowbits[(y - 3) * 2 + (xx >> 5)], 1u << (xx & 31));
                any_local = true;
            }
        }
        const int any = __syncthreads_or(any_local);
        if (any || P.min_thr == P.ini_thr) break;
    }
    const int njobs = th * halves;
    // per-keypoint mask test (orb_extractor.cc:429): one thread per mask word
    if (P.mask) {
        for (int jdx = tid; jdx < njobs; jdx += 256) {
            const int ry = jdx / halves, hx = jdx - ry * halves;
            unsigned bits = s_rowbits[ry * 2 + hx], keepbits = bits;
            while (bits) {
                const int bit = __ffs(bits) - 1;
                bits &= bits - 1;
                const int x = 3 + hx * 32 + bit, y = 3 + ry;
                const float kx = (float)x + (float)(cell.j * kCellSize), ky = (float)y + (float)(cell.i * kCellSize);
                if (masked(P, (unsigned)((float)kPatchRadius + ky), (unsigned)((float)kPatchRadius + kx), scale))
                    keepbits &= ~(1u << bit);
            }
            s_rowbits[ry * 2 + hx] = keepbits;
        }
        __syncthreads();
    }
    // exclusive prefix of the per-(row, half) counts (<= 128 entries) by warp 0
    if (warp == 0) {
        int run = 0;
        for (int base = 0; base < njobs; base += 32) {
            const int jdx = base + lane;
            const int ry = jdx / halves, hx = jdx - ry * halves;
            const int c = jdx < njobs ? __popc(s_rowbits[ry * 2 + hx]) : 0;
            int incl = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += v;
            }
            if (jdx < njobs) s_rowbase[jdx] = run + incl - c;
            run += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0) s_total[0] = run;
    }
    __syncthreads();
    // ordered (row-major) output: one thread per mask word walks its bits
    for (int jdx = tid; jdx < njobs; jdx += 256) {
        const int ry = jdx / halves, hx = jdx - ry * halves;
        unsigned bits = s_rowbits[ry * 2 + hx];
        int pos = s_rowbase[jdx];
        while (bits) {
            const int bit = __ffs(bits) - 1;
            bits &= bits - 1;
            const int x = 3 + hx * 32 + bit, y = 3 + ry;
            const int sc = score[y * kTilePitch + x + xo];
            const int lx = x + cell.j * kCellSize, ly = y + cell.i * kCellSize;  // relative to the 19-px border
            if (pos < kCellCap) buf[pos] = (uint32_t)lx | ((uint32_t)ly << 11) | ((uint32_t)sc << 21);
            ++pos;
        }
    }
    if (tid == 0) *cnt_out = min(s_total[0], kCellCap);
}

// =====================================================================================================
// 3. quadtree keypoint distribution (orb_quadtree.cuh)
// =====================================================================================================
// One instance of quadtree_kernel: <threads, node capacity, shared-memory candidate window, resident CTAs per SM>.
template <int kThreads, int NC, int CC, int kMinBlocks>
struct QtInstance {
    static constexpr int kNodes = NC;
    static constexpr size_t kSmem = qt::qt_smem_bytes<kThreads, NC, CC>();
    static const void *fn() { return (const void *)qt::quadtree_kernel<kThreads, NC, CC, kMinBlocks>; }
    static void launch(dim3 grid, cudaStream_t s, const qt::QtDev &D) {
        qt::quadtree_kernel<kThreads, NC, CC, kMinBlocks><<<grid, kThreads, kSmem, s>>>(D);
    }
};
// Any configuration (max_num_keypts up to ~2300 at scale 1.2): 226 KB of shared memory, one CTA per SM.
using QtLarge = QtInstance<512, 2048, 8192, 1>;
// The level-sized pair, used when every level fits one of them: levels needing up to 1024 nodes (0-2 of the default
// 1000-keypoint configuration; at most 1374 candidates seen there) on 71 KB / 3 CTAs per SM, the rest on 54 KB / 4 CTAs
// per SM.  The kernel is a chain of block scans and barriers, so its throughput grows with the number of resident CTAs.
using QtWide = QtInstance<256, 1024, 1664, 3>;
using QtNarrow = QtInstance<256, 512, 2048, 4>;
constexpr int kNodeCap = QtLarge::kNodes;

// =====================================================================================================
// 4. orientation + blur + steered BRIEF, one warp per keypoint
// =====================================================================================================
constexpr int kDescWarps = 4;
constexpr int kBlurDim = 39, kBlurPitch = 44;  // window rows are staged as 11 aligned words

__device__ __forceinline__ int reflect101(int p, int len) {
    if (p < 0) p = -p;
    if (p >= len) p = 2 * (len - 1) - p;
    return p;
}

// cv::fastAtan2 (SURVEY.md Appendix A.7), f32, no FMA
__device__ __forceinline__ float fast_atan2_deg(float y, float x) {
    const float scale = (float)(180.0 / 3.14159265358979323846);
    const float p1 = 0.9997878412794807f * scale, p3 = -0.3258083974640975f * scale,
                p5 = 0.1555786518463281f * scale, p7 = -0.04432655554792128f * scale;
    const float ax = fabsf(x), ay = fabsf(y);
    float a, c, c2;
    if (ax >= ay) {
        c = __fdiv_rn(ay, ax + (float)2.2204460492503131e-16);
        c2 = c * c;
        a = (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    } else {
        c = __fdiv_rn(ax, ay + (float)2.2204460492503131e-16);
        c2 = c * c;
        a = 90.f - (((p7 * c2 + p5) * c2 + p3) * c2 + p1) * c;
    }
    if (x < 0) a = 180.f - a;
    if (y < 0) a = 360.f - a;
    return a;
}

// util/trigonometric.h:42-78
__device__ __forceinline__ float poly_cos(float v) {
    const float c1 = 0.99940307f, c2 = -0.49558072f, c3 = 0.03679168f;
    const float v2 = v * v;
    return c1 + v2 * (c2 + c3 * v2);
}
__device__ __forceinline__ float util_cos(float v) {
    const float PI = 3.14159265358979f, PI_2 = PI / 2.0f, TWO_PI = 2.0f * PI, INV_TWO_PI = 1.0f / TWO_PI,
                THREE_PI_2 = 3.0f * PI_2;
    v = v - (float)cv_floor((double)(v * INV_TWO_PI)) * TWO_PI;
    v = (0.0f < v) ? v : -v;
    if (v < PI_2) return poly_cos(v);
    if (v < PI) return -poly_cos(PI - v);
    if (v < THREE_PI_2) return -poly_cos(v - PI);
    return poly_cos(TWO_PI - v);
}
__device__ __forceinline__ float util_sin(float v) {
    const float PI_2 = 3.14159265358979f / 2.0f;
    return util_cos(PI_2 - v);
}

// cv::GaussianBlur(level, 7x7, sigma 2, BORDER_REFLECT_101) of every pyramid level (orb_extractor.cc:148-149) in
// OpenCV's fixed-point form: Q8 kernel [18 34 48 56 48 34 18], exact integer passes, (v + 32768) >> 16.
// One CTA per 64 x 32 output tile: 70 x 38 source tile -> smem, horizontal pass (u16), vertical pass, 32-bit stores.
constexpr int kBtW = 64, kBtH = 32;
__global__ void __launch_bounds__(256) blur_tiles_kernel(OrbDev P) {
    __shared__ __align__(16) uint8_t s_src[(kBtH + 6) * 72];
    __shared__ __align__(16) unsigned short s_h[(kBtH + 6) * kBtW];
    const int b = blockIdx.y, tid = threadIdx.x;
    const BlurTile t = P.blur_tiles[blockIdx.x];
    const int l = t.level, W = P.lv[l].w, H = P.lv[l].h;
    const uint8_t *img = level_ptr(P, b, l);
    const int pitch = level_pitch(P, l);
    for (int i = tid; i < (kBtH + 6) * 70; i += 256) {
        const int py = i / 70, px = i - py * 70;
        // rows / columns past the image edge + 3 only feed outputs that are never stored: clamp before reflecting
        const int gy = reflect101(min(t.y0 - 3 + py, H + 2), H), gx = reflect101(min(t.x0 - 3 + px, W + 2), W);
        s_src[py * 72 + px] = img[(size_t)gy * pitch + gx];
    }
    __syncthreads();
    for (int i = tid; i < (kBtH + 6) * kBtW; i += 256) {
        const int py = i / kBtW, px = i - py * kBtW;
        const uint8_t *s = s_src + py * 72 + px;
        s_h[i] = (unsigned short)(18 * (s[0] + s[6]) + 34 * (s[1] + s[5]) + 48 * (s[2] + s[4]) + 56 * s[3]);
    }
    __syncthreads();
    uint8_t *dst = P.blur + (size_t)b * P.blur_frame_bytes + P.lv[l].blur_offset;
    const int dpitch = P.lv[l].pitch;
    for (int i = tid; i < kBtH * kBtW / 4; i += 256) {
        const int py = i / (kBtW / 4), px = (i - py * (kBtW / 4)) * 4;
        if (t.y0 + py >= H || t.x0 + px >= W) continue;
        uint32_t packed = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const unsigned short *h = s_h + py * kBtW + px + k;
            const unsigned acc = 18u * (h[0] + h[6 * kBtW]) + 34u * (h[kBtW] + h[5 * kBtW]) + 48u * (h[2 * kBtW] + h[4 * kBtW]) +
                                 56u * h[3 * kBtW];
            packed |= ((acc + 32768u) >> 16) << (8 * k);
        }
        // pitch is a multiple of 64: aligned 4-byte store; bytes past the image width are padding
        *reinterpret_cast<uint32_t *>(dst + (size_t)(t.y0 + py) * dpitch + t.x0 + px) = packed;
    }
}

// ---- the same blur with the source tile staged by TMA and the passes on byte / half-word SIMD ---------------------
// One CTA per 64 x 32 output tile.  (1) ONE bulk tensor copy (cp.async.bulk.tensor.3d, box 96 x 38 x 1 of the
// (x, y, frame) tensor of the level) completes on an mbarrier -- no per-byte address arithmetic, no loads issued by the
// SMs.  The innermost coordinate of a tiled copy must be a multiple of 16 BYTES (measured with tools/probe/tma_probe.cu: an
// unaligned x raises "illegal instruction", any y -- negative included -- is accepted, out-of-image elements arrive as
// zeros), so the box is the 16-byte aligned superset [x0 - 16, x0 + 80) of the 70 columns the tile needs.
// (2) tiles that touch the image border rebuild BORDER_REFLECT_101 inside shared memory (the mirrored pixels are part of
// the same box).  (3) horizontal pass: a thread makes 4 outputs from 3 words with funnel shifts and DP4A
// ([18 34 48 56] . bytes + [48 34 18 0] . bytes); (4) vertical pass on the u16 rows; OpenCV's rounding (v + 32768) >> 16.
struct BlurMaps {
    CUtensorMap m[kMaxLevels];
};
constexpr int kBoxW = 96, kBoxH = kBtH + 6, kBoxX = 16;  // the box starts kBoxX columns left of the tile
static_assert(kBoxW >= kBoxX + kBtW + 3 && kBoxW % 16 == 0 && kBoxX % 16 == 0 && kBtW % 16 == 0,
              "TMA box: 16-byte aligned start and extent covering the 3-pixel halo");

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <bool kMapsInGlobal>
__global__ void __launch_bounds__(256) blur_tiles_tma_kernel(const __grid_constant__ BlurMaps M, const CUtensorMap *gmaps, OrbDev P) {
    __shared__ __align__(128) uint8_t s_src[kBoxH * kBoxW];
    __shared__ __align__(16) unsigned short s_h[kBoxH * kBtW];
    __shared__ __align__(8) unsigned long long s_bar;
    const int b = blockIdx.y, tid = threadIdx.x;
    const BlurTile t = P.blur_tiles[blockIdx.x];
    const int l = t.level, W = P.lv[l].w, H = P.lv[l].h;
    const int bx0 = t.x0 - kBoxX, by0 = t.y0 - 3;  // image coordinates of box element (0, 0)
    const uint32_t bar = smem_u32(&s_bar);
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        // the descriptor: a kernel parameter (__grid_constant__) or, with PLP_TMA_MAPS=global, an array in device memory
        // (acquired through the tensormap proxy, since the level-0 entry is rewritten when the caller's buffer changes)
        const CUtensorMap *tm = kMapsInGlobal ? gmaps + l : &M.m[l];
        if (kMapsInGlobal) asm volatile("fence.proxy.tensormap::generic.acquire.gpu [%0], 128;" ::"l"(tm) : "memory");
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(kBoxH * kBoxW) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            ::"r"(smem_u32(s_src)), "l"(tm), "r"(bx0), "r"(by0), "r"(b), "r"(bar)
            : "memory");
    }
    {
        uint32_t done = 0;
        for (int spin = 0; spin < (1 << 14) && !done; ++spin)
            asm volatile(
                "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(bar)
                : "memory");
        if (!done && tid == 0) P.status[b] = 3;  // the copy never completed: report it instead of hanging the device
    }
    if (t.x0 < 3 || by0 < 0 || t.x0 + kBtW + 3 > W || by0 + kBoxH > H) {  // BORDER_REFLECT_101 from inside the box
        // only the (at most) 3 + 3 halo columns and 3 + 3 halo rows the stored outputs read are rebuilt
        for (int i = tid; i < kBoxH * 6; i += 256) {
            const int py = i / 6, k = i - py * 6;
            const int gx = k < 3 ? k - 3 : W + (k - 3), gy = by0 + py;   // image columns -3 .. -1 and W .. W + 2
            const int px = gx - bx0;
            if (gy < 0 || gy >= H || px < 0 || px >= kBoxW) continue;
            s_src[py * kBoxW + px] = s_src[py * kBoxW + (reflect101(gx, W) - bx0)];
        }
        __syncthreads();
        for (int i = tid; i < 6 * kBoxW; i += 256) {
            const int k = i / kBoxW, px = i - k * kBoxW;
            const int gy = k < 3 ? k - 3 : H + (k - 3);                  // image rows -3 .. -1 and H .. H + 2
            const int py = gy - by0;
            if (py < 0 || py >= kBoxH) continue;
            s_src[py * kBoxW + px] = s_src[(reflect101(gy, H) - by0) * kBoxW + px];
        }
        __syncthreads();
    }
    // horizontal pass: output x of box row py uses box bytes x + 13 .. x + 19 (image columns x0 + x - 3 .. + 3); for the
    // outputs 4j .. 4j + 3 that is byte 1 of word j + 3 up to byte 2 of word j + 5
    const uint32_t *src32 = reinterpret_cast<const uint32_t *>(s_src);
    for (int i = tid; i < kBoxH * (kBtW / 4); i += 256) {
        const int py = i >> 4, j = i & 15;
        const uint32_t *w = src32 + py * (kBoxW / 4) + j + (kBoxX - 4) / 4;
        const uint32_t A = w[0], B = w[1], C = w[2];
        const uint32_t kW1 = 0x38302212u, kW2 = 0x00122230u;  // bytes (18, 34, 48, 56) and (48, 34, 18, 0)
        const uint32_t h0 = __dp4a(__funnelshift_r(A, B, 8), kW1, __dp4a(__funnelshift_r(B, C, 8), kW2, 0u));
        const uint32_t h1 = __dp4a(__funnelshift_r(A, B, 16), kW1, __dp4a(__funnelshift_r(B, C, 16), kW2, 0u));
        const uint32_t h2 = __dp4a(__funnelshift_r(A, B, 24), kW1, __dp4a(__funnelshift_r(B, C, 24), kW2, 0u));
        const uint32_t h3 = __dp4a(B, kW1, __dp4a(C, kW2, 0u));
        *reinterpret_cast<uint2 *>(s_h + py * kBtW + 4 * j) = make_uint2(h0 | (h1 << 16), h2 | (h3 << 16));
    }
    __syncthreads();
    uint8_t *dst = P.blur + (size_t)b * P.blur_frame_bytes + P.lv[l].blur_offset;
    const int dpitch = P.lv[l].pitch;
    for (int i = tid; i < kBtH * (kBtW / 4); i += 256) {
        const int py = i >> 4, px = (i & 15) * 4;
        if (t.y0 + py >= H || t.x0 + px >= W) continue;
        uint2 r[7];
#pragma unroll
        for (int k = 0; k < 7; ++k) r[k] = *reinterpret_cast<const uint2 *>(s_h + (py + k) * kBtW + px);
        uint32_t packed = 0;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            uint32_t h[7];
#pragma unroll
            for (int k = 0; k < 7; ++k) {
                const uint32_t w = (c < 2) ? r[k].x : r[k].y;
                h[k] = (c & 1) ? (w >> 16) : (w & 0xffffu);
            }
            const uint32_t acc = 18u * (h[0] + h[6]) + 34u * (h[1] + h[5]) + 48u * (h[2] + h[4]) + 56u * h[3];
            packed |= ((acc + 32768u) >> 16) << (8 * c);
        }
        // pitch is a multiple of 64: aligned 4-byte store; bytes past the image width are padding
        *reinterpret_cast<uint32_t *>(dst + (size_t)(t.y0 + py) * dpitch + t.x0 + px) = packed;
    }
}

__global__ void __launch_bounds__(kDescWarps * 32) describe_kernel(OrbDev P, plp_keypoint *__restrict__ kp_out,
                                                                    uint8_t *__restrict__ desc_out,
                                                                    int32_t *__restrict__ n_out) {
    __shared__ __align__(16) uint8_t s_win[kDescWarps][kBlurDim * kBlurPitch];
    const int b = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // per-level lookups staged once per block (dynamic indexing of the by-value parameter struct costs a constant-bank
    // load per use, and the per-keypoint level search re-read lvl_cnt from global memory)
    __shared__ int s_cum[kMaxLevels + 1];
    __shared__ const uint8_t *s_img[kMaxLevels], *s_blur[kMaxLevels];
    __shared__ int s_pitch[kMaxLevels], s_bpitch[kMaxLevels], s_slot[kMaxLevels];
    __shared__ float s_scale[kMaxLevels], s_size[kMaxLevels];
    if (threadIdx.x == 0) {
        const int *lvl_cnt = P.lvl_cnt + (size_t)b * P.num_levels;
        int acc = 0;
        for (int l = 0; l < P.num_levels; ++l) {
            s_cum[l] = acc;
            acc += lvl_cnt[l];
        }
        for (int l = P.num_levels; l <= kMaxLevels; ++l) s_cum[l] = acc;
    }
    if (threadIdx.x < P.num_levels) {
        const int l = threadIdx.x;
        s_img[l] = level_ptr(P, b, l);
        s_pitch[l] = level_pitch(P, l);
        s_blur[l] = P.blur + (size_t)b * P.blur_frame_bytes + P.lv[l].blur_offset;
        s_bpitch[l] = P.lv[l].pitch;
        s_slot[l] = P.lv[l].slot_base;
        s_scale[l] = P.lv[l].scale_factor;
        s_size[l] = P.lv[l].size;
    }
    __syncthreads();
    // total keypoints of the frame (level-major output order, orb_extractor.cc:137-159)
    const int total = min(s_cum[kMaxLevels], P.out_cap);
    if (blockIdx.x == 0 && threadIdx.x == 0) n_out[b] = total;
    const LevelKp *frame_kp = P.lvl_kp + (size_t)b * P.total_slots;
    // warps stride the ACTUAL keypoints of the frame (the slot space is 4x larger than what is normally used)
    for (int out_pos = blockIdx.x * kDescWarps + warp; out_pos < total; out_pos += gridDim.x * kDescWarps) {
    int l = 0;
    while (out_pos >= s_cum[l + 1]) ++l;
    const LevelKp kp = frame_kp[s_slot[l] + out_pos - s_cum[l]];
    const uint8_t *img = s_img[l];
    const int pitch = s_pitch[l];
    const int cx = kp.x, cy = kp.y;

    // ---- ic_angle (orb_extractor.cc:708-735): integer moments over the radius-15 disc; lanes = columns, the 31 row
    //      loads are fully unrolled (u_max of orb_extractor.cc:270-286 for the fixed half patch size 15)
    int m10 = 0, m01 = 0;
    {
        constexpr int kUmax[16] = {15, 15, 15, 15, 14, 14, 14, 13, 13, 12, 11, 10, 9, 8, 6, 3};
        const int u = lane - kHalfPatch;  // lanes 0..30 -> u = -15..15
        const int au = u < 0 ? -u : u;
        const uint8_t *c0 = img + (size_t)cy * pitch + cx + u;
#pragma unroll
        for (int v = -kHalfPatch; v <= kHalfPatch; ++v) {
            const int d = kUmax[v < 0 ? -v : v];
            if (lane < 31 && au <= d) {
                const int val = __ldg(c0 + v * pitch);
                m10 += u * val;
                m01 += v * val;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            m10 += __shfl_xor_sync(0xffffffffu, m10, o);
            m01 += __shfl_xor_sync(0xffffffffu, m01, o);
        }
    }
    const float angle = fast_atan2_deg((float)m01, (float)m10);

    // ---- steered BRIEF (orb_extractor.cc:747-807) on the Gaussian-blurred level (blur_tiles_kernel): lane i
    //      produces descriptor byte i; the 16 byte gathers of a lane fall inside a 37 x 37 window (L1-resident)
    const float ang_rad = (float)((double)angle * 3.14159265358979323846 / 180.0);
    const float ca = util_cos(ang_rad), sa = util_sin(ang_rad);
    const int bpitch = s_bpitch[l];
    // stage the 39 x 39 blurred window as the 4-byte-aligned superset of every row (rows of the blurred pyramid start
    // 64-byte aligned, so an aligned word never leaves its row): two rows per step, one word per lane, 20 load / store
    // pairs per keypoint instead of 156 byte pairs; then gather the 512 samples from shared memory
    const int wx0 = cx - 19, woff = wx0 & 3, nwords = (woff + kBlurDim + 3) >> 2;  // 10 or 11 words
    const uint8_t *bsrc = s_blur[l] + (size_t)(cy - 19) * bpitch + (wx0 - woff);
    uint8_t *win = s_win[warp];
    __syncwarp();
    {
        const int half = lane >> 4, j = lane & 15;
        if (j < nwords) {
#pragma unroll 5
            for (int r = half; r < kBlurDim; r += 2)
                *reinterpret_cast<uint32_t *>(win + r * kBlurPitch + 4 * j) =
                    __ldg(reinterpret_cast<const uint32_t *>(bsrc + (size_t)r * bpitch) + j);
        }
    }
    __syncwarp();
    const uint8_t *center = win + 19 * kBlurPitch + 19 + woff;
    int val = 0;
    // the lane's 8 test pairs: 8 consecutive int8 per table = one 64-bit load each (the tables live in global
    // memory: lane-dependent indices into __constant__ memory would serialise)
    const uint2 px1 = __ldg(reinterpret_cast<const uint2 *>(kBriefX1) + lane), py1 = __ldg(reinterpret_cast<const uint2 *>(kBriefY1) + lane);
    const uint2 px2 = __ldg(reinterpret_cast<const uint2 *>(kBriefX2) + lane), py2 = __ldg(reinterpret_cast<const uint2 *>(kBriefY2) + lane);
#pragma unroll
    for (int bit = 0; bit < 8; ++bit) {
        const int sh = (bit & 3) * 8;
        const float x1 = (float)(signed char)(((bit < 4 ? px1.x : px1.y) >> sh) & 0xff);
        const float y1 = (float)(signed char)(((bit < 4 ? py1.x : py1.y) >> sh) & 0xff);
        const float x2 = (float)(signed char)(((bit < 4 ? px2.x : px2.y) >> sh) & 0xff);
        const float y2 = (float)(signed char)(((bit < 4 ? py2.x : py2.y) >> sh) & 0xff);
        const int r1 = __float2int_rn(x1 * sa + y1 * ca), c1 = __float2int_rn(x1 * ca - y1 * sa);
        const int r2 = __float2int_rn(x2 * sa + y2 * ca), c2 = __float2int_rn(x2 * ca - y2 * sa);
        val |= (center[r1 * kBlurPitch + c1] < center[r2 * kBlurPitch + c2]) << bit;
    }
    desc_out[((size_t)b * P.out_cap + out_pos) * 32 + lane] = (uint8_t)val;
    if (lane == 0) {
        plp_keypoint o;
        const float s = s_scale[l];
        o.x = l == 0 ? (float)cx : (float)cx * s;  // orb_extractor.cc:695-706
        o.y = l == 0 ? (float)cy : (float)cy * s;
        o.size = s_size[l];
        o.angle = angle;
        o.response = (float)kp.response;
        o.octave = l;
        o.class_id = -1;
        kp_out[(size_t)b * P.out_cap + out_pos] = o;
    }
    }  // keypoint loop
}

}  // namespace

}  // namespace plp

// =========================================================================================================
// handle + C ABI
// =========================================================================================================
using namespace plp;

struct plp_orb {
    plp_ctx *ctx = nullptr;
    plp_orb_params params;
    int rows = 0, cols = 0, max_batch = 0;
    OrbDev dev;  // device pointers filled in at create
    std::vector<float> scale_factors, inv_scale_factors, level_sigma_sq, inv_level_sigma_sq;
    std::vector<uint32_t> num_keypts_per_level;
    std::vector<CellDesc> cells;
    short4 *d_xtab[kMaxLevels] = {nullptr};
    short4 *d_ytab[kMaxLevels] = {nullptr};
    CellDesc *d_cells = nullptr;
    uint8_t *d_pyr = nullptr;
    uint8_t *d_blur = nullptr;
    BlurTile *d_blur_tiles = nullptr;
    std::vector<BlurTile> blur_tiles;
    uint8_t *d_img = nullptr;  // staging for host-pointer extraction (max_batch frames)
    uint8_t *d_mask = nullptr;
    uint32_t *d_cell_buf = nullptr;
    int *d_cell_cnt = nullptr;
    LevelKp *d_lvl_kp = nullptr;
    int *d_lvl_cnt = nullptr;
    uint8_t *d_qt_scratch = nullptr;
    int *d_status = nullptr;
    plp_keypoint *d_kp = nullptr;
    uint8_t *d_desc = nullptr;
    int32_t *d_n = nullptr;
    qt::QtDev qt_dev;       // quadtree parameters (status is set per run)
    bool qt_large = false;  // every level runs on QtLarge (a level does not fit the level-sized pair, or PLP_QT_LARGE)
    int qt_split = 0;       // else levels [0, qt_split) run on QtWide, [qt_split, num_levels) on QtNarrow
    // TMA descriptors of the pyramid levels as (x, y, frame) uint8 tensors; levels >= 1 live in d_pyr (encoded once),
    // level 0 is the caller's buffer (re-encoded when its address / pitch / batch changes)
    BlurMaps maps;
    bool maps_ok = false;       // levels >= 1 encoded
    bool no_tma = false;        // PLP_BLUR_NO_TMA=1
    bool maps_global = false;   // PLP_TMA_MAPS=global: descriptors read from device memory instead of kernel parameters
    CUtensorMap *d_maps = nullptr;
    bool d_maps_dirty = true;
    const uint8_t *map0_img = nullptr;
    size_t map0_step = 0;
    int map0_batch = 0;
    int last_batch = 0;
    const uint8_t *last_img0 = nullptr;
    size_t last_step = 0;
};

// cuTensorMapEncodeTiled through the runtime's driver-entry-point lookup (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
    static EncodeTiledFn fn = []() -> EncodeTiledFn {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        return (EncodeTiledFn)p;
    }();
    return fn;
}
// (x, y, frame) uint8 tensor of one pyramid level; box = the blur kernel's source tile.  false when the buffer does not
// meet TMA's alignment rules (16-byte base and strides) -- the caller then uses the plain-load kernel for this batch.
static bool encode_level_map(CUtensorMap *m, const uint8_t *base, int w, int h, int frames, size_t pitch, size_t frame_stride) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc || ((uintptr_t)base & 15) || (pitch & 15) || (frame_stride & 15) || w < 1 || h < 1 || frames < 1) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)frames};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)frame_stride};
    const cuuint32_t box[3] = {(cuuint32_t)kBoxW, (cuuint32_t)kBoxH, 1u}, estr[3] = {1u, 1u, 1u};
    return enc(m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, (void *)base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}


static void build_resize_tables(int sw, int sh, int dw, int dh, std::vector<short4> &xt, std::vector<short4> &yt) {
    // cv::resize INTER_LINEAR 8U: 11-bit coefficients, rounded half-to-even (SURVEY.md Appendix A.1)
    const double inv_scale_x = (double)dw / sw, inv_scale_y = (double)dh / sh;
    const double scale_x = 1. / inv_scale_x, scale_y = 1. / inv_scale_y;
    xt.resize(dw);
    yt.resize(dh);
    for (int dx = 0; dx < dw; ++dx) {
        float fx = (float)((dx + 0.5) * scale_x - 0.5);
        int sx = cv_floor(fx);
        fx -= sx;
        if (sx < 0) {
            fx = 0;
            sx = 0;
        }
        if (sx >= sw - 1) {
            fx = 0;
            sx = sw - 1;
        }
        short4 t;
        t.x = (short)sx;
        t.y = (short)std::min(sx + 1, sw - 1);
        t.z = (short)lrintf((1.f - fx) * 2048);
        t.w = (short)lrintf(fx * 2048);
        xt[dx] = t;
    }
    for (int dy = 0; dy < dh; ++dy) {
        float fy = (float)((dy + 0.5) * scale_y - 0.5);
        int sy = cv_floor(fy);
        fy -= sy;
        short4 t;
        t.x = (short)std::min(std::max(sy, 0), sh - 1);
        t.y = (short)std::min(std::max(sy + 1, 0), sh - 1);
        t.z = (short)lrintf((1.f - fy) * 2048);
        t.w = (short)lrintf(fy * 2048);
        yt[dy] = t;
    }
}

extern "C" {

void plp_orb_destroy(plp_orb *o) {
    if (!o) return;
    cudaSetDevice(o->ctx->device);
    cudaStreamSynchronize(o->ctx->stream);
    for (int l = 0; l < kMaxLevels; ++l) {
        if (o->d_xtab[l]) cudaFree(o->d_xtab[l]);
        if (o->d_ytab[l]) cudaFree(o->d_ytab[l]);
    }
    void *ptrs[] = {o->d_blur, o->d_blur_tiles, o->d_cells, o->d_pyr, o->d_img, o->d_mask, o->d_cell_buf, o->d_cell_cnt, o->d_lvl_kp,
                    o->d_lvl_cnt, o->d_qt_scratch, o->d_status, o->d_kp, o->d_desc, o->d_n, o->d_maps};
    for (void *p : ptrs)
        if (p) cudaFree(p);
    delete o;
}

plp_status plp_orb_create(plp_ctx *ctx, const plp_orb_params *params, int rows, int cols, int max_batch,
                          plp_orb **out) {
    PLP_REQUIRE(ctx && params && out, "null pointer");
    *out = nullptr;
    PLP_REQUIRE(rows > 0 && cols > 0 && max_batch > 0, "image size / batch");
    PLP_REQUIRE(params->num_levels >= 1 && params->num_levels <= kMaxLevels, "num_levels in [1,16]");
    PLP_REQUIRE(params->scale_factor > 1.0f || params->num_levels == 1, "scale_factor > 1");
    PLP_REQUIRE(cols <= 2047 + 2 * kPatchRadius && rows <= 1023 + 2 * kPatchRadius,
                "image larger than 2085 x 1061 (packed candidate coordinates)");
    PLP_REQUIRE(params->ini_fast_thr < 255 && params->min_fast_thr >= 1 && params->min_fast_thr <= params->ini_fast_thr,
                "FAST thresholds: 1 <= min <= ini < 255");
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    plp_orb *o = new plp_orb();
    {
        const char *nt = getenv("PLP_BLUR_NO_TMA");
        o->no_tma = nt && nt[0] == '1';
        const char *mg = getenv("PLP_TMA_MAPS");
        o->maps_global = mg && mg[0] == 'g';
    }
    o->ctx = ctx;
    o->params = *params;
    o->rows = rows;
    o->cols = cols;
    o->max_batch = max_batch;
    const unsigned L = params->num_levels;
    // ---- orb_params.cc:86-128 scale tables
    o->scale_factors.assign(L, 1.0f);
    o->inv_scale_factors.assign(L, 1.0f);
    o->level_sigma_sq.assign(L, 1.0f);
    o->inv_level_sigma_sq.assign(L, 1.0f);
    for (unsigned l = 1; l < L; ++l) o->scale_factors[l] = params->scale_factor * o->scale_factors[l - 1];
    for (unsigned l = 1; l < L; ++l) o->inv_scale_factors[l] = (1.0f / params->scale_factor) * o->inv_scale_factors[l - 1];
    {
        float s = 1.0f;
        for (unsigned l = 1; l < L; ++l) {
            s = params->scale_factor * s;
            o->level_sigma_sq[l] = s * s;
            o->inv_level_sigma_sq[l] = 1.0f / (s * s);
        }
    }
    // ---- orb_extractor.cc:244-253 per-level budget
    o->num_keypts_per_level.resize(L);
    {
        double desired = params->max_num_keypts * (1.0 - 1.0 / params->scale_factor) /
                         (1.0 - std::pow(1.0 / params->scale_factor, static_cast<double>(L)));
        if (L == 1) desired = params->max_num_keypts;
        unsigned total = 0;
        for (unsigned l = 0; l + 1 < L; ++l) {
            o->num_keypts_per_level[l] = (unsigned)std::round(desired);
            total += o->num_keypts_per_level[l];
            desired *= 1.0 / params->scale_factor;
        }
        o->num_keypts_per_level[L - 1] = (unsigned)std::max((int)params->max_num_keypts - (int)total, 0);
    }
    OrbDev &D = o->dev;
    memset(&D, 0, sizeof(D));
    D.num_levels = (int)L;
    D.rows = rows;
    D.cols = cols;
    D.ini_thr = (int)params->ini_fast_thr;
    D.min_thr = (int)params->min_fast_thr;
    // ---- orb_extractor.cc:270-286 u_max
    {
        const unsigned vmax = (unsigned)std::floor(kHalfPatch * std::sqrt(2.0) / 2 + 1);
        const unsigned vmin = (unsigned)std::ceil(kHalfPatch * std::sqrt(2.0) / 2);
        for (unsigned v = 0; v <= vmax; ++v)
            D.u_max[v] = (int)std::round(std::sqrt((double)kHalfPatch * kHalfPatch - (double)v * v));
        for (unsigned v = kHalfPatch, v0 = 0; vmin <= v; --v) {
            while (D.u_max[v0] == D.u_max[v0 + 1]) ++v0;
            D.u_max[v] = (int)v0;
            ++v0;
        }
    }
    // ---- level geometry, cells (orb_extractor.cc:344-392)
    size_t pyr_bytes = 0, blur_bytes = 0;
    int slot_base = 0, cell_base = 0;
    plp_status st = PLP_OK;
    for (unsigned l = 0; l < L; ++l) {
        LevelInfo &V = D.lv[l];
        if (l == 0) {
            V.w = cols;
            V.h = rows;
        } else {
            const double scale = o->scale_factors[l];
            V.w = (int)std::round(cols * 1.0 / scale);
            V.h = (int)std::round(rows * 1.0 / scale);
        }
        V.pitch = (V.w + 63) & ~63;
        V.offset = pyr_bytes;
        if (l > 0) pyr_bytes += (size_t)V.pitch * V.h + 256;
        pyr_bytes = (pyr_bytes + 255) & ~(size_t)255;
        V.blur_offset = blur_bytes;
        blur_bytes += (size_t)V.pitch * V.h + 256;
        blur_bytes = (blur_bytes + 255) & ~(size_t)255;
        for (int y0 = 0; y0 < V.h; y0 += kBtH)
            for (int x0 = 0; x0 < V.w; x0 += kBtW) o->blur_tiles.push_back(BlurTile{(short)l, (short)x0, (short)y0, 0});
        V.budget = (int)o->num_keypts_per_level[l];
        V.scale_factor = o->scale_factors[l];
        V.size = (float)(unsigned)(31 * o->scale_factors[l]);
        V.slot_base = slot_base;
        {
            // initial nodes of the quadtree (orb_extractor.cc:561-582): one sweep can quadruple them
            int g0 = 1;
            if (V.w > 2 * kPatchRadius && V.h > 2 * kPatchRadius) {
                const double ratio = (double)(V.w - 2 * kPatchRadius) / (V.h - 2 * kPatchRadius);
                g0 = ratio > 1 ? (int)std::round(ratio) : (int)std::round(1 / ratio);
            }
            V.slot_cap = 4 * std::max(V.budget, g0) + 8;
        }
        slot_base += V.slot_cap;
        V.cell_base = cell_base;
        V.num_cells = 0;
        if (V.slot_cap > kNodeCap) {
            set_error("orb: level %u budget %d exceeds the quadtree node capacity", l, V.budget);
            st = PLP_ERR_CAPACITY;
        }
        if (V.w > 2 * kPatchRadius && V.h > 2 * kPatchRadius && V.w >= 1 && V.h >= 1) {
            const unsigned min_bx = kPatchRadius, min_by = kPatchRadius;
            const unsigned max_bx = V.w - kPatchRadius, max_by = V.h - kPatchRadius;
            const unsigned width = max_bx - min_bx, height = max_by - min_by;
            const unsigned ncols = width / kCellSize + 1, nrows = height / kCellSize + 1;
            V.cells_x = (int)ncols;
            V.cells_y = (int)nrows;
            for (unsigned i = 0; i < nrows; ++i) {
                const unsigned min_y = min_by + i * kCellSize;
                if (max_by - kOverlap <= min_y || max_by < kOverlap) continue;
                unsigned max_y = min_y + kCellSize + kOverlap;
                if (max_by < max_y) max_y = max_by;
                for (unsigned j = 0; j < ncols; ++j) {
                    const unsigned min_x = min_bx + j * kCellSize;
                    if (max_bx - kOverlap <= min_x || max_bx < kOverlap) continue;
                    unsigned max_x = min_x + kCellSize + kOverlap;
                    if (max_bx < max_x) max_x = max_bx;
                    CellDesc c;
                    c.level = (short)l;
                    c.i = (short)i;
                    c.j = (short)j;
                    c.pad = 0;
                    c.min_x = (short)min_x;
                    c.min_y = (short)min_y;
                    c.max_x = (short)max_x;
                    c.max_y = (short)max_y;
                    o->cells.push_back(c);
                    V.num_cells++;
                }
            }
        }
        cell_base += V.num_cells;
    }
    if (st != PLP_OK) {
        delete o;
        return st;
    }
    D.num_cells = cell_base;
    D.total_slots = slot_base;
    D.out_cap = slot_base;
    D.pyr_frame_bytes = pyr_bytes ? pyr_bytes : 256;
    D.blur_frame_bytes = blur_bytes ? blur_bytes : 256;
    D.num_blur_tiles = (int)o->blur_tiles.size();
    const size_t B = (size_t)max_batch;
    // ---- device allocations
#define ORB_ALLOC(ptr, bytes)                                              \
    do {                                                                   \
        cudaError_t e_ = cudaMalloc((void **)&(ptr), (bytes) ? (bytes) : 256); \
        if (e_ != cudaSuccess) {                                           \
            set_error("orb: cudaMalloc(%zu) failed: %s", (size_t)(bytes), cudaGetErrorString(e_)); \
            plp_orb_destroy(o);                                            \
            return PLP_ERR_CUDA;                                           \
        }                                                                  \
    } while (0)
    for (unsigned l = 1; l < L; ++l) {
        std::vector<short4> xt, yt;
        build_resize_tables(D.lv[l - 1].w, D.lv[l - 1].h, D.lv[l].w, D.lv[l].h, xt, yt);
        ORB_ALLOC(o->d_xtab[l], xt.size() * sizeof(short4));
        ORB_ALLOC(o->d_ytab[l], yt.size() * sizeof(short4));
        cudaMemcpy(o->d_xtab[l], xt.data(), xt.size() * sizeof(short4), cudaMemcpyHostToDevice);
        cudaMemcpy(o->d_ytab[l], yt.data(), yt.size() * sizeof(short4), cudaMemcpyHostToDevice);
    }
    ORB_ALLOC(o->d_cells, o->cells.size() * sizeof(CellDesc));
    if (!o->cells.empty())
        cudaMemcpy(o->d_cells, o->cells.data(), o->cells.size() * sizeof(CellDesc), cudaMemcpyHostToDevice);
    ORB_ALLOC(o->d_pyr, B * D.pyr_frame_bytes);
    ORB_ALLOC(o->d_blur, B * D.blur_frame_bytes);
    ORB_ALLOC(o->d_blur_tiles, o->blur_tiles.size() * sizeof(BlurTile));
    if (!o->blur_tiles.empty())
        cudaMemcpy(o->d_blur_tiles, o->blur_tiles.data(), o->blur_tiles.size() * sizeof(BlurTile), cudaMemcpyHostToDevice);
    ORB_ALLOC(o->d_img, B * (size_t)rows * cols);
    ORB_ALLOC(o->d_mask, (size_t)rows * cols);
    ORB_ALLOC(o->d_cell_buf, B * (size_t)D.num_cells * kCellCap * sizeof(uint32_t));
    ORB_ALLOC(o->d_cell_cnt, B * (size_t)D.num_cells * sizeof(int));
    ORB_ALLOC(o->d_lvl_kp, B * (size_t)D.total_slots * sizeof(LevelKp));
    ORB_ALLOC(o->d_lvl_cnt, B * L * sizeof(int));
    const size_t qt_scratch_per_job = (size_t)(qt::kMaxCands + 1) * qt::kBytesPerCand + 256;
    ORB_ALLOC(o->d_qt_scratch, B * L * qt_scratch_per_job);
    ORB_ALLOC(o->d_status, B * sizeof(int));
    ORB_ALLOC(o->d_maps, sizeof(BlurMaps));
    ORB_ALLOC(o->d_kp, B * (size_t)D.out_cap * sizeof(plp_keypoint));
    ORB_ALLOC(o->d_desc, B * (size_t)D.out_cap * 32);
    ORB_ALLOC(o->d_n, B * sizeof(int32_t));
#undef ORB_ALLOC
    D.pyr = o->d_pyr;
    D.blur = o->d_blur;
    D.blur_tiles = o->d_blur_tiles;
    D.cells = o->d_cells;
    D.cell_buf = o->d_cell_buf;
    D.cell_cnt = o->d_cell_cnt;
    D.lvl_kp = o->d_lvl_kp;
    D.lvl_cnt = o->d_lvl_cnt;
    D.qt_scratch = o->d_qt_scratch;
    D.status = o->d_status;
    // TMA descriptors of the levels that live in the handle's own pyramid block (level 0 follows the caller's buffer)
    o->maps_ok = true;
    memset(&o->maps, 0, sizeof(o->maps));
    for (unsigned l = 1; l < L && o->maps_ok; ++l)
        o->maps_ok = encode_level_map(&o->maps.m[l], o->d_pyr + D.lv[l].offset, D.lv[l].w, D.lv[l].h, max_batch, D.lv[l].pitch,
                                      D.pyr_frame_bytes);
    {
        qt::QtDev &Q = o->qt_dev;
        memset(&Q, 0, sizeof(Q));
        Q.num_levels = D.num_levels;
        Q.num_cells = D.num_cells;
        Q.total_slots = D.total_slots;
        for (unsigned l = 0; l < L; ++l)
            Q.lv[l] = qt::QtLevel{D.lv[l].w,      D.lv[l].h,         D.lv[l].cell_base, D.lv[l].num_cells,
                                  D.lv[l].budget, D.lv[l].slot_base, D.lv[l].slot_cap};
        Q.cell_buf = o->d_cell_buf;
        Q.cell_cnt = o->d_cell_cnt;
        Q.lvl_kp = o->d_lvl_kp;
        Q.lvl_cnt = o->d_lvl_cnt;
        Q.scratch = o->d_qt_scratch;
        Q.scratch_per_job = qt_scratch_per_job;
    }
    // a level fits an instance when its node need and its cell count (the gather's prefix lives in the node scratch) do
    auto fits = [&](unsigned l, int nodes) { return D.lv[l].slot_cap <= nodes && D.lv[l].num_cells <= nodes; };
    unsigned split = L;
    while (split > 0 && fits(split - 1, QtNarrow::kNodes)) --split;
    o->qt_large = getenv("PLP_QT_LARGE") != nullptr;
    for (unsigned l = 0; l < split; ++l) o->qt_large = o->qt_large || !fits(l, QtWide::kNodes);
    o->qt_split = (int)split;
    plp_status so;
    if (o->qt_large) {
        so = ensure_smem_optin(QtLarge::fn(), QtLarge::kSmem, "quadtree_kernel<large>");
    } else {
        so = ensure_smem_optin(QtWide::fn(), QtWide::kSmem, "quadtree_kernel<wide>");
        if (so == PLP_OK) so = ensure_smem_optin(QtNarrow::fn(), QtNarrow::kSmem, "quadtree_kernel<narrow>");
    }
    if (so != PLP_OK) {
        plp_orb_destroy(o);
        return so;
    }
    *out = o;
    return PLP_OK;
}

int plp_orb_capacity(const plp_orb *o) { return o ? o->dev.out_cap : 0; }

plp_status plp_orb_get_tables(const plp_orb *o, float *sf, float *isf, float *ls, float *ils, uint32_t *nk) {
    PLP_REQUIRE(o, "orb");
    for (int l = 0; l < o->dev.num_levels; ++l) {
        if (sf) sf[l] = o->scale_factors[l];
        if (isf) isf[l] = o->inv_scale_factors[l];
        if (ls) ls[l] = o->level_sigma_sq[l];
        if (ils) ils[l] = o->inv_level_sigma_sq[l];
        if (nk) nk[l] = o->num_keypts_per_level[l];
    }
    return PLP_OK;
}

static plp_status orb_run(plp_orb *o, const uint8_t *d_imgs, int batch, size_t step, const uint8_t *d_mask,
                          size_t mask_step, plp_keypoint *d_kp, uint8_t *d_desc, int32_t *d_n, int32_t *d_status) {
    plp_ctx *ctx = o->ctx;
    OrbDev D = o->dev;
    D.img0 = d_imgs;
    D.img0_step = step;
    D.img0_frame_stride = step * (size_t)o->rows;
    D.mask = d_mask;
    D.mask_step = mask_step;
    D.status = d_status ? d_status : o->d_status;
    o->last_batch = batch;
    o->last_img0 = d_imgs;
    o->last_step = step;
    PLP_CUDA_TRY(cudaMemsetAsync(D.status, 0, (size_t)batch * sizeof(int), ctx->stream));
    for (int l = 1; l < D.num_levels; ++l) {
        const int quads = ((D.lv[l].w + 3) >> 2) * ((D.lv[l].h + kResizeRows - 1) / kResizeRows);  // threads: 4 columns x 8 rows each
        if (quads <= 0) continue;
        dim3 grid(div_up(quads, 256), batch);
        PLP_LAUNCH(ctx, pyr_resize_kernel, grid, 256, 0, D, l, o->d_xtab[l], o->d_ytab[l]);
    }
    if (D.num_cells > 0) {
        dim3 grid(D.num_cells, batch);
        PLP_LAUNCH(ctx, fast_cells_kernel_v2, grid, 256, 0, D);
    }
    if (D.num_blur_tiles > 0) {
        dim3 grid(D.num_blur_tiles, batch);
        bool tma = o->maps_ok && !o->no_tma;
        if (tma && (o->map0_img != d_imgs || o->map0_step != step || o->map0_batch != batch)) {
            tma = encode_level_map(&o->maps.m[0], d_imgs, D.lv[0].w, D.lv[0].h, batch, step, D.img0_frame_stride);
            o->map0_img = tma ? d_imgs : nullptr;
            o->d_maps_dirty = true;
            o->map0_step = step;
            o->map0_batch = batch;
        }
        if (tma && o->maps_global) {
            if (o->d_maps_dirty) {
                PLP_CUDA_TRY(cudaMemcpyAsync(o->d_maps, &o->maps, sizeof(BlurMaps), cudaMemcpyHostToDevice, ctx->stream));
                o->d_maps_dirty = false;
            }
            PLP_LAUNCH(ctx, blur_tiles_tma_kernel<true>, grid, 256, 0, o->maps, o->d_maps, D);
        } else if (tma)
            PLP_LAUNCH(ctx, blur_tiles_tma_kernel<false>, grid, 256, 0, o->maps, (const CUtensorMap *)nullptr, D);
        else  // caller buffer not 16-byte aligned / pitched (or PLP_BLUR_NO_TMA=1 for A/B runs): plain loads
            PLP_LAUNCH(ctx, blur_tiles_kernel, grid, 256, 0, D);
    }
    {
        qt::QtDev Q = o->qt_dev;
        Q.status = D.status;
        // (PLP_LAUNCH spelled out: one timing name for every instance, one timed region for both launches)
        if (ctx->timing) plp::timing_begin(ctx, "quadtree_kernel");
        if (o->qt_large) {
            QtLarge::launch(dim3(D.num_levels, batch), ctx->stream, Q);
            ctx->launches++;
        } else {
            if (o->qt_split > 0) {
                QtWide::launch(dim3(o->qt_split, batch), ctx->stream, Q);
                ctx->launches++;
            }
            if (o->qt_split < D.num_levels) {
                Q.level_base = o->qt_split;
                QtNarrow::launch(dim3(D.num_levels - o->qt_split, batch), ctx->stream, Q);
                ctx->launches++;
            }
        }
        if (ctx->timing) plp::timing_end(ctx);
    }
    {
        const int kp_est = std::max(256, (int)(3 * o->params.max_num_keypts / 2));  // warps stride the rest
        dim3 grid(div_up(std::min(D.total_slots, kp_est), kDescWarps), batch);
        PLP_LAUNCH(ctx, describe_kernel, grid, kDescWarps * 32, 0, D, d_kp, d_desc, d_n);
    }
    PLP_CHECK_LAUNCH();
    return PLP_OK;
}

plp_status plp_orb_extract_batch_dev(plp_orb *o, const uint8_t *d_imgs, int batch, size_t step, plp_keypoint *d_kp,
                                     uint8_t *d_desc, int32_t *d_n, int32_t *d_status) {
    PLP_REQUIRE(o && d_imgs && d_kp && d_desc && d_n, "null pointer");
    PLP_REQUIRE(batch >= 1 && batch <= o->max_batch, "batch exceeds the handle's max_batch");
    PLP_REQUIRE(step >= (size_t)o->cols, "step < cols");
    PLP_CUDA_TRY(cudaSetDevice(o->ctx->device));
    return orb_run(o, d_imgs, batch, step, nullptr, 0, d_kp, d_desc, d_n, d_status);
}

static plp_status orb_extract_host(plp_orb *o, const uint8_t *imgs, int batch, size_t step, const uint8_t *mask,
                                   size_t mask_step, plp_keypoint *kp_out, uint8_t *desc_out, int32_t *n_out) {
    plp_ctx *ctx = o->ctx;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const size_t rows = o->rows, cols = o->cols;
    PLP_CUDA_TRY(cudaMemcpy2DAsync(o->d_img, cols, imgs, step, cols, rows * (size_t)batch, cudaMemcpyHostToDevice,
                                   ctx->stream));
    const uint8_t *d_mask = nullptr;
    if (mask) {
        PLP_CUDA_TRY(cudaMemcpy2DAsync(o->d_mask, cols, mask, mask_step, cols, rows, cudaMemcpyHostToDevice, ctx->stream));
        d_mask = o->d_mask;
    }
    PLP_TRY(orb_run(o, o->d_img, batch, cols, d_mask, cols, o->d_kp, o->d_desc, o->d_n, nullptr));
    const size_t cap = o->dev.out_cap;
    PLP_CUDA_TRY(cudaMemcpyAsync(n_out, o->d_n, (size_t)batch * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(kp_out, o->d_kp, (size_t)batch * cap * sizeof(plp_keypoint), cudaMemcpyDeviceToHost,
                                 ctx->stream));
    PLP_CUDA_TRY(cudaMemcpyAsync(desc_out, o->d_desc, (size_t)batch * cap * 32, cudaMemcpyDeviceToHost, ctx->stream));
    std::vector<int> status(batch);
    PLP_CUDA_TRY(cudaMemcpyAsync(status.data(), o->d_status, (size_t)batch * 4, cudaMemcpyDeviceToHost, ctx->stream));
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < batch; ++b)
        if (status[b] != 0) {
            set_error("orb: capacity overflow in frame %d (code %d)", b, status[b]);
            return PLP_ERR_CAPACITY;
        }
    return PLP_OK;
}

plp_status plp_orb_extract(plp_orb *o, const uint8_t *img, int rows, int cols, size_t step, const uint8_t *mask,
                           size_t mask_step, plp_keypoint *kp_out, uint8_t *desc_out, int *n_out) {
    PLP_REQUIRE(o && n_out, "null pointer");
    *n_out = 0;
    if (!img || rows == 0 || cols == 0) return PLP_OK;  // orb_extractor.cc:76-79
    PLP_REQUIRE(rows == o->rows && cols == o->cols, "image size differs from the handle's");
    PLP_REQUIRE(kp_out && desc_out, "null output");
    PLP_REQUIRE(step >= (size_t)cols && (!mask || mask_step >= (size_t)cols), "step < cols");
    int32_t n = 0;
    PLP_TRY(orb_extract_host(o, img, 1, step, mask, mask_step, kp_out, desc_out, &n));
    *n_out = n;
    return PLP_OK;
}

plp_status plp_orb_extract_batch(plp_orb *o, const uint8_t *imgs, int batch, size_t step, plp_keypoint *kp_out,
                                 uint8_t *desc_out, int32_t *n_out) {
    PLP_REQUIRE(o && imgs && kp_out && desc_out && n_out, "null pointer");
    PLP_REQUIRE(batch >= 1 && batch <= o->max_batch, "batch exceeds the handle's max_batch");
    PLP_REQUIRE(step >= (size_t)o->cols, "step < cols");
    return orb_extract_host(o, imgs, batch, step, nullptr, 0, kp_out, desc_out, n_out);
}

plp_status plp_orb_get_pyramid(const plp_orb *o, int b, int level, plp_image_view *out) {
    PLP_REQUIRE(o && out, "null pointer");
    PLP_REQUIRE(b >= 0 && b < o->last_batch && level >= 0 && level < o->dev.num_levels, "index");
    const LevelInfo &V = o->dev.lv[level];
    out->rows = V.h;
    out->cols = V.w;
    if (level == 0) {
        out->data = o->last_img0 + (size_t)b * o->last_step * o->rows;
        out->step = o->last_step;
    } else {
        out->data = o->d_pyr + (size_t)b * o->dev.pyr_frame_bytes + V.offset;
        out->step = V.pitch;
    }
    return PLP_OK;
}

plp_status plp_orb_debug_candidates(plp_orb *o, int b, int level, plp_keypoint *out, int cap, int *n_out) {
    PLP_REQUIRE(o && out && n_out, "null pointer");
    PLP_REQUIRE(b >= 0 && b < o->last_batch && level >= 0 && level < o->dev.num_levels, "index");
    plp_ctx *ctx = o->ctx;
    PLP_CUDA_TRY(cudaSetDevice(ctx->device));
    const LevelInfo &V = o->dev.lv[level];
    std::vector<int> cnt(V.num_cells);
    std::vector<uint32_t> buf((size_t)V.num_cells * kCellCap);
    PLP_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (V.num_cells) {
        PLP_CUDA_TRY(cudaMemcpy(cnt.data(), o->d_cell_cnt + (size_t)b * o->dev.num_cells + V.cell_base,
                                cnt.size() * 4, cudaMemcpyDeviceToHost));
        PLP_CUDA_TRY(cudaMemcpy(buf.data(), o->d_cell_buf + ((size_t)b * o->dev.num_cells + V.cell_base) * kCellCap,
                                buf.size() * 4, cudaMemcpyDeviceToHost));
    }
    int n = 0;
    for (int c = 0; c < V.num_cells; ++c)
        for (int k = 0; k < cnt[c]; ++k) {
            if (n < cap) {
                const uint32_t v = buf[(size_t)c * kCellCap + k];
                plp_keypoint kp;
                kp.x = (float)(v & 0x7ff);
                kp.y = (float)((v >> 11) & 0x3ff);
                kp.size = 7.f;
                kp.angle = -1.f;
                kp.response = (float)(v >> 21);
                kp.octave = 0;
                kp.class_id = -1;
                out[n] = kp;
            }
            ++n;
        }
    *n_out = n;
    return PLP_OK;
}

}  // extern "C"
