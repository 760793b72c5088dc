// devmath.cuh -- small device helpers shared by all kernels (256-bit Hamming, descriptor loads, OpenCV rounding,
// div_up).  Depends only on <stdint.h> and CUDA built-ins, so the kernel headers that include it can also be compiled by
// tests/cta_emu.
#pragma once
#include <stdint.h>

// dynamic shared memory of a kernel: `extern __shared__` on the device; tests/cta_emu hands out a host buffer instead
#ifdef PLP_CTA_EMU
#define PLP_DYNAMIC_SMEM(name) uint8_t *name = emu_dynamic_smem
#else
#define PLP_DYNAMIC_SMEM(name) extern __shared__ __align__(16) uint8_t name[]
#endif

namespace plp {

// ---- device helpers -------------------------------------------------------

// 256-bit Hamming distance between two descriptors held as 8 x u32
__device__ __forceinline__ int hamming256(const uint32_t a[8], const uint32_t b[8]) {
    int d = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) d += __popc(a[i] ^ b[i]);
    return d;
}

__device__ __forceinline__ int hamming256(const uint4 a0, const uint4 a1, const uint4 b0,
                                          const uint4 b1) {
    return __popc(a0.x ^ b0.x) + __popc(a0.y ^ b0.y) + __popc(a0.z ^ b0.z) + __popc(a0.w ^ b0.w) +
           __popc(a1.x ^ b1.x) + __popc(a1.y ^ b1.y) + __popc(a1.z ^ b1.z) + __popc(a1.w ^ b1.w);
}

// one 32-byte descriptor as two read-only 16-byte loads (p must be 16-byte aligned)
__device__ __forceinline__ void load_desc(const uint8_t *p, uint4 &a, uint4 &b) {
    const uint4 *q = reinterpret_cast<const uint4 *>(p);
    a = __ldg(q);
    b = __ldg(q + 1);
}

// cvFloor / cvCeil / cvRound for float and double (OpenCV semantics: floor, ceil, round-half-even)
__host__ __device__ __forceinline__ int cv_floor(double v) {
    int i = (int)v;
    return i - (i > v);
}
__host__ __device__ __forceinline__ int cv_ceil(double v) {
    int i = (int)v;
    return i + (i < v);
}
__device__ __forceinline__ int cv_round_f(float v) { return __float2int_rn(v); }
__device__ __forceinline__ int cv_round_d(double v) { return __double2int_rn(v); }

template <typename T>
__host__ __device__ __forceinline__ T div_up(T a, T b) {
    return (a + b - 1) / b;
}

}  // namespace plp
