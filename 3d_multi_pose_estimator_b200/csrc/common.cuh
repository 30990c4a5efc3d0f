// Shared helpers for the b200pose kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/b200pose.h"

namespace b200pose {

void set_error(const char* fmt, ...);

#define B2_CHECK_ARG(cond, ...)                                   \
    do {                                                          \
        if (!(cond)) {                                            \
            b200pose::set_error(__VA_ARGS__);                     \
            return B200POSE_E_INVALID;                            \
        }                                                         \
    } while (0)

#define B2_CHECK_CUDA(expr)                                                                  \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            b200pose::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                                __FILE__, __LINE__);                                         \
            return B200POSE_E_CUDA;                                                          \
        }                                                                                    \
    } while (0)

#define B2_CHECK_LAUNCH() B2_CHECK_CUDA(cudaGetLastError())

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// fp32 -> (hi, lo) bf16 planes: hi = rn(x), lo = rn(x - hi). x - hi is exact in fp32.
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
    hi = __float2bfloat16_rn(x);
    lo = __float2bfloat16_rn(x - __bfloat162float(hi));
}

__device__ __forceinline__ uint32_t pack_bf16x2(__nv_bfloat16 a, __nv_bfloat16 b) {
    return (uint32_t)__bfloat16_as_ushort(a) | ((uint32_t)__bfloat16_as_ushort(b) << 16);
}

// two fp32 -> packed (hi, hi) and (lo, lo) bf16x2 words (element 0 in the low half): same rounding as split_bf16,
// but one packed convert per pair and the hi values recovered by bit operations
__device__ __forceinline__ void split_pack2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xffff0000u);
    const __nv_bfloat162 l = __floats2bfloat162_rn(x0 - h0, x1 - h1);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ float leaky(float x, float slope) { return x >= 0.f ? x : x * slope; }
// LeakyReLU for 0 <= slope <= 1: max(x, slope*x) (two instructions, no predicate)
__device__ __forceinline__ float leaky_le1(float x, float slope) { return fmaxf(x, x * slope); }

}  // namespace b200pose
