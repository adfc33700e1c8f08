// Shared helpers for libbcad (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>

namespace bcad {

void set_error(const char* fmt, ...);

#define BCAD_CUDA_CHECK(expr)                                                              \
    do {                                                                                   \
        cudaError_t _e = (expr);                                                           \
        if (_e != cudaSuccess) {                                                           \
            bcad::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),        \
                            __FILE__, __LINE__);                                           \
            return BCAD_ERR_CUDA;                                                          \
        }                                                                                  \
    } while (0)

#define BCAD_REQUIRE(cond, ...)                                                            \
    do {                                                                                   \
        if (!(cond)) {                                                                     \
            bcad::set_error(__VA_ARGS__);                                                  \
            return BCAD_ERR_INVALID;                                                       \
        }                                                                                  \
    } while (0)

__host__ __device__ static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ int cdiv_dev(int a, int b) { return (a + b - 1) / b; }
__device__ __forceinline__ float leaky(float v, float alpha) { return v > 0.f ? v : alpha * v; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// streaming 128-bit load that does not pollute L1 (read-once data)
__device__ __forceinline__ float4 ldg_stream(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}

__device__ __forceinline__ float bf16lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&t);
}

__device__ __forceinline__ uint32_t pack_f16(float lo, float hi) {
    __half2 t = __floats2half2_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float2 unpack_f16(uint32_t v) {
    return __half22float2(*reinterpret_cast<const __half2*>(&v));
}
// undo a LeakyReLU (pre-activation Grad-CAM target): z = a > 0 ? a : a * inv_slope, the fp32 cam_kernel's form
__device__ __forceinline__ float2 unleaky2(float2 v, float inv_slope) {
    return make_float2(v.x > 0.f ? v.x : v.x * inv_slope, v.y > 0.f ? v.y : v.y * inv_slope);
}

}  // namespace bcad
