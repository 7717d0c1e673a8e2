// helpers shared by the fused stage kernels (device code only)
#pragma once
#include <cuda_fp16.h>

#include "umma_common.cuh"

namespace flo {

// k_chain: 8 epilogue warps (two per TMEM lane quadrant) + TMA producer + MMA issuer
constexpr int EPI_WARPS = 8;
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int FUSED_THREADS = EPI_THREADS + 64;

// ------------------------------------------------------------------------------------------------
// 16-bit helpers (fmt: 1 = bf16, 0 = fp16)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t pack2(float a, float b, int fmt) {
    if (fmt) {
        __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    }
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
__device__ __forceinline__ float2 unpack2(uint32_t u, int fmt) {
    if (fmt) return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&u));
    return __half22float2(*reinterpret_cast<__half2*>(&u));
}
__device__ __forceinline__ uint4 pack8(const float* v, int fmt) {
    return make_uint4(pack2(v[0], v[1], fmt), pack2(v[2], v[3], fmt), pack2(v[4], v[5], fmt), pack2(v[6], v[7], fmt));
}
__device__ __forceinline__ void unpack8(uint4 u, float* v, int fmt) {
    float2 a = unpack2(u.x, fmt), b = unpack2(u.y, fmt), c = unpack2(u.z, fmt), d = unpack2(u.w, fmt);
    v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
}
// compile-time format variants (k_chain is templated on the operand format: no per-element format branches)
template <int FMT>
__device__ __forceinline__ uint32_t pack2t(float a, float b) {
    if constexpr (FMT != 0) {
        __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    } else {
        __half2 h = __floats2half2_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&h);
    }
}
template <int FMT>
__device__ __forceinline__ uint4 pack8t(const float* v) {
    return make_uint4(pack2t<FMT>(v[0], v[1]), pack2t<FMT>(v[2], v[3]), pack2t<FMT>(v[4], v[5]), pack2t<FMT>(v[6], v[7]));
}
template <int FMT>
__device__ __forceinline__ void unpack8t(uint4 u, float* v) {
    if constexpr (FMT != 0) {
        // bf16 -> fp32 is a 16-bit shift: two integer ops per pair
        v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xFFFF0000u);
        v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xFFFF0000u);
        v[4] = __uint_as_float(u.z << 16); v[5] = __uint_as_float(u.z & 0xFFFF0000u);
        v[6] = __uint_as_float(u.w << 16); v[7] = __uint_as_float(u.w & 0xFFFF0000u);
    } else {
        const float2 a = __half22float2(*reinterpret_cast<__half2*>(&u.x)), b = __half22float2(*reinterpret_cast<__half2*>(&u.y));
        const float2 c = __half22float2(*reinterpret_cast<__half2*>(&u.z)), d = __half22float2(*reinterpret_cast<__half2*>(&u.w));
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; v[4] = c.x; v[5] = c.y; v[6] = d.x; v[7] = d.y;
    }
}
constexpr int ATTN_MAX_THREADS = 576;   // k_attn with 16 epilogue warps (16x16 level) + producer + MMA issuer
__device__ __forceinline__ void epi_sync() { named_bar_sync(1, EPI_THREADS); }



// Branch-free MUFU forms: the CUDA intrinsics add denormal-range fix-ups (predicated code and reconvergence
// points) that serialise the per-element chains of an unrolled epilogue loop.
__device__ __forceinline__ float fast_exp2(float x) {
    float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}
__device__ __forceinline__ float fast_exp(float x) { return fast_exp2(x * 1.4426950408889634f); }
__device__ __forceinline__ float fast_rcp(float x) {
    float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r;
}
// SiLU (unet.py:67 nn.SiLU): y * sigmoid(y)
__device__ __forceinline__ float fast_silu(float y) { return y * fast_rcp(1.0f + fast_exp(-y)); }

}  // namespace flo
