// Tensor-core building blocks shared by the HMMA kernels (sm_100a): ldmatrix / mma.sync / cp.async wrappers,
// 16-bit pack/unpack, and the fused GroupNorm-affine + SiLU.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace dg {

// ---- small PTX wrappers -------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2(uint32_t addr, uint32_t& r0, uint32_t& r1) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
template <typename T>
__device__ __forceinline__ void mma16816(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
    if constexpr (std::is_same<T, __half>::value) {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    } else {
        asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                     : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
    }
}
// m16n8k8: half-width K step (A: 16x8 = 2 registers, B: 8x8 = 1 register) -- used when one 3x3 tap contributes 8 channels
template <typename T>
__device__ __forceinline__ void mma16808(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t b0) {
    if constexpr (std::is_same<T, __half>::value) {
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(b0));
    } else {
        asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};"
                     : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a0), "r"(a1), "r"(b0));
    }
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

template <typename T> __device__ __forceinline__ uint32_t pack2(float a, float b);
template <> __device__ __forceinline__ uint32_t pack2<__half>(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <> __device__ __forceinline__ uint32_t pack2<__nv_bfloat16>(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
}
template <typename T> __device__ __forceinline__ float2 unpack2(uint32_t v);
template <> __device__ __forceinline__ float2 unpack2<__half>(uint32_t v) {
    return __half22float2(*reinterpret_cast<__half2*>(&v));
}
template <> __device__ __forceinline__ float2 unpack2<__nv_bfloat16>(uint32_t v) {
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v));
}

// ---- SiLU of the GroupNorm affine --------------------------------------------------------------------
//  silu(y) = h + h*tanh(h), h = y/2 with the 1/2 folded into the affine coefficients: FFMA + MUFU.TANH + FFMA
//  (tanh.approx.f32: max rel. error 2^-11, the same size as the fp16 rounding of the result).
//  (__expf/__fdividef cost ~12 instructions per element because of their range handling -- profile r1.)
__device__ __forceinline__ float tanh_approx(float x) {
    float y;
    asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ float silu_affine(float x, float a, float b) {
    const float y = fmaf(x, a, b);
    return fmaf(y, tanh_approx(y), y);  // (a, b) pre-halved by the caller
}

// GroupNorm apply + SiLU on 8 packed 16-bit channels; cf = (a, b) pairs of those channels (registers), pre-halved
template <typename T>
__device__ __forceinline__ void act8(const uint4& raw, const float2 (&cf)[8], float (&y)[8]) {
    const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float2 v = unpack2<T>(w[k]);
        y[2 * k] = silu_affine(v.x, cf[2 * k].x, cf[2 * k].y);
        y[2 * k + 1] = silu_affine(v.y, cf[2 * k + 1].x, cf[2 * k + 1].y);
    }
}

template <typename T>
__device__ __forceinline__ uint4 pack8(const float (&y)[8]) {
    return make_uint4(pack2<T>(y[0], y[1]), pack2<T>(y[2], y[3]), pack2<T>(y[4], y[5]), pack2<T>(y[6], y[7]));
}

}  // namespace dg
