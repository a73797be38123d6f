// Shared device helpers for the de-glaring UNet kernels (sm_100a).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <utility>

#include "deglare.h"

namespace dg {

// ---- storage traits: activations live in HBM as T, arithmetic is fp32 -----------------
template <typename T> struct Store;
template <> struct Store<float> {
    static __device__ __forceinline__ float to_f(float v) { return v; }
    static __device__ __forceinline__ float from_f(float v) { return v; }
};
template <> struct Store<__half> {
    static __device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
    static __device__ __forceinline__ __half from_f(float v) { return __float2half_rn(v); }
};
template <> struct Store<__nv_bfloat16> {
    static __device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
    static __device__ __forceinline__ __nv_bfloat16 from_f(float v) { return __float2bfloat16_rn(v); }
};

// load `cn` (<= 8) consecutive channels starting at p into v[0..8); 128-bit path when `vec`
template <typename T>
__device__ __forceinline__ void load8(const T* __restrict__ p, int cn, bool vec, float (&v)[8]) {
    if (vec) {
        if constexpr (sizeof(T) == 4) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(p));
            const float4 b = __ldg(reinterpret_cast<const float4*>(p) + 1);
            v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w;
            v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
        } else {
            const uint4 a = __ldg(reinterpret_cast<const uint4*>(p));
            const T* h = reinterpret_cast<const T*>(&a);
#pragma unroll
            for (int k = 0; k < 8; ++k) v[k] = Store<T>::to_f(h[k]);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = (k < cn) ? Store<T>::to_f(p[k]) : 0.f;
    }
}

template <typename T>
__device__ __forceinline__ void store8(T* __restrict__ p, int cn, bool vec, const float (&v)[8]) {
    if (vec) {
        if constexpr (sizeof(T) == 4) {
            reinterpret_cast<float4*>(p)[0] = make_float4(v[0], v[1], v[2], v[3]);
            reinterpret_cast<float4*>(p)[1] = make_float4(v[4], v[5], v[6], v[7]);
        } else {
            uint4 a;
            T* h = reinterpret_cast<T*>(&a);
#pragma unroll
            for (int k = 0; k < 8; ++k) h[k] = Store<T>::from_f(v[k]);
            *reinterpret_cast<uint4*>(p) = a;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (k < cn) p[k] = Store<T>::from_f(v[k]);
    }
}

// x * sigmoid(x) = x * rcp(1 + ex2(-x*log2e)) with the raw approx instructions (rel. err ~2^-22): FMUL, MUFU.EX2,
// FADD, MUFU.RCP, FMUL.  __expf/__fdividef add range handling worth ~7 more instructions per element, and the IEEE
// divide measured 4x slower still (tools/mma_bench.cu).  Saturates correctly: ex2(+big)=inf -> rcp(inf)=0.
__device__ __forceinline__ float silu_f(float x) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.f + e));
    return x * r;
}
__device__ __forceinline__ float sigmoid_f(float x) { return 1.f / (1.f + __expf(-x)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// GroupNorm coefficients of channel c of sample n from per-channel (sum, sumsq):
//   y = raw * a + b  with  a = rstd*gamma, b = beta - mean*a   (biased variance, eps inside sqrt)
__device__ __forceinline__ void gn_coef(const double* __restrict__ stats, const float* __restrict__ gamma,
                                        const float* __restrict__ beta, int n, int C, int groups, int c,
                                        double plane, float eps, float& a, float& b) {
    const int cpg = C / groups;
    const int g0 = (c / cpg) * cpg;
    double s1 = 0.0, s2 = 0.0;
    for (int k = 0; k < cpg; ++k) {
        s1 += stats[(size_t)(n * C + g0 + k) * 2];
        s2 += stats[(size_t)(n * C + g0 + k) * 2 + 1];
    }
    // Every conv CTA runs this serial chain before it can stage its tile (the other warps wait at the barrier), so the two
    // double divisions and the double rsqrt (~100 instructions) are replaced by float seeds + Newton steps in double:
    // 1/cnt and rsqrt(var + eps) to ~1e-16 relative, i.e. the same floats a and b after rounding.
    const double cnt = plane * cpg;
    double inv = (double)__frcp_rn((float)cnt);
    inv = inv * (2.0 - cnt * inv);
    inv = inv * (2.0 - cnt * inv);
    const double mean = s1 * inv;
    double var = fma(s2, inv, -mean * mean);
    if (var < 0.0) var = 0.0;
    const double x = var + (double)eps;
    double rstd = (double)rsqrtf((float)x);
    rstd = rstd * (1.5 - 0.5 * x * rstd * rstd);
    rstd = rstd * (1.5 - 0.5 * x * rstd * rstd);
    a = (float)(rstd * (double)gamma[c]);
    b = (float)((double)beta[c] - mean * rstd * (double)gamma[c]);
}

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------------------
// The forward is a chain of ~20 short kernels, each consuming its predecessor's output.  With the stream-serialisation
// attribute a kernel may start while the previous one drains its last wave; everything before pdl_wait() (weight
// cp.async, index setup, TMEM / barrier init) overlaps that tail, and pdl_wait() blocks until the predecessor's memory
// operations are complete and visible.  pdl_launch_dependents() lets the successor begin as soon as SMs free up.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

}  // namespace dg

// ---- host side ---------------------------------------------------------------------------
namespace dg {
void set_error(const char* fmt, ...);
bool pdl_enabled();
// <<<>>> replacement that adds the programmatic-stream-serialisation attribute when PDL is on
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}
void count_launch();
int check_launch(const char* what);
int conv3x3_generic_launch(const dg_conv3x3_args& a, cudaStream_t stream);
int conv3x3_tc_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled);
int conv_first_tc_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled);
int conv3x3_t5_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled);
int conv3x3_ring_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled);
int conv3x3_dec_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled);
int dec_composite_bytes(int cl, int cu, size_t* bytes);
int pack_dec_composite(const float* ct_w, const float* ct_b, const float* conv_w, void* out, int cl, int cu, int dtype, cudaStream_t st);
int convt_t5_launch(const dg_src& s, int dtype, int N, int H, int W, void* out, float eps, int path, cudaStream_t st, bool* handled);
int head_launch(const dg_head_args& a, cudaStream_t stream);
int convt_tc_launch(const dg_src& s, int dtype, int N, int H, int W, void* out, float eps, int path, cudaStream_t st,
                    bool* handled);
int se_scale_launch(const double* act_sum, double plane, const float* w1, const float* w2, int N, int C, int hidden,
                    float* scale, cudaStream_t st);
// activation backward of the producer conv fused into the data-gradient epilogue (dgrad_tc.cu)
struct DgradAct {
    const void* raw; const double* stats; const float* gamma; const float* beta; double* P;
    int groups, dtype; float eps;
};
int conv3x3_dgrad_tc_launch(const float* dR, const void* wtc_bf16, float* out, int N, int H, int W, int ck, int cn,
                            cudaStream_t st, bool* handled, const DgradAct* act = nullptr, const void* dR_bf16 = nullptr,
                            bool dry = false, float* out2 = nullptr);
int convt_dgrad_tc_launch(const float* dCat, int stride, const void* wtc_bf16, float* dLow, int N, int H, int W, int Cl, int Cu,
                          cudaStream_t st, bool* handled, const DgradAct* act = nullptr);
// data gradient of the wide layers on the tcgen05 kernel (conv3x3_t5.cu, T5_IDENT): dR fp32 (converted into scratch_bf16) or bf16
int conv3x3_dgrad_t5_launch(const float* dR, const void* dR_bf16, void* scratch_bf16, const void* wflip_tc_bf16, float* out, int N,
                            int H, int W, int ck, int cn, cudaStream_t st, bool* handled);
// ConvTranspose2d(2,2) data gradient of the wide layers on the tcgen05 kernel: gather of the up half per position (bf16 scratch of
// N*H*W*Cu elements) + one-tap T5_IDENT GEMM with K = 4 Cu, N = Cl
int convt_dgrad_t5_launch(const float* dCat, int stride, void* scratch_bf16, const void* w2_tc_bf16, float* dLow, int N, int H, int W,
                          int Cl, int Cu, cudaStream_t st, bool* handled);
int image_metrics_launch(const float* out, const float* tgt, int N, int H, int W, int clip01, double data_range, double* acc,
                         cudaStream_t st);
int first_wgrad_launch(const float* x, const float* dR, float* dW, int N, int H, int W, int CO, cudaStream_t st, bool* handled);
int first_dgrad_launch(const float* dR, const float* w, float* dx, int N, int H, int W, int CI, int C, cudaStream_t st);

int convt_wgrad_tc_launch(int dtype, const float* dCat, int stride, const void* raw_low, const double* stats, const float* gamma,
                          const float* beta, float* dWt, float* dBias, int N, int H, int W, int Cl, int Cu, int groups, float eps,
                          cudaStream_t st, bool* handled);
int conv3x3_wgrad_tc_launch(const dg_conv3x3_args& a, const float* dR, float* dW, int s_tap, int s_ci, int s_co,
                            cudaStream_t st, bool* handled, const void* dR_bf16 = nullptr, bool dry = false);
int conv3x3_wgrad_launch(const dg_conv3x3_args& a, const float* dR, float* dW, int s_tap, int s_ci, int s_co,
                         cudaStream_t stream);
int act_bwd_launch(int dtype, const void* raw, const double* stats, const float* gamma, const float* beta, const float* dA_a,
                   int stride_a, int off_a, const float* dA_b, int stride_b, int off_b, float* G, double* P, int N, int H,
                   int W, int C, int groups, float eps, cudaStream_t st);
int gn_bwd_apply_launch(int dtype, const void* raw, const double* stats, const float* gamma, const double* P, float* G,
                        float* dgamma, float* dbeta, int N, int H, int W, int C, int groups, float eps, cudaStream_t st, void* dRb = nullptr, bool* wrote_bf16 = nullptr);
int head_bwd_launch(int dtype, const void* raw, const double* stats, const float* gamma, const float* beta, const float* dOut,
                    const float* w, float* G, double* P, float* dW, float* dB, int N, int H, int W, int C, int OC, int groups,
                    float eps, cudaStream_t st, const float* l1_y = nullptr, const float* l1_target = nullptr,
                    const float* l1_scale = nullptr, float l1_inv_numel = 0.f);
int l1_sum_launch(const float* y, const float* t, size_t n, double* out, cudaStream_t st);
int convt_bwd_launch(int dtype, const float* dCat, int stride, const float* wt, const float* wt_t, const void* raw_low, const double* stats,
                     const float* gamma, const float* beta, float* dAlow, float* dWt, float* dBias, float* coefbuf, int N,
                     int H, int W, int Cl, int Cu, int groups, float eps, cudaStream_t st, const void* wtc_bf16 = nullptr, const DgradAct* act = nullptr, bool* act_fused = nullptr,
                     const void* w2_tc_bf16 = nullptr, void* scratch_bf16 = nullptr);
int adamw_launch(float* p, const float* g, float* m, float* v, size_t n, double* sumsq_scratch, float max_norm, float lr,
                 float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale, cudaStream_t st);
int band_stats_launch(const double* kstats, const void* t, int dtype, int W, int C, int a0, int a1, int b0, int b1, double* out,
                      cudaStream_t st);
int gn_affine_launch(const double* parts, int nparts, size_t stride, const float* gamma, const float* beta, int C, int groups, double plane,
                     float eps, float* coef, cudaStream_t st);
int adamw_dev_launch(float* p, const float* g, float* m, float* v, size_t n, double* sumsq_scratch, float max_norm, const float* lr_dev,
                     float beta1, float beta2, float eps, float weight_decay, int32_t* step_dev, float grad_scale, cudaStream_t st);
// OptimizedUNet-only backward pieces (opt_bwd.cu)
int grad_gather_launch(const float* a, int sa, int oa, const float* a_scale, const float* b, int sb, int ob, const float* u, int su,
                       int ou, const float* add, float* out, int N, int H, int W, int C, cudaStream_t st);
int scale_bwd_sum_launch(int dtype, const void* raw, const double* stats, const float* gamma, const float* beta, const float* d,
                         int sd, int od, double* out, int N, int H, int W, int C, int groups, float eps, cudaStream_t st);
int se_bwd_launch(const double* act_sum, double plane, const float* w1, const float* w2, const double* dscale, int N, int C,
                  int hidden, float* add, float* dw1, float* dw2, cudaStream_t st);
int tc_conv3x3_bytes(int cin, int cout, size_t* bytes);
int tc_convt_bytes(int cl, int cu, size_t* bytes);
int pack_conv3x3_tc(const float* w, void* out, int cin, int cout, int dtype, cudaStream_t st);
int pack_convt_tc(const float* w, void* out, int cl, int cu, int dtype, cudaStream_t st);
}  // namespace dg
