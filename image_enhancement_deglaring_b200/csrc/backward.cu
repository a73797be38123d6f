// Backward of the UNet blocks (autograd of src/model.py:92-131 as driven by optimized_train.py:210/226) and the
// fused optimizer tail (clip_grad_norm_ + AdamW, optimized_train.py:215-218,230-233,440-446).
//
// Gradient flow per conv i (raw output R_i, y_i = GN(R_i), A_i = SiLU(y_i)):
//   G_i  = dL/dy_i = (sum of dL/dA_i contributions) * silu'(y_i)            -> act_bwd_kernel (+ per-(n,c) sums
//          P1 = sum G, P2 = sum G*xhat, which are also dbeta / dgamma)
//   dR_i = rstd*(gamma*G_i - m1_g - xhat*m2_g),  m1_g = mean_g(gamma*G), m2_g = mean_g(gamma*G*xhat)
//                                                                             -> gn_bwd_apply_kernel (in place on G_i)
//   dW_i = corr(A_in, dR_i)                                                   -> conv3x3_generic_kernel<WGRAD>
//   dA_in = conv3x3(dR_i, flipped W_i)                                        -> the forward generic conv kernel itself
//   ConvTranspose2d(2,2): dA_low, dW_t, dbias                                 -> convt_bwd_data / convt_bwd_weight
//   head: dA_17 = dOut * w, dW_head, dbias                                    -> head_bwd_kernel
// All gradient tensors are fp32 NHWC; the saved raw activations are read in their storage type.
#include "common.cuh"

namespace dg {

namespace {
constexpr int BW_THREADS = 256;

__device__ __forceinline__ float silu_grad(float y) {
    const float s = 1.f / (1.f + __expf(-y));
    return s * (1.f + y * (1.f - s));
}

__device__ __forceinline__ void gn_mean_rstd(const double* __restrict__ stats, int n, int C, int groups, int c, double plane,
                                             float eps, float& mean, float& rstd) {
    const int cpg = C / groups;
    const int g0 = (c / cpg) * cpg;
    double s1 = 0.0, s2 = 0.0;
    for (int k = 0; k < cpg; ++k) {
        s1 += stats[(size_t)(n * C + g0 + k) * 2];
        s2 += stats[(size_t)(n * C + g0 + k) * 2 + 1];
    }
    // float-seeded Newton steps in double instead of double division / rsqrt (see gn_coef in common.cuh)
    const double cnt = plane * cpg;
    double inv = (double)__frcp_rn((float)cnt);
    inv = inv * (2.0 - cnt * inv);
    inv = inv * (2.0 - cnt * inv);
    const double m = s1 * inv;
    double var = fma(s2, inv, -m * m);
    if (var < 0.0) var = 0.0;
    const double x = var + (double)eps;
    double r = (double)rsqrtf((float)x);
    r = r * (1.5 - 0.5 * x * r * r);
    r = r * (1.5 - 0.5 * x * r * r);
    mean = (float)m;
    rstd = (float)r;
}

// (mean, rstd) from a group's (sum, sumsq): the arithmetic of gn_mean_rstd above
__device__ __forceinline__ void mean_rstd_of(double s1, double s2, double cnt, float eps, float& mean, float& rstd) {
    double inv = (double)__frcp_rn((float)cnt);
    inv = inv * (2.0 - cnt * inv);
    inv = inv * (2.0 - cnt * inv);
    const double m = s1 * inv;
    double var = fma(s2, inv, -m * m);
    if (var < 0.0) var = 0.0;
    const double x = var + (double)eps;
    double r = (double)rsqrtf((float)x);
    r = r * (1.5 - 0.5 * x * r * r);
    r = r * (1.5 - 0.5 * x * r * r);
    mean = (float)m;
    rstd = (float)r;
}

// Wide layers (C > 128, groups of 32..128 channels): the per-channel prologue above re-sums a whole group per channel -- 2 cpg
// double loads for each of C channels in EVERY CTA (524 k loads at C = 1024).  Here one warp sums one group (lanes stride over its
// channels, shuffle tree, fixed order), lane 0 leaves the K sums in gq[g][K]; callers derive the per-channel values from them.
// w(c, k) = k-th summand of channel c.  Must be called by the whole CTA; ends with a barrier.
template <int K, typename F>
__device__ __forceinline__ void group_sums(double* gq, int C, int groups, F w) {
    const int cpg = C / groups, lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    for (int g = warp; g < groups; g += nwarps) {
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.0;
        for (int c = g * cpg + lane; c < (g + 1) * cpg; c += 32) {
#pragma unroll
            for (int k = 0; k < K; ++k) acc[k] += w(c, k);
        }
#pragma unroll
        for (int k = 0; k < K; ++k) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
            if (lane == 0) gq[g * K + k] = acc[k];
        }
    }
    __syncthreads();
}

// ---- G = (dA_a + 0.25 * up2(dA_b)) * silu'(y);  P[n][c] += (sum G, sum G*xhat) -------------------------------------
struct ActBwdArgs {
    const void* raw; const double* stats; const float* gamma; const float* beta;
    const float* dA_a; int stride_a, off_a;   // same-resolution gradient [N,H,W,stride_a], channels off_a..off_a+C
    const float* dA_b; int stride_b, off_b;   // optional half-resolution gradient (AvgPool2d backward: /4, replicated)
    float* G; double* P;
    int N, H, W, C, groups; float eps;
};

template <typename T>
__global__ void __launch_bounds__(BW_THREADS) act_bwd_kernel(const ActBwdArgs p) {
    extern __shared__ double bsm[];
    const int C = p.C;
    double* psm = bsm;                                   // [C][2]
    float* coef = reinterpret_cast<float*>(psm + 2 * C);  // [C][4] mean, rstd, gamma, beta
    const int n = blockIdx.y;
    const int HW = p.H * p.W;
    for (int c = threadIdx.x; c < C; c += BW_THREADS) {
        float m, r;
        gn_mean_rstd(p.stats, n, C, p.groups, c, (double)HW, p.eps, m, r);
        coef[4 * c] = m; coef[4 * c + 1] = r; coef[4 * c + 2] = p.gamma[c]; coef[4 * c + 3] = p.beta[c];
        psm[2 * c] = 0.0; psm[2 * c + 1] = 0.0;
    }
    __syncthreads();
    const T* raw = reinterpret_cast<const T*>(p.raw);
    // thread -> fixed channel (needs BW_THREADS*gridDim.x to be a multiple of C when C < total threads: enforced by host)
    const size_t total = (size_t)HW * C;
    const size_t stride = (size_t)gridDim.x * BW_THREADS;
    double a1 = 0.0, a2 = 0.0;
    int cur_c = -1;
    for (size_t e = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; e < total; e += stride) {
        const int c = (int)(e % C);
        const int pix = (int)(e / C);
        if (c != cur_c) {
            if (cur_c >= 0) { atomicAdd(&psm[2 * cur_c], a1); atomicAdd(&psm[2 * cur_c + 1], a2); }
            cur_c = c; a1 = 0.0; a2 = 0.0;
        }
        const float r = Store<T>::to_f(raw[(size_t)n * total + e]);
        const float xh = (r - coef[4 * c]) * coef[4 * c + 1];
        const float y = xh * coef[4 * c + 2] + coef[4 * c + 3];
        float d = 0.f;
        if (p.dA_a) d = p.dA_a[((size_t)n * HW + pix) * p.stride_a + p.off_a + c];
        if (p.dA_b) {
            const int yy = pix / p.W, xx = pix % p.W;
            d += 0.25f * p.dA_b[((size_t)(n * (p.H / 2) + yy / 2) * (p.W / 2) + xx / 2) * p.stride_b + p.off_b + c];
        }
        const float g = d * silu_grad(y);
        p.G[(size_t)n * total + e] = g;
        a1 += (double)g;
        a2 += (double)(g * xh);
    }
    if (cur_c >= 0) { atomicAdd(&psm[2 * cur_c], a1); atomicAdd(&psm[2 * cur_c + 1], a2); }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * C; i += BW_THREADS) atomicAdd(p.P + (size_t)n * C * 2 + i, psm[i]);
}

// ---- dR = rstd*(gamma*G - m1 - xhat*m2) in place; block (0,0) also reduces dgamma/dbeta over the batch -----------------
struct GnBwdArgs {
    const void* raw; const double* stats; const float* gamma; const double* P;
    float* G;  // in: G, out: dR (unless dRb)
    void* dRb; // vector kernel only: write dR as bf16 [N,H,W,C] HERE instead of fp32 in place -- the tensor-core wgrad / dgrad round
               // it to bf16 anyway, so they read half the bytes and copy instead of converting (bit-identical results)
    float* dgamma; float* dbeta;   // either NULL = not computed (frozen)
    int N, H, W, C, groups; float eps;
};

template <typename T>
__global__ void __launch_bounds__(BW_THREADS) gn_bwd_apply_kernel(const GnBwdArgs p) {
    extern __shared__ float gsm[];  // [C][5] mean, rstd, gamma, m1, m2
    const int C = p.C, n = blockIdx.y, HW = p.H * p.W;
    const int cpg = C / p.groups;
    for (int c = threadIdx.x; c < C; c += BW_THREADS) {
        float m, r;
        gn_mean_rstd(p.stats, n, C, p.groups, c, (double)HW, p.eps, m, r);
        const int g0 = (c / cpg) * cpg;
        double m1 = 0.0, m2 = 0.0;
        for (int k = 0; k < cpg; ++k) {
            m1 += (double)p.gamma[g0 + k] * p.P[((size_t)n * C + g0 + k) * 2];
            m2 += (double)p.gamma[g0 + k] * p.P[((size_t)n * C + g0 + k) * 2 + 1];
        }
        const double cnt = (double)HW * cpg;
        gsm[5 * c] = m; gsm[5 * c + 1] = r; gsm[5 * c + 2] = p.gamma[c];
        gsm[5 * c + 3] = (float)(m1 / cnt); gsm[5 * c + 4] = (float)(m2 / cnt);
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && (p.dgamma != nullptr || p.dbeta != nullptr)) {
        for (int c = threadIdx.x; c < C; c += BW_THREADS) {
            double dg = 0.0, db = 0.0;
            for (int i = 0; i < p.N; ++i) {
                db += p.P[((size_t)i * C + c) * 2];
                dg += p.P[((size_t)i * C + c) * 2 + 1];
            }
            if (p.dgamma) atomicAdd(p.dgamma + c, (float)dg);   // accumulated: concurrent sub-batches (api.cu) each add their images' share
            if (p.dbeta) atomicAdd(p.dbeta + c, (float)db);
        }
    }
    __syncthreads();
    const T* raw = reinterpret_cast<const T*>(p.raw);
    const size_t total = (size_t)HW * C;
    for (size_t e = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * BW_THREADS) {
        const int c = (int)(e % C);
        const float r = Store<T>::to_f(raw[(size_t)n * total + e]);
        const float xh = (r - gsm[5 * c]) * gsm[5 * c + 1];
        const float g = p.G[(size_t)n * total + e];
        p.G[(size_t)n * total + e] = gsm[5 * c + 1] * (gsm[5 * c + 2] * g - gsm[5 * c + 3] - xh * gsm[5 * c + 4]);
    }
}


// ---- vectorised twins of the two element-wise kernels (C % 4 == 0, C/4 a power of two <= 32, aligned pointers) ----------
// The scalar kernels above pay two 64-bit divisions per element and a shared-memory double atomicAdd (a CAS loop) per
// channel switch: 7.1 + 3.4 ms of a 47 ms step (torch profiler, batch 32).  Here an item is (pixel, 4 channels): 128-bit
// accesses, 32-bit indexing, a thread stays on one channel chunk (its coefficients and partial sums live in registers), and
// the (sum G, sum G*xhat) partials are reduced by warp shuffles and per-warp slots in a fixed order (deterministic).
template <typename T>
__device__ __forceinline__ float4 load4_raw(const T* p) {
    if constexpr (sizeof(T) == 4) {
        return __ldg(reinterpret_cast<const float4*>(p));
    } else {
        const uint2 q = __ldg(reinterpret_cast<const uint2*>(p));
        const T* h = reinterpret_cast<const T*>(&q);
        return make_float4(Store<T>::to_f(h[0]), Store<T>::to_f(h[1]), Store<T>::to_f(h[2]), Store<T>::to_f(h[3]));
    }
}

template <typename T>
__global__ void __launch_bounds__(BW_THREADS) act_bwd_vec_kernel(const ActBwdArgs p) {
    extern __shared__ double bsm[];
    const int C = p.C, C4 = C >> 2;
    float* coef = reinterpret_cast<float*>(bsm);       // [C][4] mean, rstd, gamma, beta
    float* slot = coef + 4 * C;                        // [8 warps][C][2]
    const int n = blockIdx.y;
    const int HW = p.H * p.W;
    if (C4 > 32) {
        // wide layers: per-group sums by warps; a warp holds only 32 of the C4 chunks, so the slots start at zero
        double* gq = reinterpret_cast<double*>(slot + (BW_THREADS / 32) * C * 2);   // [groups][2]
        const double* st = p.stats + (size_t)n * C * 2;
        group_sums<2>(gq, C, p.groups, [&](int c, int k) { return st[2 * c + k]; });
        const int cpg = C / p.groups;
        for (int c = threadIdx.x; c < C; c += BW_THREADS) {
            float m, r;
            mean_rstd_of(gq[(c / cpg) * 2], gq[(c / cpg) * 2 + 1], (double)HW * cpg, p.eps, m, r);
            coef[4 * c] = m; coef[4 * c + 1] = r; coef[4 * c + 2] = p.gamma[c]; coef[4 * c + 3] = p.beta[c];
        }
        for (int i = threadIdx.x; i < (BW_THREADS / 32) * C * 2; i += BW_THREADS) slot[i] = 0.f;
    } else {
        for (int c = threadIdx.x; c < C; c += BW_THREADS) {
            float m, r;
            gn_mean_rstd(p.stats, n, C, p.groups, c, (double)HW, p.eps, m, r);
            coef[4 * c] = m; coef[4 * c + 1] = r; coef[4 * c + 2] = p.gamma[c]; coef[4 * c + 3] = p.beta[c];
        }
    }
    __syncthreads();
    const int items = HW * C4;
    const int stride = gridDim.x * BW_THREADS;         // multiple of C4: the channel chunk of a thread is fixed
    const int e0 = blockIdx.x * BW_THREADS + threadIdx.x;
    const int c4 = e0 & (C4 - 1);
    float cm[4], cr[4], cg[4], cb[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        cm[k] = coef[4 * (4 * c4 + k)]; cr[k] = coef[4 * (4 * c4 + k) + 1];
        cg[k] = coef[4 * (4 * c4 + k) + 2]; cb[k] = coef[4 * (4 * c4 + k) + 3];
    }
    float a1[4] = {0.f, 0.f, 0.f, 0.f}, a2[4] = {0.f, 0.f, 0.f, 0.f};
    const T* raw = reinterpret_cast<const T*>(p.raw) + (size_t)n * HW * C;
    float* G = p.G + (size_t)n * HW * C;
    const float* dA = p.dA_a ? p.dA_a + (size_t)n * HW * p.stride_a + p.off_a + 4 * c4 : nullptr;
    const float* dB = p.dA_b ? p.dA_b + (size_t)n * (HW / 4) * p.stride_b + p.off_b + 4 * c4 : nullptr;
    const int Wh = p.W >> 1;
    for (int e = e0; e < items; e += stride) {
        const int pix = e / C4;  // C4 is a power of two: a shift after inlining? no -- runtime; one 32-bit division
        const float4 r4 = load4_raw<T>(raw + (size_t)pix * C + 4 * c4);
        float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
        if (dA) d = __ldg(reinterpret_cast<const float4*>(dA + (size_t)pix * p.stride_a));
        if (dB) {
            const int yy = pix / p.W, xx = pix - yy * p.W;
            const float4 h = __ldg(reinterpret_cast<const float4*>(dB + (size_t)((yy >> 1) * Wh + (xx >> 1)) * p.stride_b));
            d.x = fmaf(0.25f, h.x, d.x); d.y = fmaf(0.25f, h.y, d.y); d.z = fmaf(0.25f, h.z, d.z); d.w = fmaf(0.25f, h.w, d.w);
        }
        const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
        const float dd[4] = {d.x, d.y, d.z, d.w};
        float g[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float xh = (rr[k] - cm[k]) * cr[k];
            const float y = xh * cg[k] + cb[k];
            g[k] = dd[k] * silu_grad(y);
            a1[k] += g[k];
            a2[k] = fmaf(g[k], xh, a2[k]);
        }
        *reinterpret_cast<float4*>(G + (size_t)pix * C + 4 * c4) = make_float4(g[0], g[1], g[2], g[3]);
    }
    // lanes with equal (lane mod C4) hold the same channels
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        for (int o = C4; o < 32; o <<= 1) {
            a1[k] += __shfl_xor_sync(0xffffffffu, a1[k], o);
            a2[k] += __shfl_xor_sync(0xffffffffu, a2[k], o);
        }
    }
    // chunks owned by this warp: (warp*32 + lane) mod C4 for lane < min(C4, 32); a warp covers min(C4, 32) chunks
    if (lane < C4) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            slot[(warp * C + 4 * c4 + k) * 2] = a1[k];
            slot[(warp * C + 4 * c4 + k) * 2 + 1] = a2[k];
        }
    }
    __syncthreads();
    // C4 <= 32: every warp holds every chunk (32 % C4 == 0); C4 > 32: the other warps' slots are zero -> sum the 8 warp slots in a fixed order
    for (int i = threadIdx.x; i < 2 * C; i += BW_THREADS) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < BW_THREADS / 32; ++w) t += (double)slot[w * C * 2 + i];
        atomicAdd(p.P + (size_t)n * C * 2 + i, t);
    }
}

template <typename T>
__global__ void __launch_bounds__(BW_THREADS) gn_bwd_apply_vec_kernel(const GnBwdArgs p) {
    extern __shared__ float gsm[];  // [C][5] mean, rstd, gamma, m1, m2
    const int C = p.C, C4 = C >> 2, n = blockIdx.y, HW = p.H * p.W;
    const int cpg = C / p.groups;
    if (C4 > 32) {   // wide layers: the four per-group sums once per CTA (see group_sums)
        double* gq = reinterpret_cast<double*>(gsm + 5 * C + (C & 1));   // [groups][4], 8-byte aligned behind the 5 C floats
        const double* st = p.stats + (size_t)n * C * 2;
        const double* P = p.P + (size_t)n * C * 2;
        group_sums<4>(gq, C, p.groups, [&](int c, int k) { return k < 2 ? st[2 * c + k] : (double)p.gamma[c] * P[2 * c + (k - 2)]; });
        const double cnt = (double)HW * cpg;
        for (int c = threadIdx.x; c < C; c += BW_THREADS) {
            const double* q = gq + (c / cpg) * 4;
            float m, r;
            mean_rstd_of(q[0], q[1], cnt, p.eps, m, r);
            gsm[5 * c] = m; gsm[5 * c + 1] = r; gsm[5 * c + 2] = p.gamma[c];
            gsm[5 * c + 3] = (float)(q[2] / cnt); gsm[5 * c + 4] = (float)(q[3] / cnt);
        }
    } else
    for (int c = threadIdx.x; c < C; c += BW_THREADS) {
        float m, r;
        gn_mean_rstd(p.stats, n, C, p.groups, c, (double)HW, p.eps, m, r);
        const int g0 = (c / cpg) * cpg;
        double m1 = 0.0, m2 = 0.0;
        for (int k = 0; k < cpg; ++k) {
            m1 += (double)p.gamma[g0 + k] * p.P[((size_t)n * C + g0 + k) * 2];
            m2 += (double)p.gamma[g0 + k] * p.P[((size_t)n * C + g0 + k) * 2 + 1];
        }
        const double cnt = (double)HW * cpg;
        gsm[5 * c] = m; gsm[5 * c + 1] = r; gsm[5 * c + 2] = p.gamma[c];
        gsm[5 * c + 3] = (float)(m1 / cnt); gsm[5 * c + 4] = (float)(m2 / cnt);
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && (p.dgamma != nullptr || p.dbeta != nullptr)) {
        for (int c = threadIdx.x; c < C; c += BW_THREADS) {
            double dg = 0.0, db = 0.0;
            for (int i = 0; i < p.N; ++i) {
                db += p.P[((size_t)i * C + c) * 2];
                dg += p.P[((size_t)i * C + c) * 2 + 1];
            }
            if (p.dgamma) atomicAdd(p.dgamma + c, (float)dg);   // accumulated: concurrent sub-batches (api.cu) each add their images' share
            if (p.dbeta) atomicAdd(p.dbeta + c, (float)db);
        }
    }
    __syncthreads();
    const int items = HW * C4;
    const int stride = gridDim.x * BW_THREADS;
    const int e0 = blockIdx.x * BW_THREADS + threadIdx.x;
    const int c4 = e0 & (C4 - 1);
    float cm[4], cr[4], cg[4], c1[4], c2[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float* q = gsm + 5 * (4 * c4 + k);
        cm[k] = q[0]; cr[k] = q[1]; cg[k] = q[2]; c1[k] = q[3]; c2[k] = q[4];
    }
    const T* raw = reinterpret_cast<const T*>(p.raw) + (size_t)n * HW * C + 4 * c4;
    float* G = p.G + (size_t)n * HW * C + 4 * c4;
    for (int e = e0; e < items; e += stride) {
        const int pix = e / C4;
        const float4 r4 = load4_raw<T>(raw + (size_t)pix * C);
        const float4 g4 = *reinterpret_cast<const float4*>(G + (size_t)pix * C);
        const float rr[4] = {r4.x, r4.y, r4.z, r4.w};
        const float gg[4] = {g4.x, g4.y, g4.z, g4.w};
        float o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float xh = (rr[k] - cm[k]) * cr[k];
            o[k] = cr[k] * (cg[k] * gg[k] - c1[k] - xh * c2[k]);
        }
        if (p.dRb != nullptr) {
            __nv_bfloat162 lo = __floats2bfloat162_rn(o[0], o[1]), hi = __floats2bfloat162_rn(o[2], o[3]);
            *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.dRb) + ((size_t)n * HW + pix) * C + 4 * c4) =
                make_uint2(*reinterpret_cast<uint32_t*>(&lo), *reinterpret_cast<uint32_t*>(&hi));
        } else {
            *reinterpret_cast<float4*>(G + (size_t)pix * C) = make_float4(o[0], o[1], o[2], o[3]);
        }
    }
}

// ---- head backward: dA = dOut * w -> G_last, P_last; dW_head, dbias -----------------------------------------------------
struct HeadBwdArgs {
    const void* raw; const double* stats; const float* gamma; const float* beta;
    const float* dOut;    // [N,OC,H,W]
    const float* w;       // [OC][C]
    float* G; double* P;  // [N,H,W,C], [N,C,2]
    float* dW; float* dB; // [OC][C], [OC] accumulated atomically (zero on entry); either NULL = not computed (frozen)
    int N, H, W, C, OC, groups; float eps;
    // nn.L1Loss backward fused (optimized_train.py:439,210/226): when `target` is set, dOut is not read at all -- the seed
    // sign(y - target) * (*scale) * inv_numel is generated here from the forward output y (sign(0) = 0, as torch)
    const float* y; const float* target; const float* scale; float inv_numel;
};

__device__ __forceinline__ float l1_seed(float y, float t, float s) { return y > t ? s : (y < t ? -s : 0.f); }

template <typename T>
__global__ void __launch_bounds__(BW_THREADS) head_bwd_kernel(const HeadBwdArgs p) {
    extern __shared__ double hbs[];
    const int C = p.C, OC = p.OC, n = blockIdx.y, HW = p.H * p.W;
    double* psm = hbs;                                        // [C][2]
    double* wacc = psm + 2 * C;                               // [OC][C] + [OC]
    float* coef = reinterpret_cast<float*>(wacc + OC * C + OC);  // [C][4]
    float* wsm = coef + 4 * C;                                // [OC][C]
    for (int c = threadIdx.x; c < C; c += BW_THREADS) {
        float m, r;
        gn_mean_rstd(p.stats, n, C, p.groups, c, (double)HW, p.eps, m, r);
        coef[4 * c] = m; coef[4 * c + 1] = r; coef[4 * c + 2] = p.gamma[c]; coef[4 * c + 3] = p.beta[c];
        psm[2 * c] = 0.0; psm[2 * c + 1] = 0.0;
    }
    for (int i = threadIdx.x; i < OC * C + OC; i += BW_THREADS) wacc[i] = 0.0;
    for (int i = threadIdx.x; i < OC * C; i += BW_THREADS) wsm[i] = p.w[i];
    __syncthreads();
    const T* raw = reinterpret_cast<const T*>(p.raw);
    const int lane = threadIdx.x & 31;
    // whole warps iterate together (inactive lanes contribute zeros) so the per-channel sums reduce with shuffles
    const int npix_round = (HW + 31) & ~31;
    for (int pix = blockIdx.x * BW_THREADS + threadIdx.x; pix < npix_round; pix += gridDim.x * BW_THREADS) {
        const bool live = pix < HW;
        float dO[4] = {0.f, 0.f, 0.f, 0.f};
        for (int j = 0; j < OC; ++j) {
            if (live) {
                const size_t oi = ((size_t)n * OC + j) * HW + pix;
                dO[j] = p.target ? l1_seed(p.y[oi], p.target[oi], (p.scale ? __ldg(p.scale) : 1.f) * p.inv_numel) : p.dOut[oi];
            }
            const float t = warp_sum(dO[j]);
            if (lane == 0) atomicAdd(&wacc[OC * C + j], (double)t);
        }
        for (int c = 0; c < C; ++c) {
            float g = 0.f, gx = 0.f, a = 0.f;
            if (live) {
                const float r = Store<T>::to_f(raw[((size_t)n * HW + pix) * C + c]);
                const float xh = (r - coef[4 * c]) * coef[4 * c + 1];
                const float y = xh * coef[4 * c + 2] + coef[4 * c + 3];
                a = silu_f(y);
                float d = 0.f;
                for (int j = 0; j < OC; ++j) d = fmaf(dO[j], wsm[j * C + c], d);
                g = d * silu_grad(y);
                gx = g * xh;
                p.G[((size_t)n * HW + pix) * C + c] = g;
            }
            const float t1 = warp_sum(g), t2 = warp_sum(gx);
            if (lane == 0) { atomicAdd(&psm[2 * c], (double)t1); atomicAdd(&psm[2 * c + 1], (double)t2); }
            for (int j = 0; j < OC; ++j) {
                const float t3 = warp_sum(dO[j] * a);
                if (lane == 0) atomicAdd(&wacc[j * C + c], (double)t3);
            }
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * C; i += BW_THREADS) atomicAdd(p.P + (size_t)n * C * 2 + i, psm[i]);
    if (p.dW) for (int i = threadIdx.x; i < OC * C; i += BW_THREADS) atomicAdd(p.dW + i, (float)wacc[i]);
    if (p.dB) for (int i = threadIdx.x; i < OC; i += BW_THREADS) atomicAdd(p.dB + i, (float)wacc[OC * C + i]);
}

// ---- ConvTranspose2d(k=2,s=2) backward ---------------------------------------------------------------------------------
//   up[n, 2i+a, 2j+b, co] = bias[co] + sum_ci Alow[n,i,j,ci] * Wt[ab][ci][co]       (src/model.py:47-53)
struct ConvtBwdArgs {
    const float* dCat; int stride;      // gradient of the concat [N,H,W,stride]; the up half is channels 0..Cu
    const float* wt;                    // [2][2][Cl][Cu]
    const float* wt_t;                  // [2][2][Cu][Cl] (transposed copy: the data-gradient kernel reads it coalesced over ci)
    const void* raw_low; const double* stats; const float* gamma; const float* beta;  // low-res producer (for A_low)
    float* dAlow;                       // [N,H/2,W/2,Cl]
    float* dWt; float* dBias;           // accumulated atomically
    float* coefbuf;                     // scratch [N][Cl][2] (mean, rstd) of the low-res producer
    int N, H, W, Cl, Cu, groups; float eps;
};

__global__ void __launch_bounds__(BW_THREADS) convt_bwd_data_kernel(const ConvtBwdArgs p) {
    // one thread per (low pixel, ci): dAlow = sum_{ab,co} dUp[2i+a, 2j+b, co] * Wt[ab][ci][co]
    const int Hl = p.H / 2, Wl = p.W / 2;
    const size_t total = (size_t)p.N * Hl * Wl * p.Cl;
    for (size_t e = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * BW_THREADS) {
        const int ci = (int)(e % p.Cl);
        const size_t lp = e / p.Cl;
        const int j = (int)(lp % Wl);
        const int i = (int)((lp / Wl) % Hl);
        const int n = (int)(lp / ((size_t)Wl * Hl));
        float acc = 0.f;
        for (int ab = 0; ab < 4; ++ab) {
            // all ci-threads of a pixel read the same gradient (broadcast); the weights are coalesced over ci
            const float4* d = reinterpret_cast<const float4*>(p.dCat + ((size_t)(n * p.H + 2 * i + (ab >> 1)) * p.W + 2 * j + (ab & 1)) * p.stride);
            const float* w = p.wt_t + (size_t)ab * p.Cu * p.Cl + ci;
            for (int co = 0; co < p.Cu; co += 4) {
                const float4 g = __ldg(d + (co >> 2));
                acc = fmaf(g.x, __ldg(w + (size_t)co * p.Cl), acc);
                acc = fmaf(g.y, __ldg(w + (size_t)(co + 1) * p.Cl), acc);
                acc = fmaf(g.z, __ldg(w + (size_t)(co + 2) * p.Cl), acc);
                acc = fmaf(g.w, __ldg(w + (size_t)(co + 3) * p.Cl), acc);
            }
        }
        p.dAlow[e] = acc;
    }
}

__global__ void gn_mean_rstd_kernel(const double* stats, float* out, int C, int groups, double plane, float eps) {
    const int n = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float m, r;
        gn_mean_rstd(stats, n, C, groups, c, plane, eps, m, r);
        out[((size_t)n * C + c) * 2] = m;
        out[((size_t)n * C + c) * 2 + 1] = r;
    }
}

template <typename T>
__global__ void __launch_bounds__(BW_THREADS) convt_bwd_weight_kernel(const ConvtBwdArgs p, int slab) {
    // grid.x: groups of 256 consecutive (ab, ci, co) combos (co fastest); grid.y: strided slabs of low pixels.  A CTA stages
    // only the activated input channels [ci_lo, ci_hi] and the gradient positions [ab_lo, ab_hi] its combos touch.
    extern __shared__ float csm[];
    const int Cl = p.Cl, Cu = p.Cu;
    const int Hl = p.H / 2, Wl = p.W / 2;
    const int npix = p.N * Hl * Wl;
    const int ncombo = 4 * Cl * Cu;
    const int c_first = blockIdx.x * BW_THREADS;
    const int c_last = min(c_first + BW_THREADS, ncombo) - 1;
    const int ab_lo = c_first / (Cl * Cu), ab_hi = c_last / (Cl * Cu);
    int ci_lo = (c_first / Cu) % Cl, ci_hi = (c_last / Cu) % Cl;
    if (ab_hi > ab_lo) { ci_lo = 0; ci_hi = Cl - 1; }
    const int nci = ci_hi - ci_lo + 1, nab = ab_hi - ab_lo + 1;
    float* alow = csm;                    // [slab][nci]
    float* dup = alow + slab * nci;       // [slab][nab][Cu]
    const int combo = c_first + threadIdx.x;
    const int co = combo % Cu, ci = (combo / Cu) % Cl, ab = combo / (Cu * Cl);
    const T* raw = reinterpret_cast<const T*>(p.raw_low);
    float acc = 0.f, bacc = 0.f;
    const bool do_bias = blockIdx.x == 0 && threadIdx.x < 4 * Cu && p.dBias != nullptr;  // needs all four positions: see host
    for (int base = blockIdx.y * slab; base < npix; base += gridDim.y * slab) {
        __syncthreads();
        for (int idx = threadIdx.x; idx < slab * nci; idx += BW_THREADS) {
            const int c = ci_lo + idx % nci, lp = base + idx / nci;
            float v = 0.f;
            if (lp < npix) {
                const int n = lp / (Hl * Wl);
                const float m = p.coefbuf[((size_t)n * Cl + c) * 2], r = p.coefbuf[((size_t)n * Cl + c) * 2 + 1];
                const float y = (Store<T>::to_f(raw[(size_t)lp * Cl + c]) - m) * r * p.gamma[c] + p.beta[c];
                v = silu_f(y);
            }
            alow[idx] = v;
        }
        for (int idx = threadIdx.x; idx < slab * nab * Cu; idx += BW_THREADS) {
            const int c = idx % Cu, q = ab_lo + (idx / Cu) % nab, lp = base + idx / (nab * Cu);
            float v = 0.f;
            if (lp < npix) {
                const int j = lp % Wl, i = (lp / Wl) % Hl, n = lp / (Hl * Wl);
                v = p.dCat[((size_t)(n * p.H + 2 * i + (q >> 1)) * p.W + 2 * j + (q & 1)) * p.stride + c];
            }
            dup[idx] = v;
        }
        __syncthreads();
        if (combo < ncombo) {
            const float* ap = alow + (ci - ci_lo);
            const float* dp = dup + (ab - ab_lo) * Cu + co;
#pragma unroll 4
            for (int s = 0; s < slab; ++s) acc = fmaf(ap[s * nci], dp[s * nab * Cu], acc);
        }
        if (do_bias) {
            const float* dp = dup + threadIdx.x;   // block 0 covers ab 0..nab-1; (ab', co') = thread index
            if ((int)threadIdx.x < nab * Cu)
                for (int s = 0; s < slab; ++s) bacc += dp[s * nab * Cu];
        }
    }
    if (combo < ncombo) atomicAdd(p.dWt + ((size_t)ci * Cu + co) * 4 + ab, acc);  // parameter layout [Cl][Cu][2][2]
    if (do_bias && (int)threadIdx.x < nab * Cu) atomicAdd(p.dBias + threadIdx.x % Cu, bacc);
}

// dbias[co] = sum over every up-sampled pixel of the gradient (separate, trivially parallel reduction)
__global__ void __launch_bounds__(BW_THREADS) convt_bwd_bias_kernel(const ConvtBwdArgs p) {
    extern __shared__ float bsum[];  // [Cu]
    for (int c = threadIdx.x; c < p.Cu; c += BW_THREADS) bsum[c] = 0.f;
    __syncthreads();
    const size_t total = (size_t)p.N * p.H * p.W * p.Cu;
    const size_t stride = (size_t)gridDim.x * BW_THREADS;   // multiple of Cu for power-of-two Cu <= 256
    float acc = 0.f;
    int cur = -1;
    for (size_t e = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; e < total; e += stride) {
        const int c = (int)(e % p.Cu);
        if (c != cur) {
            if (cur >= 0) atomicAdd(&bsum[cur], acc);
            cur = c; acc = 0.f;
        }
        acc += p.dCat[(e / p.Cu) * p.stride + c];
    }
    if (cur >= 0) atomicAdd(&bsum[cur], acc);
    __syncthreads();
    for (int c = threadIdx.x; c < p.Cu; c += BW_THREADS) atomicAdd(p.dBias + c, bsum[c]);
}

// ---- optimizer tail over the flat parameter / gradient buffers -------------------------------------------------------------
__global__ void __launch_bounds__(BW_THREADS) sumsq_kernel(const float* __restrict__ g, size_t n, double* out) {
    double acc = 0.0;
    for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < n; i += (size_t)gridDim.x * BW_THREADS)
        acc += (double)g[i] * (double)g[i];
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    __shared__ double red[BW_THREADS / 32];
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < BW_THREADS / 32; ++i) t += red[i];
        atomicAdd(out, t);
    }
}

struct AdamwArgs {
    float* p; const float* g; float* m; float* v; size_t n;
    const double* sumsq;  // global grad sum of squares (device), for clip_grad_norm_
    float max_norm, lr, beta1, beta2, eps, weight_decay, bc1, bc2_sqrt, grad_scale;
};

__global__ void __launch_bounds__(BW_THREADS) adamw_kernel(const AdamwArgs a) {
    // torch.nn.utils.clip_grad_norm_: coef = min(1, max_norm / (total_norm + 1e-6)); torch.optim.AdamW (decoupled decay)
    float coef = a.grad_scale;
    if (a.max_norm > 0.f) {
        const float total = (float)sqrt(*a.sumsq) * a.grad_scale;
        coef *= fminf(1.f, a.max_norm / (total + 1e-6f));
    }
    for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < a.n; i += (size_t)gridDim.x * BW_THREADS) {
        const float g = a.g[i] * coef;
        float p = a.p[i] * (1.f - a.lr * a.weight_decay);
        const float m = a.beta1 * a.m[i] + (1.f - a.beta1) * g;
        const float v = a.beta2 * a.v[i] + (1.f - a.beta2) * g * g;
        a.m[i] = m;
        a.v[i] = v;
        const float denom = sqrtf(v) / a.bc2_sqrt + a.eps;
        a.p[i] = p - (a.lr / a.bc1) * (m / denom);
    }
}

// CUDA-graph-capturable flavour: the step count and the learning rate live in device memory, so a captured training step can be
// replayed with nothing baked in -- `step_bump_kernel` increments the counter, the update kernel derives the bias corrections.
__global__ void step_bump_kernel(int32_t* step) { *step += 1; }

struct AdamwDevArgs {
    float* p; const float* g; float* m; float* v; size_t n;
    const double* sumsq; const int32_t* step; const float* lr;
    float max_norm, beta1, beta2, eps, weight_decay, grad_scale;
};

__global__ void __launch_bounds__(BW_THREADS) adamw_dev_kernel(const AdamwDevArgs a) {
    float coef = a.grad_scale;
    if (a.max_norm > 0.f) {
        const float total = (float)sqrt(*a.sumsq) * a.grad_scale;
        coef *= fminf(1.f, a.max_norm / (total + 1e-6f));
    }
    const int step = *a.step;
    const float lr = *a.lr;
    const float bc1 = (float)(1.0 - pow((double)a.beta1, (double)step));         // same double-precision corrections as the host flavour
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)a.beta2, (double)step));
    for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < a.n; i += (size_t)gridDim.x * BW_THREADS) {
        const float g = a.g[i] * coef;
        float p = a.p[i] * (1.f - lr * a.weight_decay);
        const float m = a.beta1 * a.m[i] + (1.f - a.beta1) * g;
        const float v = a.beta2 * a.v[i] + (1.f - a.beta2) * g * g;
        a.m[i] = m;
        a.v[i] = v;
        const float denom = sqrtf(v) / bc2_sqrt + a.eps;
        a.p[i] = p - (lr / bc1) * (m / denom);
    }
}

inline int ew_blocks(size_t elems, int C) {
    // element-wise kernels keep a thread on one channel across its stride loop only if the stride is a multiple of C
    size_t b = (elems + BW_THREADS - 1) / BW_THREADS;
    if (b > 2048) b = 2048;
    if (b < 1) b = 1;
    (void)C;
    return (int)b;
}

// ---- head backward, common case (one output channel, C = 8 or 16): a thread owns whole pixels, keeps the 3C + 1 partial sums
// (sum G, sum G*xhat, dW_head, dbias) in registers over its pixels and reduces them once (the general kernel above does three
// warp reductions per channel per pixel round: 0.45 ms at batch 32 for 0.44 GB of traffic) --------------------------------------
template <typename T, int C>
__global__ void __launch_bounds__(BW_THREADS) head_bwd_fast_kernel(const HeadBwdArgs p) {
    __shared__ float coef[C][4];
    __shared__ float wsm[C];
    __shared__ float slot[BW_THREADS / 32][3 * C + 1];
    const int n = blockIdx.y, HW = p.H * p.W;
    if (threadIdx.x < C) {
        float m, r;
        gn_mean_rstd(p.stats, n, C, p.groups, threadIdx.x, (double)HW, p.eps, m, r);
        coef[threadIdx.x][0] = m; coef[threadIdx.x][1] = r; coef[threadIdx.x][2] = p.gamma[threadIdx.x];
        coef[threadIdx.x][3] = p.beta[threadIdx.x];
        wsm[threadIdx.x] = p.w[threadIdx.x];
    }
    __syncthreads();
    float cm[C], cr[C], cg[C], cb[C], w[C];
#pragma unroll
    for (int c = 0; c < C; ++c) { cm[c] = coef[c][0]; cr[c] = coef[c][1]; cg[c] = coef[c][2]; cb[c] = coef[c][3]; w[c] = wsm[c]; }
    float p1[C], p2[C], dw[C], db = 0.f;
#pragma unroll
    for (int c = 0; c < C; ++c) p1[c] = p2[c] = dw[c] = 0.f;
    const T* raw = reinterpret_cast<const T*>(p.raw) + (size_t)n * HW * C;
    float* G = p.G + (size_t)n * HW * C;
    const float* dOut = p.dOut + (size_t)n * HW;
    const float* yo = p.y + (size_t)n * HW;
    const float* tg = p.target + (size_t)n * HW;
    const float seed = p.target ? (p.scale ? __ldg(p.scale) : 1.f) * p.inv_numel : 0.f;
    for (int pix = blockIdx.x * BW_THREADS + threadIdx.x; pix < HW; pix += gridDim.x * BW_THREADS) {
        const float d = p.target ? l1_seed(__ldg(yo + pix), __ldg(tg + pix), seed) : __ldg(dOut + pix);
        db += d;
        float r[C];
#pragma unroll
        for (int c4 = 0; c4 < C / 4; ++c4) {
            const float4 v = load4_raw<T>(raw + (size_t)pix * C + 4 * c4);
            r[4 * c4] = v.x; r[4 * c4 + 1] = v.y; r[4 * c4 + 2] = v.z; r[4 * c4 + 3] = v.w;
        }
        float g[C];
#pragma unroll
        for (int c = 0; c < C; ++c) {
            const float xh = (r[c] - cm[c]) * cr[c];
            const float y = xh * cg[c] + cb[c];
            dw[c] = fmaf(d, silu_f(y), dw[c]);
            g[c] = d * w[c] * silu_grad(y);
            p1[c] += g[c];
            p2[c] = fmaf(g[c], xh, p2[c]);
        }
#pragma unroll
        for (int c4 = 0; c4 < C / 4; ++c4)
            *reinterpret_cast<float4*>(G + (size_t)pix * C + 4 * c4) = make_float4(g[4 * c4], g[4 * c4 + 1], g[4 * c4 + 2], g[4 * c4 + 3]);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const float a = warp_sum(p1[c]), b = warp_sum(p2[c]), e = warp_sum(dw[c]);
        if (lane == 0) { slot[warp][c] = a; slot[warp][C + c] = b; slot[warp][2 * C + c] = e; }
    }
    db = warp_sum(db);
    if (lane == 0) slot[warp][3 * C] = db;
    __syncthreads();
    for (int i = threadIdx.x; i < 3 * C + 1; i += BW_THREADS) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < BW_THREADS / 32; ++k) t += (double)slot[k][i];
        if (i < C) atomicAdd(p.P + ((size_t)n * C + i) * 2, t);
        else if (i < 2 * C) atomicAdd(p.P + ((size_t)n * C + (i - C)) * 2 + 1, t);
        else if (i < 3 * C) { if (p.dW) atomicAdd(p.dW + (i - 2 * C), (float)t); }
        else if (p.dB) atomicAdd(p.dB, (float)t);
    }
}

// ---- weight gradient of the first conv (1 -> CO channels, src/model.py:93 of enc1): 9 CO sums over every pixel --------------
// dW[co][0][ky][kx] = sum x[n, y+ky-1, x+kx-1] * dR[n, y, x, co].  Pure streaming (x fp32 + dR fp32 read once): the generic
// WGRAD mode took 0.56 ms at batch 32 for what is 0.3 GB of traffic.  Persistent CTAs, the haloed x tile in shared memory,
// 9 x CO partial sums per thread in registers, one shuffle / shared / atomic reduction per CTA at the end.
template <int CO>
__global__ void __launch_bounds__(BW_THREADS) first_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dR,
                                                                  float* __restrict__ dW, int N, int H, int W, int tiles_x, int tiles_y) {
    constexpr int TH = 16, TW = 64, PW = TW + 2;
    __shared__ float xs[(TH + 2) * PW];
    __shared__ float red[BW_THREADS / 32][9 * CO];
    float acc[9][CO];
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int c = 0; c < CO; ++c) acc[t][c] = 0.f;
    const int tiles_per_img = tiles_x * tiles_y, ntiles = tiles_per_img * N;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int n = tile / tiles_per_img, tr = tile - n * tiles_per_img;
        const int y0 = (tr / tiles_x) * TH, x0 = (tr % tiles_x) * TW;
        __syncthreads();
        for (int i = threadIdx.x; i < (TH + 2) * PW; i += BW_THREADS) {
            const int r = i / PW, c = i - r * PW;
            const int gy = y0 + r - 1, gx = x0 + c - 1;
            xs[i] = ((unsigned)gy < (unsigned)H && (unsigned)gx < (unsigned)W) ? __ldg(x + ((size_t)n * H + gy) * W + gx) : 0.f;
        }
        __syncthreads();
#pragma unroll 2
        for (int pix = threadIdx.x; pix < TH * TW; pix += BW_THREADS) {
            const int r = pix / TW, c = pix - r * TW;
            const int gy = y0 + r, gx = x0 + c;
            if (gy >= H || gx >= W) continue;
            float d[CO];
            const float4* q = reinterpret_cast<const float4*>(dR + (((size_t)n * H + gy) * W + gx) * CO);
#pragma unroll
            for (int k = 0; k < CO / 4; ++k) {
                const float4 v = __ldg(q + k);
                d[4 * k] = v.x; d[4 * k + 1] = v.y; d[4 * k + 2] = v.z; d[4 * k + 3] = v.w;
            }
#pragma unroll
            for (int t = 0; t < 9; ++t) {
                const float xv = xs[(r + t / 3) * PW + c + t % 3];
#pragma unroll
                for (int k = 0; k < CO; ++k) acc[t][k] = fmaf(xv, d[k], acc[t][k]);
            }
        }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int k = 0; k < CO; ++k) {
            float v = acc[t][k];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) red[warp][t * CO + k] = v;
        }
    __syncthreads();
    for (int i = threadIdx.x; i < 9 * CO; i += BW_THREADS) {
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < BW_THREADS / 32; ++w) v += red[w][i];
        const int t = i / CO, k = i - t * CO;
        atomicAdd(dW + k * 9 + t, v);   // parameter layout [CO][1][3][3]
    }
}

// ---- data gradient of the first conv w.r.t. the input image (enc1.0, src/model.py:93) ------------------------------------------
// dX[n,ci,y,x] = sum_{ky,kx,co} dR[n, y+1-ky, x+1-kx, co] * W[ky][kx][ci][co], zero padding.  Memory-bound: dR fp32 read once,
// dX fp32 written once, every output pixel its own sum (no atomics).  One CTA per output tile.
// in_channels == 1: every dR pixel of the haloed tile is first contracted over co with all 9 taps (v[t] = sum_co dR[co] W[t][co],
// dR read straight from global memory), then each output pixel adds its 9 shifted v[t] out of shared memory -- 72 B of shared
// traffic per pixel instead of 9 * C * 4 for re-reading a staged dR tile per tap.
template <int C>
__global__ void __launch_bounds__(BW_THREADS, 4) first_dgrad_kernel(const float* __restrict__ dR, const float* __restrict__ w,
                                                                     float* __restrict__ dx, int H, int W, int tiles_x, int tiles_y) {
    constexpr int TH = 16, TW = 64, PH = TH + 2, PW = TW + 2;
    __shared__ float wsm[9 * C];          // [tap][co]
    __shared__ float v[9][PH * PW];       // per tap: the contracted haloed tile
    for (int i = threadIdx.x; i < 9 * C; i += BW_THREADS) wsm[i] = __ldg(w + i);
    const int tiles_per_img = tiles_x * tiles_y;
    const int n = blockIdx.x / tiles_per_img, tr = blockIdx.x - n * tiles_per_img;
    const int y0 = (tr / tiles_x) * TH, x0 = (tr % tiles_x) * TW;
    __syncthreads();
    for (int q = threadIdx.x; q < PH * PW; q += BW_THREADS) {
        const int r = q / PW, c = q - r * PW;
        const int gy = y0 + r - 1, gx = x0 + c - 1;
        float d[C];
        if ((unsigned)gy < (unsigned)H && (unsigned)gx < (unsigned)W) {
            const float4* s = reinterpret_cast<const float4*>(dR + (((size_t)n * H + gy) * W + gx) * C);
#pragma unroll
            for (int k = 0; k < C / 4; ++k) {
                const float4 f = __ldg(s + k);
                d[4 * k] = f.x; d[4 * k + 1] = f.y; d[4 * k + 2] = f.z; d[4 * k + 3] = f.w;
            }
        } else {
#pragma unroll
            for (int k = 0; k < C; ++k) d[k] = 0.f;
        }
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            float a = 0.f;
#pragma unroll
            for (int k = 0; k < C; ++k) a = fmaf(d[k], wsm[t * C + k], a);
            v[t][q] = a;
        }
    }
    __syncthreads();
    for (int pix = threadIdx.x; pix < TH * TW; pix += BW_THREADS) {
        const int r = pix / TW, c = pix - r * TW;
        const int gy = y0 + r, gx = x0 + c;
        if (gy >= H || gx >= W) continue;
        float s = 0.f;
#pragma unroll
        for (int t = 0; t < 9; ++t) s += v[t][(r + 2 - t / 3) * PW + c + 2 - t % 3];
        dx[((size_t)n * H + gy) * W + gx] = s;
    }
}

// any in_channels and C (fs=12 with in=3, the wide fs=64 variant): the haloed dR tile staged in shared memory with an odd row
// stride (conflict-free reads for every C), one output pixel per thread, all input channels
__global__ void __launch_bounds__(BW_THREADS) first_dgrad_any_kernel(const float* __restrict__ dR, const float* __restrict__ w,
                                                                     float* __restrict__ dx, int H, int W, int CI, int C, int tiles_x,
                                                                     int tiles_y) {
    constexpr int TH = 8, TW = 32, PW = TW + 2;
    static_assert(TH * TW == BW_THREADS, "one output pixel per thread");
    extern __shared__ float dsm[];        // [(TH + 2) * PW][SC]
    const int SC = C | 1;
    const int tiles_per_img = tiles_x * tiles_y;
    const int n = blockIdx.x / tiles_per_img, tr = blockIdx.x - n * tiles_per_img;
    const int y0 = (tr / tiles_x) * TH, x0 = (tr % tiles_x) * TW;
    for (int i = threadIdx.x; i < (TH + 2) * PW * C; i += BW_THREADS) {
        const int q = i / C, co = i - q * C;
        const int r = q / PW, c = q - r * PW;
        const int gy = y0 + r - 1, gx = x0 + c - 1;
        dsm[q * SC + co] = ((unsigned)gy < (unsigned)H && (unsigned)gx < (unsigned)W) ? __ldg(dR + (((size_t)n * H + gy) * W + gx) * C + co) : 0.f;
    }
    __syncthreads();
    const int r = threadIdx.x / TW, c = threadIdx.x % TW;
    const int gy = y0 + r, gx = x0 + c;
    if (gy >= H || gx >= W) return;
    for (int ci = 0; ci < CI; ++ci) {
        float s = 0.f;
        for (int t = 0; t < 9; ++t) {
            const float* d = dsm + ((r + 2 - t / 3) * PW + c + 2 - t % 3) * SC;
            const float* wt = w + ((size_t)t * CI + ci) * C;
            for (int co = 0; co < C; ++co) s = fmaf(d[co], __ldg(wt + co), s);
        }
        dx[(((size_t)n * CI + ci) * H + gy) * W + gx] = s;
    }
}

// vector path: (pixel, 4-channel) items; C/4 a power of two <= 32 keeps a thread on one chunk and lets a warp cover all chunks
// vector kernels: C a power of two, 4 .. 128 (the shipped widths) and -- with the per-group prologue -- 256 .. 1024 (wider variants,
// groups of at most 32 warps' worth of work: groups <= C / 32 is not required, any divisor works)
inline bool ew_vec_ok(int dtype, int C, int H, int W) {
    (void)dtype;
    const int c4 = C / 4;
    return C % 4 == 0 && c4 >= 1 && c4 <= 256 && (c4 & (c4 - 1)) == 0 && (size_t)H * W * c4 < (size_t)1 << 30;
}
template <typename K>
inline int ew_allow_smem(K kern, size_t bytes, bool* done) {
    if (bytes <= 48 * 1024 || *done) return 0;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(element-wise backward): %s", cudaGetErrorString(e)); return 4; }
    *done = true;
    return 0;
}
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
inline bool aligned_raw(int dtype, const void* p) { return (reinterpret_cast<uintptr_t>(p) & (dtype == DG_F32 ? 15 : 7)) == 0; }
inline int ew_vec_blocks(size_t items) {
    // >= 8 items per thread where the image allows it: fewer CTAs, fewer double atomics on the [N,C,2] sums
    size_t b = (items + (size_t)BW_THREADS * 8 - 1) / ((size_t)BW_THREADS * 8);
    if (b > 1024) b = 1024;
    if (b < 1) b = 1;
    return (int)b;
}
}  // namespace

#define DG_BY_DTYPE(dt, CALL)                                          \
    switch (dt) {                                                      \
        case DG_F32: { using T = float; CALL; break; }                 \
        case DG_F16: { using T = __half; CALL; break; }                \
        case DG_BF16: { using T = __nv_bfloat16; CALL; break; }        \
        default: set_error("bad dtype %d", dt); return 2;             \
    }

int act_bwd_launch(int dtype, const void* raw, const double* stats, const float* gamma, const float* beta, const float* dA_a,
                   int stride_a, int off_a, const float* dA_b, int stride_b, int off_b, float* G, double* P, int N, int H,
                   int W, int C, int groups, float eps, cudaStream_t st) {
    ActBwdArgs a{raw, stats, gamma, beta, dA_a, stride_a, off_a, dA_b, stride_b, off_b, G, P, N, H, W, C, groups, eps};
    if (ew_vec_ok(dtype, C, H, W) && aligned16(G) && aligned16(dA_a) && aligned16(dA_b) && (stride_a & 3) == 0 &&
        (off_a & 3) == 0 && (stride_b & 3) == 0 && (off_b & 3) == 0 && aligned_raw(dtype, raw)) {
        dim3 vgrid(ew_vec_blocks((size_t)H * W * (C / 4)), N);
        const size_t vsmem = (size_t)C * 4 * sizeof(float) + (size_t)(BW_THREADS / 32) * C * 2 * sizeof(float) +
                             (C > 128 ? (size_t)groups * 2 * sizeof(double) : 0);
        if (vsmem > 96 * 1024) { set_error("act backward: %d channels need %zu B of shared memory", C, vsmem); return 3; }
        static bool attr[3] = {false, false, false};
        { int rc = 0; DG_BY_DTYPE(dtype, (rc = ew_allow_smem(act_bwd_vec_kernel<T>, vsmem, &attr[dtype]))); if (rc) return rc; }
        DG_BY_DTYPE(dtype, (act_bwd_vec_kernel<T><<<vgrid, BW_THREADS, vsmem, st>>>(a)));
        count_launch();
        return check_launch("act_bwd_vec");
    }
    dim3 grid(ew_blocks((size_t)H * W * C, C), N);
    const size_t smem = (size_t)C * 2 * sizeof(double) + (size_t)C * 4 * sizeof(float);
    DG_BY_DTYPE(dtype, (act_bwd_kernel<T><<<grid, BW_THREADS, smem, st>>>(a)));
    count_launch();
    return check_launch("act_bwd");
}

// dW [CO][1][3][3] += first-layer weight gradient; x fp32 [N,1,H,W], dR fp32 [N,H,W,CO]
int first_wgrad_launch(const float* x, const float* dR, float* dW, int N, int H, int W, int CO, cudaStream_t st, bool* handled) {
    *handled = false;
    if ((CO != 8 && CO != 16) || (reinterpret_cast<uintptr_t>(dR) & 15)) return 0;
    const int tx = (W + 63) / 64, ty = (H + 15) / 16;
    int blocks = tx * ty * N;
    if (blocks > 148 * 4) blocks = 148 * 4;
    if (CO == 8) first_wgrad_kernel<8><<<blocks, BW_THREADS, 0, st>>>(x, dR, dW, N, H, W, tx, ty);
    else first_wgrad_kernel<16><<<blocks, BW_THREADS, 0, st>>>(x, dR, dW, N, H, W, tx, ty);
    *handled = true;
    count_launch();
    return check_launch("first_wgrad");
}

// dX fp32 NCHW [N,CI,H,W] = first-layer input gradient; dR fp32 [N,H,W,C], w = the packed [3][3][CI][C] forward weights
int first_dgrad_launch(const float* dR, const float* w, float* dx, int N, int H, int W, int CI, int C, cudaStream_t st) {
    if (N < 1 || H < 1 || W < 1 || CI < 1 || C < 1) { set_error("first dgrad: bad shape %dx%dx%dx%d -> %d", N, C, H, W, CI); return 3; }
    if (CI == 1 && (C == 8 || C == 16) && aligned16(dR)) {
        const int tx = (W + 63) / 64, ty = (H + 15) / 16;
        if ((size_t)tx * ty * N > 0x7fffffff) { set_error("first dgrad: too many tiles"); return 3; }
        if (C == 8) first_dgrad_kernel<8><<<tx * ty * N, BW_THREADS, 0, st>>>(dR, w, dx, H, W, tx, ty);
        else first_dgrad_kernel<16><<<tx * ty * N, BW_THREADS, 0, st>>>(dR, w, dx, H, W, tx, ty);
        count_launch();
        return check_launch("first_dgrad");
    }
    const int tx = (W + 31) / 32, ty = (H + 7) / 8;
    if ((size_t)tx * ty * N > 0x7fffffff) { set_error("first dgrad: too many tiles"); return 3; }
    const size_t smem = (size_t)10 * 34 * (C | 1) * sizeof(float);
    if (smem > 227 * 1024) { set_error("first dgrad: %d channels need %zu B of shared memory", C, smem); return 3; }
    static size_t smem_set = 48 * 1024;
    if (smem > smem_set) {
        cudaError_t e = cudaFuncSetAttribute(first_dgrad_any_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) { set_error("first dgrad: cudaFuncSetAttribute(%zu B): %s", smem, cudaGetErrorString(e)); return 4; }
        smem_set = smem;
    }
    first_dgrad_any_kernel<<<tx * ty * N, BW_THREADS, smem, st>>>(dR, w, dx, H, W, CI, C, tx, ty);
    count_launch();
    return check_launch("first_dgrad_any");
}

// dRb (optional): ask for the bf16 copy instead of the in-place fp32 result; *wrote_bf16 reports whether that happened (only the
// vector kernel can: otherwise dR is in G as always)
int gn_bwd_apply_launch(int dtype, const void* raw, const double* stats, const float* gamma, const double* P, float* G,
                        float* dgamma, float* dbeta, int N, int H, int W, int C, int groups, float eps, cudaStream_t st,
                        void* dRb, bool* wrote_bf16) {
    if (wrote_bf16) *wrote_bf16 = false;
    GnBwdArgs a{raw, stats, gamma, P, G, nullptr, dgamma, dbeta, N, H, W, C, groups, eps};
    if (ew_vec_ok(dtype, C, H, W) && aligned16(G) && aligned_raw(dtype, raw)) {
        if (dRb != nullptr && wrote_bf16 != nullptr && (reinterpret_cast<uintptr_t>(dRb) & 15) == 0) {
            a.dRb = dRb;
            *wrote_bf16 = true;
        }
        dim3 vgrid(ew_vec_blocks((size_t)H * W * (C / 4)), N);
        const size_t gsmem = (size_t)(C * 5 + (C & 1)) * sizeof(float) + (C > 128 ? (size_t)groups * 4 * sizeof(double) : 0);
        DG_BY_DTYPE(dtype, (gn_bwd_apply_vec_kernel<T><<<vgrid, BW_THREADS, gsmem, st>>>(a)));
        count_launch();
        return check_launch("gn_bwd_apply_vec");
    }
    dim3 grid(ew_blocks((size_t)H * W * C, C), N);
    const size_t smem = (size_t)C * 5 * sizeof(float);
    DG_BY_DTYPE(dtype, (gn_bwd_apply_kernel<T><<<grid, BW_THREADS, smem, st>>>(a)));
    count_launch();
    return check_launch("gn_bwd_apply");
}

// nn.L1Loss forward (optimized_train.py:439,207/223): sum |y - t| in double, one atomic per CTA
__global__ void __launch_bounds__(BW_THREADS) l1_sum_kernel(const float* __restrict__ y, const float* __restrict__ t, size_t n, double* out) {
    __shared__ double red[BW_THREADS / 32];
    float acc = 0.f;
    const size_t n4 = n / 4;
    for (size_t i = (size_t)blockIdx.x * BW_THREADS + threadIdx.x; i < n4; i += (size_t)gridDim.x * BW_THREADS) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(y) + i), b = __ldg(reinterpret_cast<const float4*>(t) + i);
        acc += fabsf(a.x - b.x) + fabsf(a.y - b.y) + fabsf(a.z - b.z) + fabsf(a.w - b.w);
    }
    if (blockIdx.x == 0)
        for (size_t i = 4 * n4 + threadIdx.x; i < n; i += BW_THREADS) acc += fabsf(y[i] - t[i]);
    double d = (double)warp_sum(acc);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int k = 0; k < BW_THREADS / 32; ++k) s += red[k];
        atomicAdd(out, s);
    }
}

int l1_sum_launch(const float* y, const float* t, size_t n, double* out, cudaStream_t st) {
    if ((reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(t)) & 15) { set_error("l1: pointers must be 16-byte aligned"); return 2; }
    size_t blocks = (n / 4 + BW_THREADS * 8 - 1) / (BW_THREADS * 8);
    if (blocks < 1) blocks = 1;
    if (blocks > 1184) blocks = 1184;
    l1_sum_kernel<<<(unsigned)blocks, BW_THREADS, 0, st>>>(y, t, n, out);
    count_launch();
    return check_launch("l1_sum");
}

int head_bwd_launch(int dtype, const void* raw, const double* stats, const float* gamma, const float* beta, const float* dOut,
                    const float* w, float* G, double* P, float* dW, float* dB, int N, int H, int W, int C, int OC, int groups,
                    float eps, cudaStream_t st, const float* l1_y, const float* l1_target, const float* l1_scale, float l1_inv_numel) {
    if (OC > 4) { set_error("head backward: out_channels %d > 4", OC); return 3; }
    HeadBwdArgs a{raw, stats, gamma, beta, dOut, w, G, P, dW, dB, N, H, W, C, OC, groups, eps, l1_y, l1_target, l1_scale, l1_inv_numel};
    if (OC == 1 && (C == 8 || C == 16) && aligned16(G) && aligned_raw(dtype, raw) && N <= 65535) {
        int fx = (H * W + BW_THREADS * 16 - 1) / (BW_THREADS * 16);
        if (fx < 1) fx = 1;
        dim3 fgrid(fx, N);
        if (C == 8) { DG_BY_DTYPE(dtype, (head_bwd_fast_kernel<T, 8><<<fgrid, BW_THREADS, 0, st>>>(a))); }
        else { DG_BY_DTYPE(dtype, (head_bwd_fast_kernel<T, 16><<<fgrid, BW_THREADS, 0, st>>>(a))); }
        count_launch();
        return check_launch("head_bwd_fast");
    }
    int bx = (H * W + BW_THREADS * 4 - 1) / (BW_THREADS * 4);
    if (bx > 512) bx = 512;
    dim3 grid(bx, N);
    const size_t smem = (size_t)(2 * C + OC * C + OC) * sizeof(double) + (size_t)(4 * C + OC * C) * sizeof(float);
    DG_BY_DTYPE(dtype, (head_bwd_kernel<T><<<grid, BW_THREADS, smem, st>>>(a)));
    count_launch();
    return check_launch("head_bwd");
}

int convt_bwd_launch(int dtype, const float* dCat, int stride, const float* wt, const float* wt_t, const void* raw_low,
                     const double* stats, const float* gamma, const float* beta, float* dAlow, float* dWt, float* dBias,
                     float* coefbuf, int N, int H, int W, int Cl, int Cu, int groups, float eps, cudaStream_t st,
                     const void* wtc_bf16, const DgradAct* act, bool* act_fused, const void* w2_tc_bf16, void* scratch_bf16) {
    if (act_fused) *act_fused = false;
    if (Cu % 4 || (stride % 4) || (reinterpret_cast<uintptr_t>(dCat) & 15)) { set_error("convT backward: unaligned gradient"); return 3; }
    ConvtBwdArgs a{dCat, stride, wt, wt_t, raw_low, stats, gamma, beta, dAlow, dWt, nullptr, coefbuf, N, H, W, Cl, Cu, groups, eps};
    if (dWt != nullptr) {
        gn_mean_rstd_kernel<<<N, 128, 0, st>>>(stats, coefbuf, Cl, groups, (double)(H / 2) * (W / 2), eps);
        count_launch();
    }
    const size_t total = (size_t)N * (H / 2) * (W / 2) * Cl;
    int rc = 0;
    bool data_done = dAlow == nullptr;   // NULL: nothing below the ConvTranspose wants a gradient
    if (!data_done && dtype != DG_F32 && wtc_bf16 != nullptr) {   // tensor cores where covered (dgrad_tc.cu)
        if (act != nullptr && act_fused != nullptr) {   // dAlow is then G of the low-resolution producer, never the plain gradient
            rc = convt_dgrad_tc_launch(dCat, stride, wtc_bf16, dAlow, N, H, W, Cl, Cu, st, &data_done, act);
            if (rc) return rc;
            *act_fused = data_done;
        }
        if (!data_done) {
            rc = convt_dgrad_tc_launch(dCat, stride, wtc_bf16, dAlow, N, H, W, Cl, Cu, st, &data_done);
            if (rc) return rc;
        }
    }
    if (!data_done && dtype != DG_F32 && w2_tc_bf16 != nullptr && scratch_bf16 != nullptr) {   // wider variants: tcgen05 GEMM (conv3x3_t5.cu)
        rc = convt_dgrad_t5_launch(dCat, stride, scratch_bf16, w2_tc_bf16, dAlow, N, H, W, Cl, Cu, st, &data_done);
        if (rc) return rc;
    }
    if (!data_done) {
        if (wt_t == nullptr) { set_error("convT backward: the CUDA-core data gradient needs up_w_t"); return 2; }
        convt_bwd_data_kernel<<<ew_blocks(total, Cl), BW_THREADS, 0, st>>>(a);
        count_launch();
        rc = check_launch("convt_bwd_data");
        if (rc) return rc;
    }
    // weight + bias gradient on the tensor cores where the configuration is covered (wgrad_tc.cu: the bias sum rides on the
    // gradient staging), else the two CUDA-core kernels below.  dWt / dBias NULL = frozen: its kernel does not run (a frozen
    // weight with a trained bias takes the bias kernel alone)
    if (dWt != nullptr) {
        bool handled = false;
        rc = convt_wgrad_tc_launch(dtype, dCat, stride, raw_low, stats, gamma, beta, dWt, dBias, N, H, W, Cl, Cu, groups, eps, st, &handled);
        if (rc || handled) return rc;
    }
    if (dBias != nullptr) {
        ConvtBwdArgs ab = a;
        ab.dBias = dBias;
        int bb = (int)(((size_t)N * H * W * Cu + BW_THREADS * 16 - 1) / (BW_THREADS * 16));
        if (bb > 1024) bb = 1024;
        if (bb < 1) bb = 1;
        convt_bwd_bias_kernel<<<bb, BW_THREADS, (size_t)Cu * sizeof(float), st>>>(ab);
        count_launch();
    }
    if (dWt == nullptr) return check_launch("convt_bwd_bias");
    // weight gradient: 256 combos per CTA
    // slab sized for ~32 KB of staged operands
    const int ncombo = 4 * Cl * Cu;
    const int per_cta_ci = (BW_THREADS / Cu) < 1 ? 1 : (BW_THREADS / Cu) + 1;
    int width = (Cl * Cu >= BW_THREADS) ? (per_cta_ci + Cu) : (Cl + 4 * Cu);  // floats staged per low pixel (upper bound)
    // ... which the kernel's own (ci, position) ranges can exceed when Cl * Cu is not a multiple of BW_THREADS (a CTA whose combos
    // cross a position stages every input channel and two positions): take the largest nci + nab * Cu over the CTAs
    for (int c_first = 0; c_first < ncombo; c_first += BW_THREADS) {
        const int c_last = min(c_first + BW_THREADS, ncombo) - 1;
        const int ab_lo = c_first / (Cl * Cu), ab_hi = c_last / (Cl * Cu);
        const int nci = ab_hi > ab_lo ? Cl : (c_last / Cu) % Cl - (c_first / Cu) % Cl + 1;
        width = max(width, nci + (ab_hi - ab_lo + 1) * Cu);
    }
    int slab = 8192 / width;
    if (slab > 128) slab = 128;
    if (slab < 8) slab = 8;
    const int npix = N * (H / 2) * (W / 2);
    int slabs = (npix + slab - 1) / slab;
    const int gx = (ncombo + BW_THREADS - 1) / BW_THREADS;
    int gy = 2048 / gx;
    if (gy < 1) gy = 1;
    if (gy > slabs) gy = slabs;
    dim3 grid(gx, gy);
    const size_t smem = (size_t)slab * (size_t)width * sizeof(float);
    if (smem > 96 * 1024) { set_error("convT backward: %zu B of shared memory", smem); return 3; }
    static bool attr[3] = {false, false, false};
    const int di = dtype == DG_F32 ? 0 : (dtype == DG_F16 ? 1 : 2);
    if (!attr[di]) {
        DG_BY_DTYPE(dtype, (cudaFuncSetAttribute(convt_bwd_weight_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024)));
        attr[di] = true;
    }
    DG_BY_DTYPE(dtype, (convt_bwd_weight_kernel<T><<<grid, BW_THREADS, smem, st>>>(a, slab)));
    count_launch();
    return check_launch("convt_bwd_weight");
}

int adamw_launch(float* p, const float* g, float* m, float* v, size_t n, double* sumsq_scratch, float max_norm, float lr,
                 float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(sumsq_scratch, 0, sizeof(double), st);
    if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return 10; }
    int blocks = (int)((n + BW_THREADS - 1) / BW_THREADS);
    if (blocks > 592) blocks = 592;
    sumsq_kernel<<<blocks, BW_THREADS, 0, st>>>(g, n, sumsq_scratch);
    count_launch();
    AdamwArgs a{p, g, m, v, n, sumsq_scratch, max_norm, lr, beta1, beta2, eps, weight_decay,
                (float)(1.0 - pow((double)beta1, step)), (float)sqrt(1.0 - pow((double)beta2, step)), grad_scale};
    adamw_kernel<<<blocks, BW_THREADS, 0, st>>>(a);
    count_launch();
    return check_launch("adamw");
}

int adamw_dev_launch(float* p, const float* g, float* m, float* v, size_t n, double* sumsq_scratch, float max_norm, const float* lr_dev,
                     float beta1, float beta2, float eps, float weight_decay, int32_t* step_dev, float grad_scale, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(sumsq_scratch, 0, sizeof(double), st);
    if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return 10; }
    int blocks = (int)((n + BW_THREADS - 1) / BW_THREADS);
    if (blocks > 592) blocks = 592;
    step_bump_kernel<<<1, 1, 0, st>>>(step_dev);
    count_launch();
    sumsq_kernel<<<blocks, BW_THREADS, 0, st>>>(g, n, sumsq_scratch);
    count_launch();
    AdamwDevArgs a{p, g, m, v, n, sumsq_scratch, step_dev, lr_dev, max_norm, beta1, beta2, eps, weight_decay, grad_scale};
    adamw_dev_kernel<<<blocks, BW_THREADS, 0, st>>>(a);
    count_launch();
    return check_launch("adamw (device step)");
}

}  // namespace dg
