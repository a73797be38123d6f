// Backward pieces that only OptimizedUNet needs (autograd of src/optimized_model.py:118-158 as driven by
// optimized_train.py:210/226); everything else of its backward is the per-op kernels LightweightUNet already uses
// (act_bwd / gn_bwd_apply / head_bwd in backward.cu, the generic conv as data gradient, the WGRAD mode of the same kernel).
//
//   nn.Upsample(x2, nearest) + conv (_upblock, :111-116): the conv's input gradient lives on the up-sampled grid; the producer
//       gets the SUM of the 2x2 positions that replicate it                                              -> grad_gather (u)
//   torch.cat((dec, enc * att)) (:141-156): the skip half of the decoder conv's input gradient reaches the activated skip
//       tensor multiplied by att[n][c]; the same tensor also feeds the next encoder level through AvgPool2d (x0.25,
//       replicated) and ChannelAttention's global mean (a per-(n, c) constant)                            -> grad_gather (a, b, add)
//   ChannelAttention (:185-202): d att[n][c] = sum_pixels d(enc*att) * enc                                -> scale_bwd_sum
//       then the two bias-free Linear layers with SiLU / Sigmoid backwards (one CTA per sample)            -> se_bwd
// All gradient tensors are fp32 NHWC; saved raw activations are read in their storage type.
#include "common.cuh"

namespace dg {

namespace {
constexpr int OB_THREADS = 256;

struct GatherArgs {
    const float* a; int sa, oa; const float* a_scale;   // same-resolution gradient [N,H,W,sa], channels oa..oa+C, optional x scale[n][c]
    const float* b; int sb, ob;                         // half-resolution gradient [N,H/2,W/2,sb]: AvgPool2d backward (x 0.25, replicated)
    const float* u; int su, ou;                         // double-resolution gradient [N,2H,2W,su]: nearest-x2 backward (2x2 sum)
    const float* add;                                   // per-(n, c) constant [N,C]
    float* out;                                         // dense [N,H,W,C]
    int N, H, W, C;
};

template <int V>
__device__ __forceinline__ void ld(const float* p, float (&v)[V]) {
    if constexpr (V == 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
        v[0] = __ldg(p);
    }
}

// V = 4: C, every stride and offset are multiples of 4 and every pointer is 16-byte aligned (checked by the host)
template <int V>
__global__ void __launch_bounds__(OB_THREADS) grad_gather_kernel(const GatherArgs p) {
    const int CV = p.C / V;
    const size_t total = (size_t)p.N * p.H * p.W * CV;
    for (size_t e = (size_t)blockIdx.x * OB_THREADS + threadIdx.x; e < total; e += (size_t)gridDim.x * OB_THREADS) {
        const int c = (int)(e % CV) * V;
        const size_t pix = e / CV;   // (n*H + y)*W + x
        const int x = (int)(pix % p.W);
        const size_t row = pix / p.W;
        const int y = (int)(row % p.H);
        const int n = (int)(row / p.H);
        float acc[V];
#pragma unroll
        for (int k = 0; k < V; ++k) acc[k] = 0.f;
        if (p.a != nullptr) {
            float t[V];
            ld<V>(p.a + pix * p.sa + p.oa + c, t);
            if (p.a_scale != nullptr) {
                float s[V];
                ld<V>(p.a_scale + (size_t)n * p.C + c, s);
#pragma unroll
                for (int k = 0; k < V; ++k) t[k] *= s[k];
            }
#pragma unroll
            for (int k = 0; k < V; ++k) acc[k] += t[k];
        }
        if (p.b != nullptr) {
            float t[V];
            const size_t q = ((size_t)n * (p.H / 2) + y / 2) * (p.W / 2) + x / 2;
            ld<V>(p.b + q * p.sb + p.ob + c, t);
#pragma unroll
            for (int k = 0; k < V; ++k) acc[k] = fmaf(0.25f, t[k], acc[k]);
        }
        if (p.u != nullptr) {
#pragma unroll
            for (int dy = 0; dy < 2; ++dy)
#pragma unroll
                for (int dx = 0; dx < 2; ++dx) {
                    float t[V];
                    const size_t q = ((size_t)n * (2 * p.H) + 2 * y + dy) * (2 * p.W) + 2 * x + dx;
                    ld<V>(p.u + q * p.su + p.ou + c, t);
#pragma unroll
                    for (int k = 0; k < V; ++k) acc[k] += t[k];
                }
        }
        if (p.add != nullptr) {
            float t[V];
            ld<V>(p.add + (size_t)n * p.C + c, t);
#pragma unroll
            for (int k = 0; k < V; ++k) acc[k] += t[k];
        }
        float* o = p.out + pix * p.C + c;
        if constexpr (V == 4) *reinterpret_cast<float4*>(o) = make_float4(acc[0], acc[1], acc[2], acc[3]);
        else *o = acc[0];
    }
}

// ---- out[n][c] += sum_pixels d[n,pix,od+c] * SiLU(GN(raw))[n,pix,c] --------------------------------------------------------
struct ScaleBwdArgs {
    const void* raw; const double* stats; const float* gamma; const float* beta;
    const float* d; int sd, od;
    double* out;
    int N, H, W, C, groups; float eps;
};

template <typename T>
__global__ void __launch_bounds__(OB_THREADS) scale_bwd_sum_kernel(const ScaleBwdArgs p) {
    extern __shared__ double osm[];                       // [C] partial sums, then float [C][2] GroupNorm affine
    const int C = p.C;
    double* psm = osm;
    float* coef = reinterpret_cast<float*>(psm + C);
    const int n = blockIdx.y;
    const int HW = p.H * p.W;
    for (int c = threadIdx.x; c < C; c += OB_THREADS) {
        float a, b;
        gn_coef(p.stats, p.gamma, p.beta, n, C, p.groups, c, (double)HW, p.eps, a, b);
        coef[2 * c] = a; coef[2 * c + 1] = b;
        psm[c] = 0.0;
    }
    __syncthreads();
    const T* raw = reinterpret_cast<const T*>(p.raw);
    const size_t total = (size_t)HW * C;
    const size_t stride = (size_t)gridDim.x * OB_THREADS;
    double acc = 0.0;
    int cur_c = -1;   // a thread stays on one channel when the grid stride is a multiple of C (C a power of two <= 256)
    for (size_t e = (size_t)blockIdx.x * OB_THREADS + threadIdx.x; e < total; e += stride) {
        const int c = (int)(e % C);
        const size_t pix = e / C;
        if (c != cur_c) {
            if (cur_c >= 0) atomicAdd(&psm[cur_c], acc);
            cur_c = c; acc = 0.0;
        }
        const float y = fmaf(Store<T>::to_f(raw[(size_t)n * total + e]), coef[2 * c], coef[2 * c + 1]);
        const float act = y / (1.f + __expf(-y));
        acc += (double)(act * __ldg(p.d + ((size_t)n * HW + pix) * p.sd + p.od + c));
    }
    if (cur_c >= 0) atomicAdd(&psm[cur_c], acc);
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += OB_THREADS) atomicAdd(p.out + (size_t)n * C + c, psm[c]);
}

// ---- ChannelAttention backward: one CTA per sample --------------------------------------------------------------------------
// forward (se.cu): m = act_sum / plane; a = W1 m; h = silu(a); z = W2 h; att = sigmoid(z)
// backward: dz = datt * att (1 - att); dW2 += dz h^T; dh = W2^T dz; da = dh * silu'(a); dW1 += da m^T; dm = W1^T da;
//           every pixel of the activated tensor receives dm[c] / plane (the mean's gradient)
// WANT_W: accumulate dW1 / dW2 (a frozen ChannelAttention skips them); WANT_ADD: write dm / plane (nothing upstream of the
// attended tensor needs a gradient: skip it).  The launcher never instantiates <false, false>.
template <bool WANT_W, bool WANT_ADD>
__global__ void se_bwd_kernel(const double* __restrict__ act_sum, double inv_plane, const float* __restrict__ w1,
                              const float* __restrict__ w2, const double* __restrict__ dscale, int C, int hidden,
                              float* __restrict__ add, float* __restrict__ dw1, float* __restrict__ dw2) {
    extern __shared__ float bsm[];   // mean[C], dz[C], a[hidden], h[hidden], da[hidden]
    float* mean = bsm;
    float* dz = mean + C;
    float* pre = dz + C;
    float* h = pre + hidden;
    float* da = h + hidden;
    const int n = blockIdx.x;
    for (int c = threadIdx.x; c < C; c += blockDim.x) mean[c] = (float)(act_sum[(size_t)n * C + c] * inv_plane);
    __syncthreads();
    for (int j = threadIdx.x; j < hidden; j += blockDim.x) {
        float a = 0.f;
        for (int c = 0; c < C; ++c) a = fmaf(w1[j * C + c], mean[c], a);
        pre[j] = a;
        h[j] = a / (1.f + __expf(-a));
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        float z = 0.f;
        for (int j = 0; j < hidden; ++j) z = fmaf(w2[c * hidden + j], h[j], z);
        const float s = 1.f / (1.f + __expf(-z));
        dz[c] = (float)dscale[(size_t)n * C + c] * s * (1.f - s);
    }
    __syncthreads();
    for (int j = threadIdx.x; j < hidden; j += blockDim.x) {
        float d = 0.f;
        for (int c = 0; c < C; ++c) d = fmaf(w2[c * hidden + j], dz[c], d);
        const float s = 1.f / (1.f + __expf(-pre[j]));
        da[j] = d * s * (1.f + pre[j] * (1.f - s));
    }
    if constexpr (WANT_W) {
        for (int i = threadIdx.x; i < C * hidden; i += blockDim.x) atomicAdd(dw2 + i, dz[i / hidden] * h[i % hidden]);
    }
    __syncthreads();
    if constexpr (WANT_W) {
        for (int i = threadIdx.x; i < hidden * C; i += blockDim.x) atomicAdd(dw1 + i, da[i / C] * mean[i % C]);
    }
    if constexpr (WANT_ADD) {
        for (int c = threadIdx.x; c < C; c += blockDim.x) {
            float d = 0.f;
            for (int j = 0; j < hidden; ++j) d = fmaf(w1[j * C + c], da[j], d);
            add[(size_t)n * C + c] = (float)((double)d * inv_plane);
        }
    }
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
}  // namespace

int grad_gather_launch(const float* a, int sa, int oa, const float* a_scale, const float* b, int sb, int ob, const float* u, int su,
                       int ou, const float* add, float* out, int N, int H, int W, int C, cudaStream_t st) {
    GatherArgs g{a, sa, oa, a_scale, b, sb, ob, u, su, ou, add, out, N, H, W, C};
    const bool vec = (C % 4 == 0) && al16(out) && (a == nullptr || (al16(a) && sa % 4 == 0 && oa % 4 == 0)) &&
                     (a_scale == nullptr || al16(a_scale)) && (b == nullptr || (al16(b) && sb % 4 == 0 && ob % 4 == 0)) &&
                     (u == nullptr || (al16(u) && su % 4 == 0 && ou % 4 == 0)) && (add == nullptr || al16(add));
    const size_t items = (size_t)N * H * W * (vec ? C / 4 : C);
    size_t blocks = (items + OB_THREADS - 1) / OB_THREADS;
    if (blocks > 148 * 16) blocks = 148 * 16;
    if (blocks < 1) blocks = 1;
    if (vec) grad_gather_kernel<4><<<(unsigned)blocks, OB_THREADS, 0, st>>>(g);
    else grad_gather_kernel<1><<<(unsigned)blocks, OB_THREADS, 0, st>>>(g);
    count_launch();
    return check_launch("grad_gather");
}

int scale_bwd_sum_launch(int dtype, const void* raw, const double* stats, const float* gamma, const float* beta, const float* d,
                         int sd, int od, double* out, int N, int H, int W, int C, int groups, float eps, cudaStream_t st) {
    ScaleBwdArgs a{raw, stats, gamma, beta, d, sd, od, out, N, H, W, C, groups, eps};
    size_t bx = ((size_t)H * W * C + (size_t)OB_THREADS * 16 - 1) / ((size_t)OB_THREADS * 16);
    if (bx > 148 * 4) bx = 148 * 4;
    if (bx < 1) bx = 1;
    dim3 grid((unsigned)bx, N);
    const size_t smem = (size_t)C * sizeof(double) + (size_t)C * 2 * sizeof(float);
    switch (dtype) {
        case DG_F32: scale_bwd_sum_kernel<float><<<grid, OB_THREADS, smem, st>>>(a); break;
        case DG_F16: scale_bwd_sum_kernel<__half><<<grid, OB_THREADS, smem, st>>>(a); break;
        case DG_BF16: scale_bwd_sum_kernel<__nv_bfloat16><<<grid, OB_THREADS, smem, st>>>(a); break;
        default: set_error("bad dtype %d", dtype); return 2;
    }
    count_launch();
    return check_launch("scale_bwd_sum");
}

int se_bwd_launch(const double* act_sum, double plane, const float* w1, const float* w2, const double* dscale, int N, int C,
                  int hidden, float* add, float* dw1, float* dw2, cudaStream_t st) {
    const size_t smem = (size_t)(2 * C + 3 * hidden) * sizeof(float);
    if (dw1 != nullptr && add != nullptr)
        se_bwd_kernel<true, true><<<N, 128, smem, st>>>(act_sum, 1.0 / plane, w1, w2, dscale, C, hidden, add, dw1, dw2);
    else if (dw1 != nullptr)
        se_bwd_kernel<true, false><<<N, 128, smem, st>>>(act_sum, 1.0 / plane, w1, w2, dscale, C, hidden, add, dw1, dw2);
    else
        se_bwd_kernel<false, true><<<N, 128, smem, st>>>(act_sum, 1.0 / plane, w1, w2, dscale, C, hidden, add, dw1, dw2);
    count_launch();
    return check_launch("se_bwd");
}

}  // namespace dg
