// Generic fused 3x3 conv (CUDA cores, fp32 accumulate), any channel counts / storage type.
//
// This is the fp32 tier and the any-shape path of dg_conv3x3_fused: one CTA computes a
// 32 x (4*NTY) output tile for 8*NCOG output channels; input channels are streamed through
// shared memory in chunks of 8 after the consumer-side prologue (GroupNorm apply + SiLU
// [+ SE scale], then identity / 2x2 average pool / nearest x2 / fused ConvTranspose2d(2,2)),
// so neither the normalised, pooled, up-sampled nor the concatenated tensor reaches HBM.
// The epilogue writes the raw conv output once (NHWC) and accumulates its per-(n, channel)
// sum / sum-of-squares for the next layer's GroupNorm.
//
// Reference semantics: src/model.py:92-99 (block), :35-41 (AvgPool2d), :47-53 (ConvTranspose2d),
// :116-128 (torch.cat((up, skip), 1)); src/optimized_model.py:111-116 (_upblock), :199-202 (SE scale).
#include "common.cuh"

namespace dg {

constexpr int CK = 8;        // input channels per smem chunk
constexpr int TW = 32;       // tile width (one warp along x)
constexpr int AW = TW + 2;   // halo tile width
constexpr int LW = TW / 2 + 2;
constexpr int NTHREADS = 256;

__host__ __device__ inline int src_out_channels(const dg_src& s) {
    return s.xform == DG_X_CONVT2 ? s.ct_cout : s.channels;
}

struct GenericCfg {
    int lch;        // low-res channels staged per pass (CONVT2)
    int coef_off;   // float offsets into dynamic smem
    int low_off;
    int cobatches;
    // WGRAD mode (backward of the conv weights, autograd of src/model.py:93,96): the same staging prologue rebuilds the
    // activated input tile, and instead of the convolution the CTA correlates it with the output-gradient tile:
    //   dW[tap][ci][co] += sum_pixels act[pixel + tap][ci] * dR[pixel][co]
    const float* dR;  // [N,H,W,cout] fp32 gradient w.r.t. the raw conv output
    float* dW;        // fp32, accumulated atomically at dW[tap*s_tap + ci*s_ci + co*s_co]
    int s_tap, s_ci, s_co;
};

template <typename T, int NTY, int NCOG, bool WGRAD>
__global__ void __launch_bounds__(NTHREADS) conv3x3_generic_kernel(const dg_conv3x3_args p, const GenericCfg cfg) {
    constexpr int TH = 4 * NTY;
    constexpr int AH = TH + 2;
    constexpr int LH = TH / 2 + 2;
    constexpr int COB = 8 * NCOG;  // output channels per CTA

    extern __shared__ double smem_d[];
    double* statsm = smem_d;                                   // [COB][2]
    float* act = reinterpret_cast<float*>(statsm + 2 * COB);   // [CK][AH][AW]
    float* wsm = act + CK * AH * AW;                           // [9][CK][COB]
    float* coef = reinterpret_cast<float*>(smem_d) + cfg.coef_off;  // per source [C][3] (a, b, scale)
    float* low = reinterpret_cast<float*>(smem_d) + cfg.low_off;  // [LH][LW][lch+1]

    const int tid = threadIdx.x;
    const int tx = tid & 31;
    const int wrp = tid >> 5;
    const int ty = wrp % NTY;
    const int cog = wrp / NTY;
    const int n = blockIdx.z / cfg.cobatches;
    const int cob = blockIdx.z % cfg.cobatches;
    const int x0 = blockIdx.x * TW;
    const int y0 = blockIdx.y * TH;
    const int H = p.H, W = p.W, Cout = p.cout;
    const int co_cta = cob * COB;

    int cin_total = 0;
    for (int s = 0; s < p.nsrc; ++s) cin_total += src_out_channels(p.src[s]);

    // ---- prologue: GroupNorm coefficients of every source channel -------------------------
    {
        float* cf = coef;
        for (int s = 0; s < p.nsrc; ++s) {
            const dg_src& S = p.src[s];
            int Hs = H, Ws = W;
            if (S.xform == DG_X_POOL2) { Hs = 2 * H; Ws = 2 * W; }
            if (S.xform == DG_X_UP2 || S.xform == DG_X_CONVT2) { Hs = H / 2; Ws = W / 2; }
            for (int c = tid; c < S.channels; c += NTHREADS) {
                float a = 1.f, b = 0.f;
                if (S.coef != nullptr) {
                    a = __ldg(S.coef + (size_t)(n * S.channels + c) * 2);
                    b = __ldg(S.coef + (size_t)(n * S.channels + c) * 2 + 1);
                } else if (S.stats != nullptr) {
                    gn_coef(S.stats, S.gamma, S.beta, n, S.channels, S.groups, c, (double)Hs * Ws, p.eps, a, b);
                }
                cf[3 * c] = a;
                cf[3 * c + 1] = b;
                cf[3 * c + 2] = S.scale ? S.scale[(size_t)n * S.channels + c] : 1.f;
            }
            cf += 3 * S.channels;
        }
        if (tid < 2 * COB) statsm[tid] = 0.0;
        if constexpr (WGRAD) {
            // output-gradient tile dRs[(r*32 + c)*COB + co] (aliases the weight-chunk region), zero outside the image
            for (int idx = tid; idx < TH * TW * COB; idx += NTHREADS) {
                const int co = idx % COB;
                const int pix = idx / COB;
                const int gy = y0 + pix / TW, gx = x0 + pix % TW;
                float v = 0.f;
                if (gy < H && gx < W && co_cta + co < Cout)
                    v = __ldg(cfg.dR + ((size_t)(n * H + gy) * W + gx) * Cout + co_cta + co);
                wsm[idx] = v;
            }
        }
    }
    __syncthreads();

    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int k = 0; k < 8; ++k) acc[i][k] = 0.f;

    int ci_base = 0;  // channel offset of the current source inside the concat
    const float* cf = coef;
    for (int s = 0; s < p.nsrc; ++s) {
        const dg_src& S = p.src[s];
        const int Cs = S.channels;
        const int Co_s = src_out_channels(S);
        const T* raw = reinterpret_cast<const T*>(S.raw);
        const bool vec_in = (Cs % 8 == 0) && ((reinterpret_cast<uintptr_t>(S.raw) & 15) == 0);
        bool low_staged = false;

        for (int c0 = 0; c0 < Co_s; c0 += CK) {
            const int cn = min(CK, Co_s - c0);
            // ---- (1) stage the activated input chunk into act[ck][r][c] ----------------------
            if (S.xform == DG_X_CONVT2) {
                const int Hl = H / 2, Wl = W / 2;
                const int li0 = (y0 >> 1) - 1, lj0 = (x0 >> 1) - 1;
                const int lp = cfg.lch + 1;
                for (int lc0 = 0; lc0 < Cs; lc0 += cfg.lch) {
                    const int lcn = min(cfg.lch, Cs - lc0);
                    if (!(low_staged && Cs <= cfg.lch)) {
                        __syncthreads();  // previous users of `low` are done
                        // stage activated low-res tile, 8 channels per thread-iteration
                        const int lchunks = (lcn + 7) / 8;
                        for (int idx = tid; idx < LH * LW * lchunks; idx += NTHREADS) {
                            const int ch = idx % lchunks;
                            const int pix = idx / lchunks;
                            const int lj = pix % LW, li = pix / LW;
                            const int gi = li0 + li, gj = lj0 + lj;
                            const int cc = lc0 + ch * 8;
                            const int ccn = min(8, lc0 + lcn - cc);
                            float v[8];
                            if (gi >= 0 && gi < Hl && gj >= 0 && gj < Wl) {
                                load8<T>(raw + ((size_t)(n * Hl + gi) * Wl + gj) * Cs + cc, ccn, vec_in, v);
#pragma unroll
                                for (int k = 0; k < 8; ++k) {
                                    if (k < ccn) {
                                        float y = v[k] * cf[3 * (cc + k)] + cf[3 * (cc + k) + 1];
                                        if (S.silu) y = silu_f(y);
                                        v[k] = y * cf[3 * (cc + k) + 2];
                                    }
                                }
                            } else {
#pragma unroll
                                for (int k = 0; k < 8; ++k) v[k] = 0.f;
                            }
#pragma unroll
                            for (int k = 0; k < 8; ++k)
                                if (k < ccn) low[pix * lp + ch * 8 + k] = v[k];
                        }
                        low_staged = true;
                        __syncthreads();
                    }
                    // accumulate the transposed conv for up-channels [c0, c0+cn) into act
                    for (int idx = tid; idx < AH * AW; idx += NTHREADS) {
                        const int c = idx % AW, r = idx / AW;
                        const int gy = y0 + r - 1, gx = x0 + c - 1;
                        float u[8];
                        if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
                            if (lc0 == 0) {
#pragma unroll
                                for (int k = 0; k < 8; ++k) u[k] = (k < cn) ? S.ct_b[c0 + k] : 0.f;
                            } else {
#pragma unroll
                                for (int k = 0; k < 8; ++k) u[k] = act[(k * AH + r) * AW + c];
                            }
                            const int li = (gy >> 1) - li0, lj = (gx >> 1) - lj0;
                            const int ab = ((gy & 1) << 1) | (gx & 1);
                            const float* lrow = low + (li * LW + lj) * lp;
                            const float* wrow = S.ct_w + ((size_t)ab * Cs + lc0) * Co_s + c0;
                            for (int ci = 0; ci < lcn; ++ci) {
                                const float xv = lrow[ci];
#pragma unroll
                                for (int k = 0; k < 8; ++k)
                                    if (k < cn) u[k] = fmaf(xv, __ldg(wrow + (size_t)ci * Co_s + k), u[k]);
                            }
                        } else {
#pragma unroll
                            for (int k = 0; k < 8; ++k) u[k] = 0.f;  // zero pad of the CONCATENATED tensor
                        }
#pragma unroll
                        for (int k = 0; k < 8; ++k) act[(k * AH + r) * AW + c] = u[k];
                    }
                }
            } else {
                double asum[8];
                const bool want_sum = (p.act_sum != nullptr) && s == 0 && cob == 0;
#pragma unroll
                for (int k = 0; k < 8; ++k) asum[k] = 0.0;
                for (int idx = tid; idx < AH * AW; idx += NTHREADS) {
                    const int c = idx % AW, r = idx / AW;
                    const int gy = y0 + r - 1, gx = x0 + c - 1;
                    float v[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = 0.f;
                    if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
                        if (S.xform == DG_X_IMAGE) {
                            const float* img = reinterpret_cast<const float*>(S.raw);
#pragma unroll
                            for (int k = 0; k < 8; ++k)
                                if (k < cn) v[k] = __ldg(img + ((size_t)(n * Cs + c0 + k) * H + gy) * W + gx);
                        } else if (S.xform == DG_X_IMAGE_U8) {  // float32(u) / 255.0f, api/app.py:153
                            const unsigned char* img = reinterpret_cast<const unsigned char*>(S.raw);
#pragma unroll
                            for (int k = 0; k < 8; ++k)
                                if (k < cn) v[k] = __fdiv_rn((float)__ldg(img + ((size_t)(n * Cs + c0 + k) * H + gy) * W + gx), 255.f);
                        } else if (S.xform == DG_X_POOL2) {
                            const int Hs = 2 * H, Ws = 2 * W;
#pragma unroll
                            for (int q = 0; q < 4; ++q) {
                                float t[8];
                                load8<T>(raw + ((size_t)(n * Hs + 2 * gy + (q >> 1)) * Ws + 2 * gx + (q & 1)) * Cs + c0,
                                         cn, vec_in, t);
#pragma unroll
                                for (int k = 0; k < 8; ++k) {
                                    if (k < cn) {
                                        float y = t[k] * cf[3 * (c0 + k)] + cf[3 * (c0 + k) + 1];
                                        if (S.silu) y = silu_f(y);
                                        v[k] += y;
                                    }
                                }
                            }
                            const bool interior = r >= 1 && r <= TH && c >= 1 && c <= TW;
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                if (k < cn) {
                                    if (want_sum && interior) asum[k] += (double)v[k];
                                    v[k] *= 0.25f * cf[3 * (c0 + k) + 2];
                                }
                            }
                        } else {
                            int sy = gy, sx = gx, Hs = H, Ws = W;
                            if (S.xform == DG_X_UP2) { sy = gy >> 1; sx = gx >> 1; Hs = H / 2; Ws = W / 2; }
                            load8<T>(raw + ((size_t)(n * Hs + sy) * Ws + sx) * Cs + c0, cn, vec_in, v);
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                if (k < cn) {
                                    float y = v[k] * cf[3 * (c0 + k)] + cf[3 * (c0 + k) + 1];
                                    if (S.silu) y = silu_f(y);
                                    v[k] = y * cf[3 * (c0 + k) + 2];
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int k = 0; k < 8; ++k) act[(k * AH + r) * AW + c] = v[k];
                }
                if (want_sum) {
#pragma unroll
                    for (int k = 0; k < 8; ++k) {
                        double t = asum[k];
                        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
                        if (tx == 0 && k < cn) atomicAdd(p.act_sum + (size_t)n * Cs + c0 + k, t);
                    }
                }
            }
            if constexpr (WGRAD) {
                __syncthreads();
                // task = (tap, input channel of the chunk, group of 8 output channels, pixel split): 8 accumulators in
                // registers, one activation load + two broadcast 128-bit gradient loads per 8 FMAs
                constexpr int COG = COB / 8;
                constexpr int NTASK = 9 * CK * COG;
                constexpr int SPLIT = NTASK >= NTHREADS ? 1 : NTHREADS / NTASK;   // spare threads split the tile rows
                for (int task = tid; task < NTASK * SPLIT; task += NTHREADS) {
                    const int sp = task / NTASK;
                    const int t2 = task - sp * NTASK;
                    const int cg = t2 % COG;
                    const int ck = (t2 / COG) % CK;
                    const int tap = t2 / (COG * CK);
                    if (ck >= cn || co_cta + cg * 8 >= Cout) continue;
                    const float* a0 = act + (ck * AH + tap / 3) * AW + tap % 3;
                    const float* d0 = wsm + cg * 8;
                    float sum[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) sum[k] = 0.f;
                    for (int r = sp; r < TH; r += SPLIT)
#pragma unroll 4
                        for (int c = 0; c < TW; ++c) {
                            const float xv = a0[r * AW + c];
                            const float4 g0 = *reinterpret_cast<const float4*>(d0 + (r * TW + c) * COB);
                            const float4 g1 = *reinterpret_cast<const float4*>(d0 + (r * TW + c) * COB + 4);
                            sum[0] = fmaf(xv, g0.x, sum[0]); sum[1] = fmaf(xv, g0.y, sum[1]);
                            sum[2] = fmaf(xv, g0.z, sum[2]); sum[3] = fmaf(xv, g0.w, sum[3]);
                            sum[4] = fmaf(xv, g1.x, sum[4]); sum[5] = fmaf(xv, g1.y, sum[5]);
                            sum[6] = fmaf(xv, g1.z, sum[6]); sum[7] = fmaf(xv, g1.w, sum[7]);
                        }
                    float* dst = cfg.dW + (size_t)tap * cfg.s_tap + (size_t)(ci_base + c0 + ck) * cfg.s_ci;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (co_cta + cg * 8 + k < Cout) atomicAdd(dst + (size_t)(co_cta + cg * 8 + k) * cfg.s_co, sum[k]);
                }
                __syncthreads();
                continue;
            }
            // ---- (2) stage the weight chunk wsm[tap][ck][co] ---------------------------------
            for (int idx = tid; idx < 9 * CK * COB; idx += NTHREADS) {
                const int co = idx % COB;
                const int ck = (idx / COB) % CK;
                const int tap = idx / (COB * CK);
                float w = 0.f;
                if (ck < cn && co_cta + co < Cout)
                    w = __ldg(p.weight + ((size_t)tap * cin_total + ci_base + c0 + ck) * Cout + co_cta + co);
                wsm[idx] = w;
            }
            __syncthreads();
            // ---- (3) 4 rows x 8 output channels per thread ------------------------------------
            for (int ck = 0; ck < cn; ++ck) {
                float in[6][3];
#pragma unroll
                for (int r = 0; r < 6; ++r)
#pragma unroll
                    for (int k = 0; k < 3; ++k) in[r][k] = act[(ck * AH + 4 * ty + r) * AW + tx + k];
#pragma unroll
                for (int ky = 0; ky < 3; ++ky)
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const float4 w0 = *reinterpret_cast<const float4*>(wsm + ((ky * 3 + kx) * CK + ck) * COB + cog * 8);
                        const float4 w1 = *reinterpret_cast<const float4*>(wsm + ((ky * 3 + kx) * CK + ck) * COB + cog * 8 + 4);
#pragma unroll
                        for (int py = 0; py < 4; ++py) {
                            const float xv = in[py + ky][kx];
                            acc[py][0] = fmaf(xv, w0.x, acc[py][0]);
                            acc[py][1] = fmaf(xv, w0.y, acc[py][1]);
                            acc[py][2] = fmaf(xv, w0.z, acc[py][2]);
                            acc[py][3] = fmaf(xv, w0.w, acc[py][3]);
                            acc[py][4] = fmaf(xv, w1.x, acc[py][4]);
                            acc[py][5] = fmaf(xv, w1.y, acc[py][5]);
                            acc[py][6] = fmaf(xv, w1.z, acc[py][6]);
                            acc[py][7] = fmaf(xv, w1.w, acc[py][7]);
                        }
                    }
            }
            __syncthreads();
        }
        ci_base += Co_s;
        cf += 3 * Cs;
    }

    if constexpr (WGRAD) return;
    // ---- epilogue: store raw output (rounded to T) + GroupNorm statistics of the stored values
    const int co0 = co_cta + cog * 8;
    const int con = min(8, Cout - co0);  // may be <= 0 for padded channel groups
    T* out = reinterpret_cast<T*>(p.out);
    const bool vec_out = (Cout % 8 == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
    float s1[8], s2[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { s1[k] = 0.f; s2[k] = 0.f; }
    const int gx = x0 + tx;
#pragma unroll
    for (int py = 0; py < 4; ++py) {
        const int gy = y0 + 4 * ty + py;
        if (gy < H && gx < W && con > 0) {
            float v[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                v[k] = Store<T>::to_f(Store<T>::from_f(acc[py][k]));
                if (k < con) { s1[k] += v[k]; s2[k] += v[k] * v[k]; }
            }
            store8<T>(out + ((size_t)(n * H + gy) * W + gx) * Cout + co0, con, vec_out, v);
        }
    }
    if (p.out_stats != nullptr) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const float a = warp_sum(s1[k]);
            const float b = warp_sum(s2[k]);
            if (tx == 0 && k < con) {
                atomicAdd(&statsm[(cog * 8 + k) * 2], (double)a);
                atomicAdd(&statsm[(cog * 8 + k) * 2 + 1], (double)b);
            }
        }
        __syncthreads();
        if (tid < 2 * COB) {
            const int co = co_cta + (tid >> 1);
            if (co < Cout) atomicAdd(p.out_stats + ((size_t)n * Cout + co) * 2 + (tid & 1), statsm[tid]);
        }
    }
}

template <typename T, int NTY, int NCOG, bool WGRAD>
static int launch_cfg(const dg_conv3x3_args& a, cudaStream_t stream, const float* dR, float* dW, const int* strides) {
    constexpr int TH = 4 * NTY;
    constexpr int AH = TH + 2;
    constexpr int LH = TH / 2 + 2;
    constexpr int COB = 8 * NCOG;
    GenericCfg cfg{};
    int ncoef = 0;
    int low_c = 0;
    for (int s = 0; s < a.nsrc; ++s) {
        ncoef += 3 * a.src[s].channels;
        if (a.src[s].xform == DG_X_CONVT2) low_c = a.src[s].channels > low_c ? a.src[s].channels : low_c;
    }
    cfg.dR = dR;
    cfg.dW = dW;
    if (strides) { cfg.s_tap = strides[0]; cfg.s_ci = strides[1]; cfg.s_co = strides[2]; }
    const size_t wregion = WGRAD ? (size_t)TH * TW * COB : (size_t)9 * CK * COB;  // weight chunk or dR tile
    size_t floats = (size_t)(2 * COB) * 2 + (size_t)CK * AH * AW + wregion;
    cfg.coef_off = (int)floats;
    floats += ncoef;
    cfg.low_off = (int)floats;
    cfg.lch = 0;
    if (low_c > 0) {
        cfg.lch = low_c < 128 ? low_c : 128;
        floats += (size_t)LH * LW * (cfg.lch + 1);
    }
    cfg.cobatches = (a.cout + COB - 1) / COB;
    const size_t smem = floats * sizeof(float);
    if (smem > 200 * 1024) {
        set_error("conv3x3 generic: %zu bytes of shared memory needed (channels too large)", smem);
        return 3;
    }
    auto kern = conv3x3_generic_kernel<T, NTY, NCOG, WGRAD>;
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) {
            set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e));
            return 4;
        }
    }
    dim3 grid((a.W + TW - 1) / TW, (a.H + TH - 1) / TH, a.N * cfg.cobatches);
    if (grid.z > 65535u || grid.y > 65535u) {
        set_error("conv3x3 generic: grid too large (N*cobatches=%u)", grid.z);
        return 3;
    }
    kern<<<grid, NTHREADS, smem, stream>>>(a, cfg);
    count_launch();
    return check_launch("conv3x3_generic");
}

template <typename T, bool WGRAD>
static int launch_T(const dg_conv3x3_args& a, cudaStream_t stream, const float* dR, float* dW, const int* strides) {
    if (a.cout <= 8) return launch_cfg<T, 8, 1, WGRAD>(a, stream, dR, dW, strides);
    if (a.cout <= 16) return launch_cfg<T, 4, 2, WGRAD>(a, stream, dR, dW, strides);
    if (a.cout <= 32) return launch_cfg<T, 2, 4, WGRAD>(a, stream, dR, dW, strides);
    return launch_cfg<T, 1, 8, WGRAD>(a, stream, dR, dW, strides);
}

int conv3x3_generic_launch(const dg_conv3x3_args& a, cudaStream_t stream) {
    switch (a.dtype) {
        case DG_F32: return launch_T<float, false>(a, stream, nullptr, nullptr, nullptr);
        case DG_F16: return launch_T<__half, false>(a, stream, nullptr, nullptr, nullptr);
        case DG_BF16: return launch_T<__nv_bfloat16, false>(a, stream, nullptr, nullptr, nullptr);
        default: set_error("conv3x3: bad dtype %d", a.dtype); return 2;
    }
}

// dW += correlation of the activated input (rebuilt by the forward prologue from a.src) with dR; a.weight/a.out unused
int conv3x3_wgrad_launch(const dg_conv3x3_args& a, const float* dR, float* dW, int s_tap, int s_ci, int s_co,
                         cudaStream_t stream) {
    const int strides[3] = {s_tap, s_ci, s_co};
    switch (a.dtype) {
        case DG_F32: return launch_T<float, true>(a, stream, dR, dW, strides);
        case DG_F16: return launch_T<__half, true>(a, stream, dR, dW, strides);
        case DG_BF16: return launch_T<__nv_bfloat16, true>(a, stream, dR, dW, strides);
        default: set_error("conv3x3 wgrad: bad dtype %d", a.dtype); return 2;
    }
}

}  // namespace dg
