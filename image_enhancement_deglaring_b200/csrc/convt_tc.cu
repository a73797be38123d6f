// ConvTranspose2d(CL -> CU, k=2, s=2) + bias on the tensor cores, with the producer's GroupNorm + SiLU applied on load
// (src/model.py:47-53 applied to the activated output of the previous block).  Used for the DEEP decoder levels
// (upconv4, upconv3): there the fused variant inside conv3x3_tc (M_UPCAT) drags 16-65 KB of ConvTranspose weights and a
// serial scatter phase into every conv CTA (1 CTA/SM, 23-30 % tensor-pipe utilisation, profile r1c), while the `up` tensor
// is tiny (<= 1 MB per image), so materialising it costs ~1.5 % extra HBM traffic and frees the conv kernel.
//
//   up[n, 2i+a, 2j+b, co] = bias[co] + sum_ci SiLU(GN(low))[n,i,j,ci] * Wt[ci][co][a][b]
// as a GEMM [low pixels x CL] x [CL x 4*CU]: one CTA = 128 low pixels (one 16-pixel m-tile per warp), A fragments of all
// K chunks stay in registers across the n-tile groups, B tiles come from the packed weights (dg_pack_convt2x2_tc).
#include "tc_common.cuh"

namespace dg {

namespace {
constexpr int CT_THREADS = 256;
constexpr int CT_MP = 128;  // low pixels per CTA

constexpr int ct_pad_plane(int pix, int nc8) {
    const int want = nc8 >= 8 ? 1 : (nc8 <= 1 ? 0 : 8 / nc8);
    if (nc8 <= 1) return pix;
    int p = pix;
    while (p % 8 != want) ++p;
    return p;
}

struct ConvtArgs {
    const void* low; const double* stats; const float* gamma; const float* beta; const float* coef; int groups;
    const void* ctw; const float* ctb; void* out;
    int N, h, w; float eps;  // h, w: LOW resolution
};

template <typename T, int CL, int CU>
__global__ void __launch_bounds__(CT_THREADS) convt_tc_kernel(const ConvtArgs p) {
    constexpr int NCL8 = CL / 8, LPLANE = ct_pad_plane(CT_MP, NCL8);
    constexpr int CHUNKS = CL / 16, CT_N = 4 * CU, CT_NT = CT_N / 8, NTG = CT_NT < 8 ? CT_NT : 8;
    static_assert(CT_NT % NTG == 0, "n-tile groups");
    constexpr int LOW_BYTES = NCL8 * LPLANE * 16, CTW_BYTES = CHUNKS * 2 * CT_N * 16;
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* low = smem;
    unsigned char* ctw = smem + LOW_BYTES;
    float2* coef = reinterpret_cast<float2*>(ctw + CTW_BYTES);
    float* bias = reinterpret_cast<float*>(coef + CL);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int n = blockIdx.y;
    const int hw = p.h * p.w;
    const int p_base = blockIdx.x * CT_MP;

    {
        const unsigned char* src = reinterpret_cast<const unsigned char*>(p.ctw);
        const uint32_t dst = smem_u32(ctw);
        for (int i = tid * 16; i < CTW_BYTES; i += CT_THREADS * 16) cp_async16(dst + i, src + i);
        cp_async_commit();
    }
    pdl_launch_dependents();
    pdl_wait();
    for (int c = tid; c < CL; c += CT_THREADS) {
        float a, b;
        if (p.coef) { a = __ldg(p.coef + (size_t)(n * CL + c) * 2); b = __ldg(p.coef + (size_t)(n * CL + c) * 2 + 1); }
        else gn_coef(p.stats, p.gamma, p.beta, n, CL, p.groups, c, (double)hw, p.eps, a, b);
        a *= 0.5f; b *= 0.5f;
        coef[c] = make_float2(a, b);
    }
    for (int c = tid; c < CU; c += CT_THREADS) bias[c] = p.ctb[c];
    __syncthreads();

    // ---- stage the activated low pixels as channel planes ---------------------------------------------------
    {
        const T* raw = reinterpret_cast<const T*>(p.low) + (size_t)n * hw * CL;
        const int c8 = tid % NCL8;
        float2 cf[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) cf[k] = coef[c8 * 8 + k];
#pragma unroll 4
        for (int idx = tid; idx < CT_MP * NCL8; idx += CT_THREADS) {
            const int lp = idx / NCL8;
            uint4 o = make_uint4(0u, 0u, 0u, 0u);
            if (p_base + lp < hw) {
                float y[8];
                const uint4 q = __ldg(reinterpret_cast<const uint4*>(raw + (size_t)(p_base + lp) * CL + c8 * 8));
                act8<T>(q, cf, y);
                o = pack8<T>(y);
            }
            *reinterpret_cast<uint4*>(low + ((size_t)c8 * LPLANE + lp) * 16) = o;
        }
    }
    cp_async_wait<0>();
    __syncthreads();

    // ---- GEMM: this warp's 16 low pixels x all 4*CU outputs -------------------------------------------------------
    const uint32_t low_u = smem_u32(low), ctw_u = smem_u32(ctw);
    uint32_t af[CHUNKS][4];
#pragma unroll
    for (int ch = 0; ch < CHUNKS; ++ch)
        ldsm_x4(low_u + (uint32_t)(((2 * ch + (lane >> 4)) * LPLANE + warp * 16 + (lane & 15)) * 16), af[ch][0], af[ch][1],
                af[ch][2], af[ch][3]);
    T* outp = reinterpret_cast<T*>(p.out);
    const int W2 = 2 * p.w;
    // the two accumulator rows of this lane: low pixels P0, P0 + 8
    size_t obase[2];
    bool live[2];
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
        const int P = p_base + warp * 16 + (lane >> 2) + 8 * hf;
        live[hf] = P < hw;
        const int i = P / p.w, j = P - i * p.w;
        obase[hf] = ((size_t)(n * 2 * p.h + 2 * i) * W2 + 2 * j) * CU;
    }
#pragma unroll 1
    for (int ng = 0; ng < CT_NT; ng += NTG) {
        float acc[NTG][4];
#pragma unroll
        for (int i = 0; i < NTG; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
#pragma unroll
        for (int ch = 0; ch < CHUNKS; ++ch) {
#pragma unroll
            for (int np = 0; np < NTG / 2; ++np) {
                uint32_t b0, b1, b2, b3;
                const int nrow = (ng + 2 * np + (lane >> 4)) * 8 + (lane & 7);
                ldsm_x4(ctw_u + (uint32_t)(((ch * 2 + ((lane >> 3) & 1)) * CT_N + nrow) * 16), b0, b1, b2, b3);
                mma16816<T>(acc[2 * np], af[ch][0], af[ch][1], af[ch][2], af[ch][3], b0, b1);
                mma16816<T>(acc[2 * np + 1], af[ch][0], af[ch][1], af[ch][2], af[ch][3], b2, b3);
            }
        }
#pragma unroll
        for (int i = 0; i < NTG; ++i) {
            const int nn = (ng + i) * 8 + 2 * (lane & 3);
            const int pos = nn / CU, co = nn % CU;
            const float bias0 = bias[co], bias1 = bias[co + 1];
            const size_t poff = ((size_t)(pos >> 1) * W2 + (pos & 1)) * CU + co;
#pragma unroll
            for (int hf = 0; hf < 2; ++hf)
                if (live[hf])
                    *reinterpret_cast<uint32_t*>(outp + obase[hf] + poff) = pack2<T>(acc[i][2 * hf] + bias0, acc[i][2 * hf + 1] + bias1);
        }
    }
}

template <typename T, int CL, int CU>
int launch_convt(const ConvtArgs& a, cudaStream_t st) {
    constexpr int NCL8 = CL / 8, LPLANE = ct_pad_plane(CT_MP, NCL8);
    constexpr int SMEM = NCL8 * LPLANE * 16 + (CL / 16) * 2 * 4 * CU * 16 + CL * 8 + CU * 4;
    auto kern = convt_tc_kernel<T, CL, CU>;
    static bool done = false;
    if (!done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%d B): %s", SMEM, cudaGetErrorString(e)); return 4; }
        done = true;
    }
    dim3 grid((a.h * a.w + CT_MP - 1) / CT_MP, a.N);
    cudaError_t le = launch_kernel(kern, grid, dim3(CT_THREADS), (size_t)SMEM, st, a);
    if (le != cudaSuccess) { set_error("convt_tc launch: %s", cudaGetErrorString(le)); return 10; }
    count_launch();
    return check_launch("convt_tc");
}

template <typename T>
int dispatch_convt(const ConvtArgs& a, int cl, int cu, cudaStream_t st, bool* handled) {
    *handled = true;
    if (cl == 128 && cu == 64) return launch_convt<T, 128, 64>(a, st);   // upconv4
    if (cl == 64 && cu == 32) return launch_convt<T, 64, 32>(a, st);     // upconv3
    if (cl == 32 && cu == 16) return launch_convt<T, 32, 16>(a, st);     // upconv2
    if (cl == 16 && cu == 8) return launch_convt<T, 16, 8>(a, st);       // upconv1 (training: wgrad of dec1.0 reads `up`)
    *handled = false;
    return 0;
}
}  // namespace

// out: NHWC [N, 2h, 2w, cu] in `dtype`; src describes the LOW-resolution producer (raw + statistics / affine)
int convt_tc_launch(const dg_src& s, int dtype, int N, int H, int W, void* out, float eps, int path, cudaStream_t st,
                    bool* handled) {
    *handled = false;
    if (dtype != DG_F16 && dtype != DG_BF16) return 0;
    // Channel sets the mma.sync kernel below does not cover (the wide variant's 1024 -> 512 ... 128 -> 64) go to the tcgen05 kernel;
    // on the shipped model's upconv4 / upconv3 the mma.sync kernel measured faster (0.043 / 0.055 vs 0.059 / 0.067 ms at batch 64).
    const bool hmma_covers = (s.channels == 128 && s.ct_cout == 64) || (s.channels == 64 && s.ct_cout == 32) ||
                             (s.channels == 32 && s.ct_cout == 16) || (s.channels == 16 && s.ct_cout == 8);
    if (!hmma_covers || (path & 256)) {
        int rc = convt_t5_launch(s, dtype, N, H, W, out, eps, path, st, handled);
        if (rc || *handled) return rc;
    }
    if (s.xform != DG_X_CONVT2 || s.ct_w_tc == nullptr || s.ct_b == nullptr || s.stats == nullptr || !s.silu || s.scale) return 0;
    if ((H | W) & 1) return 0;
    if ((reinterpret_cast<uintptr_t>(s.raw) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(s.ct_w_tc)) & 15) return 0;
    if (N > 65535) return 0;
    ConvtArgs a{s.raw, s.stats, s.gamma, s.beta, s.coef, s.groups, s.ct_w_tc, s.ct_b, out, N, H / 2, W / 2, eps};
    if (dtype == DG_F16) return dispatch_convt<__half>(a, s.channels, s.ct_cout, st, handled);
    return dispatch_convt<__nv_bfloat16>(a, s.channels, s.ct_cout, st, handled);
}

}  // namespace dg
