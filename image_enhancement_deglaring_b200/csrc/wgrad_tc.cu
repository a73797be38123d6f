// Weight gradient of the fused 3x3 convs on the tensor cores (16-bit storage tiers).
//
//   dW[co][ci][ky][kx] = sum over (n, y, x) of  A[n, y+ky-1, x+kx-1, ci] * dR[n, y, x, co]
// with A the ACTIVATED conv input (GroupNorm + SiLU (+ 2x2 average pool / channel concat) of the saved raw tensors,
// rebuilt on load exactly as the forward prologue does: src/model.py:92-99,107-128) and dR the gradient at the raw conv
// output (backward.cu).  Per tap this is a GEMM with M = ci, N = co and K = pixels -- the long dimension is K, so a CTA
// walks spatial tiles, keeps its [taps x ci x co] block of dW in mma.sync accumulators across all of them, and issues one
// fp32 atomicAdd per element at the very end.  Both operands are pixel-major in shared memory (the forward kernels'
// channel-plane layout: 16 bytes = 8 channels of one pixel), which is the TRANSPOSE of what the MMA wants for an
// M x K / K x N operand pair -- ldmatrix.trans delivers the fragments directly, with the 3x3 tap again a +16 B/pixel shift.
// Operands are bf16 whatever the storage type (dR ~ 1/numel underflows fp16; bf16 keeps fp32's exponent), accumulation
// fp32.  The generic CUDA-core WGRAD mode (conv3x3_generic.cu) stays the fp32-tier and any-shape path: 20.7 ms of a
// 39 ms training step at batch 32 before this kernel (torch profiler).
#include <type_traits>

#include "tc_common.cuh"

namespace dg {

namespace {

constexpr int WG_THREADS = 256;
enum { WG_SAME = 0, WG_POOL = 1, WG_CAT2 = 2 };

constexpr int wg_pad_plane(int pix, int nc8) {
    const int want = nc8 >= 8 ? 1 : (nc8 <= 1 ? 0 : 8 / nc8);
    if (nc8 <= 1) return pix;
    int p = pix;
    while (p % 8 != want) ++p;
    return p;
}

struct WgArgs {
    const void* src0; const double* st0; const float* g0; const float* b0; int groups0;   // SAME/POOL source, or `up` (CAT2)
    const void* src1; const double* st1; const float* g1; const float* b1; int groups1;   // CAT2: skip
    const float* dR; float* dW;
    const void* dRb;   // optional: dR already rounded to bf16 [N,H,W,CO] (gn_bwd_apply's second output form): copied, not converted
    int dry;           // probe only: report whether a kernel exists for this configuration, launch nothing
    int N, H, W;
    int s_tap, s_ci, s_co;
    float eps;
    int tiles_x, tiles_y;
};

__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t addr, uint32_t& r0, uint32_t& r1) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}

template <typename T>
__device__ __forceinline__ uint4 to_bf16x8(const uint4& q) {
    if constexpr (std::is_same<T, __nv_bfloat16>::value) {
        return q;
    } else {
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
        uint32_t o[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 v = unpack2<T>(w[k]);
            o[k] = pack2<__nv_bfloat16>(v.x, v.y);
        }
        return make_uint4(o[0], o[1], o[2], o[3]);
    }
}

// CI: input channels of the conv (both concat halves), CO: output channels.  A CTA owns the dW block of ALL nine taps x
// CIB input channels x (8 NTW) output channels: grid = (persistent CTAs, CI / CIB, CO / (8 NTW)).  Splitting over input
// channels (not taps) means the expensive operand -- the activated tile -- is staged exactly once per tile over the whole grid
// (a CTA stages only its CIB / 8 planes); only the cheap dR conversion repeats CI / CIB times.  Nine warps, one per tap, each
// with CIB / 16 m-tiles (a tap-split version re-activated the tile up to 9x and left dec4.0 at 595 us; this one: see DESIGN).
// CI == 8: an m-tile is a PAIR of taps (rows 0-7 / 8-15), five warps of eight work.
template <typename T, int CI, int CO, int MODE, int TH, int TW, int CIB, int NTW>
struct WgGeo {
    static constexpr bool PAIR = CI == 8;
    static constexpr int THREADS = PAIR ? 256 : 288;
    static constexpr int PH = TH + 2, PW = TW + 2, NC8 = CIB / 8;
    static constexpr int APLANE = wg_pad_plane(PH * PW, NC8);
    static constexpr int DPLANE = wg_pad_plane(TH * TW, NTW);
    static constexpr int IPW = PAIR ? 1 : CIB / 16;             // m-tiles per warp
    static constexpr int SEGS = TW / 16;
    static constexpr int A_BYTES = NC8 * APLANE * 16, D_BYTES = NTW * DPLANE * 16;
    static constexpr int NCOEF = MODE == WG_CAT2 ? CI / 2 : CI;
    static constexpr int SMEM = A_BYTES + D_BYTES + NCOEF * 8;
    // the narrow layers are staging-latency bound: make the register allocator leave room for 3 (288-thread) / 4 (256-thread)
    // resident CTAs -- dec1.0 sat at 84 registers = 2 CTAs/SM and ran 2x slower than its 8-channel neighbours
    static constexpr int MIN_CTAS = (IPW * NTW * 4 <= 16) ? (PAIR ? 4 : 3) : 2;
    static_assert(!PAIR || CIB == 8, "8 input channels: one block");
    static_assert(CI % CIB == 0 && (PAIR || CIB % 16 == 0) && CO % (8 * NTW) == 0 && TW % 16 == 0, "shape");
    static_assert(IPW * NTW * 4 <= 64, "accumulator budget");
    static_assert(NTW == 1 || NTW % 2 == 0, "n-tiles come in ldmatrix.x4 pairs");
    static_assert(THREADS % NC8 == 0 && THREADS % NTW == 0, "chunk ownership");
};

template <typename T, int CI, int CO, int MODE, int TH, int TW, int CIB, int NTW>
__global__ void __launch_bounds__(WgGeo<T, CI, CO, MODE, TH, TW, CIB, NTW>::THREADS, WgGeo<T, CI, CO, MODE, TH, TW, CIB, NTW>::MIN_CTAS)
wgrad_tc_kernel(const WgArgs p) {
    using G = WgGeo<T, CI, CO, MODE, TH, TW, CIB, NTW>;
    constexpr int WG_THREADS = G::THREADS;
    using BF = __nv_bfloat16;
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* act = smem;
    unsigned char* dsm = smem + G::A_BYTES;
    float2* coef = reinterpret_cast<float2*>(smem + G::A_BYTES + G::D_BYTES);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ci0 = blockIdx.y * CIB;            // first input channel of this CTA
    const int co0 = blockIdx.z * NTW * 8;        // first output channel of this CTA
    const int H = p.H, W = p.W;
    const int tiles_per_img = p.tiles_x * p.tiles_y;
    const int ntiles = tiles_per_img * p.N;

    float acc[G::IPW][NTW][4];
#pragma unroll
    for (int s = 0; s < G::IPW; ++s)
#pragma unroll
        for (int j = 0; j < NTW; ++j) acc[s][j][0] = acc[s][j][1] = acc[s][j][2] = acc[s][j][3] = 0.f;

    const uint32_t act_u = smem_u32(act), dsm_u = smem_u32(dsm);
    int cur_n = -1;
#pragma unroll 1
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int n = tile / tiles_per_img;
        const int tr = tile - n * tiles_per_img;
        const int y0 = (tr / p.tiles_x) * TH, x0 = (tr % p.tiles_x) * TW;
        __syncthreads();  // everyone is done reading the previous tile (and the previous image's coefficients)
        if (n != cur_n) {
            cur_n = n;
            // GroupNorm affine (a, b) per activated source channel, pre-halved for silu(y) = h + h tanh(h)
            // only the channels this CTA stages: its CIB-channel block (CAT2: the part of the block that lies in the skip half).
            // Each coefficient sums a whole group's statistics in double: all CI of them per image per CTA was ~260 k loads at 1024 channels
            constexpr int CHALF = MODE == WG_CAT2 ? CI / 2 : 0;
            const int c_lo = ci0 - CHALF > 0 ? ci0 - CHALF : 0, c_hi = ci0 + CIB - CHALF;
            for (int c = c_lo + tid; c < c_hi; c += WG_THREADS) {
                float a, b;
                if constexpr (MODE == WG_CAT2) {
                    gn_coef(p.st1, p.g1, p.b1, n, CI / 2, p.groups1, c, (double)H * W, p.eps, a, b);
                } else {
                    const double plane = MODE == WG_POOL ? (double)(2 * H) * (2 * W) : (double)H * W;
                    gn_coef(p.st0, p.g0, p.b0, n, CI, p.groups0, c, plane, p.eps, a, b);
                }
                coef[c] = make_float2(0.5f * a, 0.5f * b);
            }
            __syncthreads();
        }
        // ---- stage the activated haloed input tile as bf16 channel planes ------------------------------------------
        {
            constexpr int NPIX = G::PH * G::PW;
            const int c8 = tid % G::NC8;              // plane of this CTA's block
            const int c8g = ci0 / 8 + c8;              // 8-channel chunk of the conv input
            constexpr bool HAS_IDENT = MODE == WG_CAT2;
            const bool ident = HAS_IDENT && c8g < CI / 16;          // CAT2: chunks [0, CI/16) = materialised `up`, copied
            constexpr int CS = MODE == WG_CAT2 ? CI / 2 : CI;       // channels of the tensor a chunk is read from
            const int cc8 = (MODE == WG_CAT2 && !ident) ? c8g - CI / 16 : c8g;
            float2 cf[8];
            if (!ident) {
#pragma unroll
                for (int k = 0; k < 8; ++k) cf[k] = coef[cc8 * 8 + k];
            }
            const unsigned char* base;
            if constexpr (MODE == WG_CAT2) base = reinterpret_cast<const unsigned char*>(ident ? p.src0 : p.src1) + (size_t)n * H * W * CS * 2;
            else if constexpr (MODE == WG_POOL) base = reinterpret_cast<const unsigned char*>(p.src0) + (size_t)n * H * W * CS * 8;
            else base = reinterpret_cast<const unsigned char*>(p.src0) + (size_t)n * H * W * CS * 2;
            base += cc8 * 16;
            unsigned char* dst = act + (size_t)c8 * G::APLANE * 16;
            // (explicitly batching 4 loads per thread here and in the dR loop was measured: the persistent accumulators stay
            // live across the staging, registers went to 128-168 (or 64-360 B of spills under a launch bound) and the wgrad
            // total rose from 2.57 to 2.76 ms.  The cure for the long-scoreboard stalls ncu shows on the narrow layers
            // (profiles/r01_ncu_wgrad.txt) is not more registers.  A cp.async version -- every 16-byte piece of both raw tiles in
            // flight at once, the 16-bit input activated in place in its plane slot -- was ALSO measured and is no faster
            // (2.37 vs 2.34 ms): these kernels execute ~5.5 warp-instructions per pixel, 2.5 of them in the K loop, where each
            // of the five tap-pair warps re-loads the B fragment for every 16 pixels to feed ONE small MMA.  Splitting K (rows)
            // across warps so that every warp sweeps all taps per B load (shared-memory reduction at the end) was measured
            // too: 2.42 vs 2.34 ms -- more accumulators per warp, spills under the launch bound.  Left as is.)
#pragma unroll 4
            for (int pix = tid / G::NC8; pix < NPIX; pix += WG_THREADS / G::NC8) {
                const int r = pix / G::PW, c = pix - r * G::PW;
                const int gy = y0 + r - 1, gx = x0 + c - 1;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if ((unsigned)gy < (unsigned)H && (unsigned)gx < (unsigned)W) {
                    if constexpr (MODE == WG_POOL) {
                        const size_t rowb = (size_t)(2 * W) * CS * 2;
                        const unsigned char* q0 = base + (size_t)(2 * gy) * rowb + (size_t)(2 * gx) * CS * 2;
                        float y[8], t[8];
                        act8<T>(__ldg(reinterpret_cast<const uint4*>(q0)), cf, y);
                        act8<T>(__ldg(reinterpret_cast<const uint4*>(q0 + CS * 2)), cf, t);
#pragma unroll
                        for (int k = 0; k < 8; ++k) y[k] += t[k];
                        act8<T>(__ldg(reinterpret_cast<const uint4*>(q0 + rowb)), cf, t);
#pragma unroll
                        for (int k = 0; k < 8; ++k) y[k] += t[k];
                        act8<T>(__ldg(reinterpret_cast<const uint4*>(q0 + rowb + CS * 2)), cf, t);
#pragma unroll
                        for (int k = 0; k < 8; ++k) y[k] = 0.25f * (y[k] + t[k]);
                        o = pack8<BF>(y);
                    } else {
                        const uint4 q = __ldg(reinterpret_cast<const uint4*>(base + ((size_t)gy * W + gx) * CS * 2));
                        if (ident) {
                            o = to_bf16x8<T>(q);
                        } else {
                            float y[8];
                            act8<T>(q, cf, y);
                            o = pack8<BF>(y);
                        }
                    }
                }
                *reinterpret_cast<uint4*>(dst + (size_t)pix * 16) = o;
            }
        }
        // ---- stage dR (fp32 NHWC) for this CTA's output channels as bf16 planes, zero outside the image -------------
        {
            const int j8 = tid % NTW;
            const float* gsrc = p.dR + (size_t)n * H * W * CO + co0 + j8 * 8;
            const unsigned char* bsrc = reinterpret_cast<const unsigned char*>(p.dRb) + ((size_t)n * H * W * CO + co0 + j8 * 8) * 2;
            unsigned char* dst = dsm + (size_t)j8 * G::DPLANE * 16;
#pragma unroll 4
            for (int pix = tid / NTW; pix < TH * TW; pix += WG_THREADS / NTW) {
                const int r = pix / TW, c = pix - r * TW;
                const int gy = y0 + r, gx = x0 + c;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (p.dRb != nullptr) {
                    if (gy < H && gx < W) o = __ldg(reinterpret_cast<const uint4*>(bsrc + ((size_t)gy * W + gx) * CO * 2));
                } else if (gy < H && gx < W) {
                    const float4 a = __ldg(reinterpret_cast<const float4*>(gsrc + ((size_t)gy * W + gx) * CO));
                    const float4 b = __ldg(reinterpret_cast<const float4*>(gsrc + ((size_t)gy * W + gx) * CO) + 1);
                    o = make_uint4(pack2<BF>(a.x, a.y), pack2<BF>(a.z, a.w), pack2<BF>(b.x, b.y), pack2<BF>(b.z, b.w));
                }
                *reinterpret_cast<uint4*>(dst + (size_t)pix * 16) = o;
            }
        }
        __syncthreads();
        // ---- K loop over the tile's 16-pixel row segments ----------------------------------------------------------
        // A matrices of a lane: (plane lo, px 0-7), (plane hi, px 0-7), (plane lo, px 8-15), (plane hi, px 8-15); "plane hi"
        // is the second TAP of the pair when CI == 8.  B: (plane j, px 0-7), (plane j, px 8-15), (plane j+1, ...), ...
        const bool active = G::PAIR ? warp < 5 : true;
        if (active) {
            uint32_t a_lane;
            if constexpr (G::PAIR) {
                const int t_lo = 2 * warp, t_hi = (2 * warp + 1 < 9) ? 2 * warp + 1 : 2 * warp;
                const int t = ((lane >> 3) & 1) ? t_hi : t_lo;
                a_lane = (uint32_t)((((t / 3) * G::PW + (t % 3)) + (lane & 7) + 8 * (lane >> 4)) * 16);
            } else {
                const int tap = warp;
                a_lane = (uint32_t)(((((lane >> 3) & 1) * G::APLANE) + (tap / 3) * G::PW + (tap % 3) + (lane & 7) + 8 * (lane >> 4)) * 16);
            }
            const uint32_t b_lane = NTW == 1 ? (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * 16)
                                             : (uint32_t)((((lane >> 4) * G::DPLANE) + (lane & 7) + 8 * ((lane >> 3) & 1)) * 16);
#pragma unroll 1
            for (int r = 0; r < TH; ++r) {
#pragma unroll
                for (int sg = 0; sg < G::SEGS; ++sg) {
                    uint32_t bf[NTW][2];
                    const uint32_t boff = dsm_u + b_lane + (uint32_t)((r * TW + sg * 16) * 16);
                    if constexpr (NTW == 1) {
                        ldsm_x2_t(boff, bf[0][0], bf[0][1]);
                    } else {
#pragma unroll
                        for (int jp = 0; jp < NTW / 2; ++jp)
                            ldsm_x4_t(boff + (uint32_t)(2 * jp * G::DPLANE * 16), bf[2 * jp][0], bf[2 * jp][1], bf[2 * jp + 1][0],
                                      bf[2 * jp + 1][1]);
                    }
#pragma unroll
                    for (int s = 0; s < G::IPW; ++s) {
                        uint32_t a0, a1, a2, a3;
                        ldsm_x4_t(act_u + a_lane + (uint32_t)((2 * s * G::APLANE + r * G::PW + sg * 16) * 16), a0, a1, a2, a3);
#pragma unroll
                        for (int j = 0; j < NTW; ++j) mma16816<BF>(acc[s][j], a0, a1, a2, a3, bf[j][0], bf[j][1]);
                    }
                }
            }
        }
    }
    // ---- one atomicAdd per element of this CTA's dW block ---------------------------------------------------------------
    const int g = lane >> 2, q = lane & 3;
    if (G::PAIR && warp >= 5) return;
#pragma unroll
    for (int s = 0; s < G::IPW; ++s) {
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {   // accumulator rows g and g + 8
            int tap, ci;
            if constexpr (G::PAIR) {
                tap = 2 * warp + hf;
                ci = g;
                if (tap > 8) continue;
            } else {
                tap = warp;
                ci = ci0 + s * 16 + g + 8 * hf;
            }
#pragma unroll
            for (int j = 0; j < NTW; ++j) {
                const int co = co0 + j * 8 + 2 * q;
                float* d = p.dW + (size_t)tap * p.s_tap + (size_t)ci * p.s_ci;
                atomicAdd(d + (size_t)co * p.s_co, acc[s][j][2 * hf]);
                atomicAdd(d + (size_t)(co + 1) * p.s_co, acc[s][j][2 * hf + 1]);
            }
        }
    }
}

template <typename T, int CI, int CO, int MODE, int TH, int TW, int CIB, int NTW>
int launch_wg(WgArgs a, cudaStream_t st) {
    using G = WgGeo<T, CI, CO, MODE, TH, TW, CIB, NTW>;
    auto kern = wgrad_tc_kernel<T, CI, CO, MODE, TH, TW, CIB, NTW>;
    static bool done = false;
    if (!done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM);
        if (e != cudaSuccess) { set_error("wgrad_tc: cudaFuncSetAttribute(%d B): %s", G::SMEM, cudaGetErrorString(e)); return 4; }
        done = true;
    }
    if (a.dry) return 0;
    a.tiles_x = (a.W + TW - 1) / TW;
    a.tiles_y = (a.H + TH - 1) / TH;
    const int ntiles = a.tiles_x * a.tiles_y * a.N;
    constexpr int GY = CI / CIB, GZ = CO / (8 * NTW);
    // persistent CTAs: two per SM over all channel blocks.  Every CTA ends with one atomicAdd per element of its dW block, so
    // CTAs must walk several tiles each: with one tile per CTA the 64-channel layers spent most of their time in 19 M atomics
    // (measured: 64->64 189 -> 103 us, 128->128 218 -> 94 us).  The narrow layers are staging-latency bound and their dW
    // blocks are tiny, so they keep two waves of four CTAs per SM (two per SM cost them 221 -> 269 us).
    constexpr int FIT = (227 * 1024) / (G::SMEM + 1024);
    constexpr bool SMALL = 9 * CIB * NTW * 8 <= 2304;
    constexpr int RES = SMALL ? (FIT > 4 ? 8 : 2 * FIT) : (FIT >= 2 ? 2 : 1);
    int gx = (148 * RES + GY * GZ - 1) / (GY * GZ);
    if (gx > ntiles) gx = ntiles;
    if (gx < 1) gx = 1;
    kern<<<dim3(gx, GY, GZ), G::THREADS, G::SMEM, st>>>(a);
    count_launch();
    return check_launch("wgrad_tc");
}

template <typename T>
int dispatch_wg(const WgArgs& a, int ci, int co, int mode, cudaStream_t st, bool* handled) {
    *handled = true;
#define DG_WG(CI_, CO_, MODE_, TH_, TW_, CIB_, NTW_) \
    if (ci == CI_ && co == CO_ && mode == MODE_) return launch_wg<T, CI_, CO_, MODE_, TH_, TW_, CIB_, NTW_>(a, st);
    DG_WG(8, 8, WG_SAME, 16, 64, 8, 1)        // enc1.3, dec1.3
    DG_WG(8, 16, WG_POOL, 16, 64, 8, 2)       // enc2.0
    DG_WG(16, 16, WG_SAME, 16, 64, 16, 2)     // enc2.3, dec2.3
    DG_WG(16, 32, WG_POOL, 16, 32, 16, 4)     // enc3.0
    DG_WG(32, 32, WG_SAME, 16, 32, 32, 4)     // enc3.3, dec3.3
    DG_WG(32, 64, WG_POOL, 8, 32, 32, 8)      // enc4.0
    DG_WG(64, 64, WG_SAME, 8, 32, 32, 8)      // enc4.3, dec4.3
    DG_WG(64, 128, WG_POOL, 8, 32, 16, 16)    // bottleneck.0 (pooled staging is the expensive side: never repeat it)
    DG_WG(128, 128, WG_SAME, 8, 32, 32, 8)    // bottleneck.3
    DG_WG(128, 64, WG_CAT2, 8, 32, 32, 8)     // dec4.0
    DG_WG(64, 32, WG_CAT2, 8, 32, 32, 4)      // dec3.0
    DG_WG(32, 16, WG_CAT2, 16, 32, 16, 2)     // dec2.0
    DG_WG(16, 8, WG_CAT2, 16, 64, 16, 1)      // dec1.0
    // wider variants (features_start = 16 / 32 / 64, BASELINE.json configs[4]): same CTA block (32 input x 64 output channels, all
    // nine taps) as the 128-channel layers -- shared memory and registers depend on the block, not on CI / CO; the grid just gets
    // more (ci-block, co-block) columns and each persistent CTA walks all tiles of its column
    DG_WG(128, 256, WG_POOL, 8, 32, 16, 16)
    DG_WG(256, 256, WG_SAME, 8, 32, 32, 8)
    DG_WG(256, 512, WG_POOL, 8, 32, 16, 16)
    DG_WG(512, 512, WG_SAME, 8, 32, 32, 8)
    DG_WG(512, 1024, WG_POOL, 8, 32, 16, 16)
    DG_WG(1024, 1024, WG_SAME, 8, 32, 32, 8)
    DG_WG(256, 128, WG_CAT2, 8, 32, 32, 8)
    DG_WG(512, 256, WG_CAT2, 8, 32, 32, 8)
    DG_WG(1024, 512, WG_CAT2, 8, 32, 32, 8)
#undef DG_WG
    *handled = false;
    return 0;
}


// ---- ConvTranspose2d(k=2, s=2) weight gradient (src/model.py:47-53 backward) -------------------------------------------
//   dWt[ci][co][a][b] = sum over (n, i, j) of  A_low[n, i, j, ci] * dUp[n, 2i+a, 2j+b, co]
// the same GEMM shape (M = ci, N = co, K = low pixels) once per kernel position (a, b): the "tap" is now the position, the A
// tile needs no halo and the B tile of a position gathers every second pixel of the concat gradient's up half.
struct CtWgArgs {
    const void* raw_low; const double* stats; const float* gamma; const float* beta; int groups;
    const float* dCat; int stride;   // [N, 2Hl, 2Wl, stride], up half = channels 0..CU
    float* dWt;                      // [CL][CU][2][2], accumulated atomically
    float* dBias;                    // optional [CU]: sum of the up-half gradient over every pixel (ConvTranspose bias gradient)
    int N, Hl, Wl; float eps;
    int tiles_x, tiles_y;
};

// A CTA owns the dWt block of CLB input x CUB output channels x POSG positions: grid = (persistent CTAs, 4 / POSG, (CL / CLB) * (CU / CUB)).
// The shipped widths use one block (CLB = CL, CUB = CU); the wider variants (configs[4]: 256 -> 128 ... 1024 -> 512) tile the
// proven 128 x 64 block over grid.z -- shared memory and accumulators depend on the block only.
template <typename T, int CL, int CU, int CLB, int CUB, int TH, int TW, int POSG>
__global__ void __launch_bounds__(WG_THREADS) convt_wgrad_tc_kernel(const CtWgArgs p) {
    using BF = __nv_bfloat16;
    constexpr int NC8 = CLB / 8, NTW = CUB / 8, MT = CLB / 16, ITEMS = POSG * MT, IPW = (ITEMS + 7) / 8, SEGS = TW / 16;
    static_assert(CL % CLB == 0 && CU % CUB == 0, "channel blocks");
    constexpr int APLANE = wg_pad_plane(TH * TW, NC8), DPLANE = wg_pad_plane(TH * TW, NTW);
    constexpr int A_BYTES = NC8 * APLANE * 16, D_BYTES = POSG * NTW * DPLANE * 16;
    static_assert(IPW * NTW * 4 <= 64 && (NTW == 1 || NTW % 2 == 0) && TW % 16 == 0, "shape");
    static_assert(WG_THREADS % NC8 == 0 && WG_THREADS % NTW == 0, "chunk ownership");
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* act = smem;
    unsigned char* dsm = smem + A_BYTES;
    float2* coef = reinterpret_cast<float2*>(smem + A_BYTES + D_BYTES);
    float* bias_sm = reinterpret_cast<float*>(coef + CLB);   // [CUB]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int pos0 = blockIdx.y * POSG;
    const int ci0 = (blockIdx.z % (CL / CLB)) * CLB, co0 = (blockIdx.z / (CL / CLB)) * CUB;   // this CTA's channel block
    float bsum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};   // bias gradient partials of this thread's 8 output channels
    for (int c = tid; c < CUB; c += WG_THREADS) bias_sm[c] = 0.f;
    const int Hl = p.Hl, Wl = p.Wl, H = 2 * Hl, W = 2 * Wl;
    const int tiles_per_img = p.tiles_x * p.tiles_y, ntiles = tiles_per_img * p.N;
    float acc[IPW][NTW][4];
#pragma unroll
    for (int s = 0; s < IPW; ++s)
#pragma unroll
        for (int j = 0; j < NTW; ++j) acc[s][j][0] = acc[s][j][1] = acc[s][j][2] = acc[s][j][3] = 0.f;
    const uint32_t act_u = smem_u32(act), dsm_u = smem_u32(dsm);
    int cur_n = -1;
#pragma unroll 1
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int n = tile / tiles_per_img;
        const int tr = tile - n * tiles_per_img;
        const int y0 = (tr / p.tiles_x) * TH, x0 = (tr % p.tiles_x) * TW;   // low-resolution tile origin
        __syncthreads();
        if (n != cur_n) {
            cur_n = n;
            for (int c = tid; c < CLB; c += WG_THREADS) {
                float a, b;
                gn_coef(p.stats, p.gamma, p.beta, n, CL, p.groups, ci0 + c, (double)Hl * Wl, p.eps, a, b);
                coef[c] = make_float2(0.5f * a, 0.5f * b);
            }
            __syncthreads();
        }
        {   // activated low tile
            const int c8 = tid % NC8;
            float2 cf[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) cf[k] = coef[c8 * 8 + k];
            const unsigned char* base = reinterpret_cast<const unsigned char*>(p.raw_low) + (size_t)n * Hl * Wl * CL * 2 + (ci0 / 8 + c8) * 16;
            unsigned char* dst = act + (size_t)c8 * APLANE * 16;
            for (int pix = tid / NC8; pix < TH * TW; pix += WG_THREADS / NC8) {
                const int r = pix / TW, c = pix - r * TW;
                const int gy = y0 + r, gx = x0 + c;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (gy < Hl && gx < Wl) {
                    float y[8];
                    act8<T>(__ldg(reinterpret_cast<const uint4*>(base + ((size_t)gy * Wl + gx) * CL * 2)), cf, y);
                    o = pack8<BF>(y);
                }
                *reinterpret_cast<uint4*>(dst + (size_t)pix * 16) = o;
            }
        }
        {   // gradient of the up half, one plane set per kernel position
            const int j8 = tid % NTW;
            const float* gsrc = p.dCat + (size_t)n * H * W * p.stride + co0 + j8 * 8;
            for (int it = tid / NTW; it < POSG * TH * TW; it += WG_THREADS / NTW) {
                const int ps = it / (TH * TW), pix = it - ps * (TH * TW);
                const int pos = pos0 + ps;
                const int r = pix / TW, c = pix - r * TW;
                const int gy = y0 + r, gx = x0 + c;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (gy < Hl && gx < Wl) {
                    const float* q = gsrc + ((size_t)(2 * gy + (pos >> 1)) * W + 2 * gx + (pos & 1)) * p.stride;
                    const float4 a = __ldg(reinterpret_cast<const float4*>(q));
                    const float4 b = __ldg(reinterpret_cast<const float4*>(q) + 1);
                    o = make_uint4(pack2<BF>(a.x, a.y), pack2<BF>(a.z, a.w), pack2<BF>(b.x, b.y), pack2<BF>(b.z, b.w));
                    // every up-half gradient element passes through here exactly once over the whole grid
                    bsum[0] += a.x; bsum[1] += a.y; bsum[2] += a.z; bsum[3] += a.w;
                    bsum[4] += b.x; bsum[5] += b.y; bsum[6] += b.z; bsum[7] += b.w;
                }
                *reinterpret_cast<uint4*>(dsm + ((size_t)(ps * NTW + j8) * DPLANE + pix) * 16) = o;
            }
        }
        __syncthreads();
#pragma unroll
        for (int s = 0; s < IPW; ++s) {
            const int item = warp + 8 * s;
            if (item >= ITEMS) continue;
            const int ps = item / MT, mt = item % MT;
            const uint32_t a_lane = (uint32_t)((((2 * mt + ((lane >> 3) & 1)) * APLANE) + (lane & 7) + 8 * (lane >> 4)) * 16);
            const uint32_t b_lane = (NTW == 1 ? (uint32_t)(((lane & 7) + 8 * ((lane >> 3) & 1)) * 16)
                                              : (uint32_t)((((lane >> 4) * DPLANE) + (lane & 7) + 8 * ((lane >> 3) & 1)) * 16)) +
                                    (uint32_t)(ps * NTW * DPLANE * 16);
#pragma unroll 2
            for (int k16 = 0; k16 < TH * SEGS; ++k16) {
                uint32_t a0, a1, a2, a3;
                ldsm_x4_t(act_u + a_lane + (uint32_t)(k16 * 256), a0, a1, a2, a3);
                const uint32_t boff = dsm_u + b_lane + (uint32_t)(k16 * 256);
                if constexpr (NTW == 1) {
                    uint32_t b0, b1;
                    ldsm_x2_t(boff, b0, b1);
                    mma16816<BF>(acc[s][0], a0, a1, a2, a3, b0, b1);
                } else {
#pragma unroll
                    for (int jp = 0; jp < NTW / 2; ++jp) {
                        uint32_t b0, b1, b2, b3;
                        ldsm_x4_t(boff + (uint32_t)(2 * jp * DPLANE * 16), b0, b1, b2, b3);
                        mma16816<BF>(acc[s][2 * jp], a0, a1, a2, a3, b0, b1);
                        mma16816<BF>(acc[s][2 * jp + 1], a0, a1, a2, a3, b2, b3);
                    }
                }
            }
        }
    }
    if (p.dBias != nullptr && ci0 == 0) {   // every up-half gradient element is staged once per input-channel block: count it once
        const int j8 = tid % NTW;
#pragma unroll
        for (int k = 0; k < 8; ++k) atomicAdd(&bias_sm[j8 * 8 + k], bsum[k]);
        __syncthreads();
        for (int c = tid; c < CUB; c += WG_THREADS) atomicAdd(p.dBias + co0 + c, bias_sm[c]);
    }
    const int g = lane >> 2, q = lane & 3;
#pragma unroll
    for (int s = 0; s < IPW; ++s) {
        const int item = warp + 8 * s;
        if (item >= ITEMS) continue;
        const int pos = pos0 + item / MT, mt = item % MT;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
            const int ci = ci0 + mt * 16 + g + 8 * hf;
#pragma unroll
            for (int j = 0; j < NTW; ++j) {
                const int co = co0 + j * 8 + 2 * q;
                atomicAdd(p.dWt + ((size_t)ci * CU + co) * 4 + pos, acc[s][j][2 * hf]);
                atomicAdd(p.dWt + ((size_t)ci * CU + co + 1) * 4 + pos, acc[s][j][2 * hf + 1]);
            }
        }
    }
}

template <typename T, int CL, int CU, int POSG, int CLB = CL, int CUB = CU>
int launch_ctwg(CtWgArgs a, cudaStream_t st) {
    constexpr int TH = 8, TW = 32;
    constexpr int NC8 = CLB / 8, NTW = CUB / 8;
    constexpr int SMEM = NC8 * wg_pad_plane(TH * TW, NC8) * 16 + POSG * NTW * wg_pad_plane(TH * TW, NTW) * 16 + CLB * 8 + CUB * 4;
    auto kern = convt_wgrad_tc_kernel<T, CL, CU, CLB, CUB, TH, TW, POSG>;
    static bool done = false;
    if (!done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM);
        if (e != cudaSuccess) { set_error("convt_wgrad_tc: cudaFuncSetAttribute(%d B): %s", SMEM, cudaGetErrorString(e)); return 4; }
        done = true;
    }
    a.tiles_x = (a.Wl + TW - 1) / TW;
    a.tiles_y = (a.Hl + TH - 1) / TH;
    const int ntiles = a.tiles_x * a.tiles_y * a.N;
    constexpr int GY = 4 / POSG, GZ = (CL / CLB) * (CU / CUB);
    constexpr int RES = (227 * 1024) / (SMEM + 1024) >= 2 ? 2 : 1;
    int gx = (148 * RES + GY * GZ - 1) / (GY * GZ);
    if (gx > ntiles) gx = ntiles;
    if (gx < 1) gx = 1;
    kern<<<dim3(gx, GY, GZ), WG_THREADS, SMEM, st>>>(a);
    count_launch();
    return check_launch("convt_wgrad_tc");
}

template <typename T>
int dispatch_ctwg(const CtWgArgs& a, int cl, int cu, cudaStream_t st, bool* handled) {
    *handled = true;
    if (cl == 128 && cu == 64) return launch_ctwg<T, 128, 64, 1>(a, st);
    if (cl == 64 && cu == 32) return launch_ctwg<T, 64, 32, 4>(a, st);
    if (cl == 32 && cu == 16) return launch_ctwg<T, 32, 16, 4>(a, st);
    if (cl == 16 && cu == 8) return launch_ctwg<T, 16, 8, 4>(a, st);
    if (cl == 256 && cu == 128) return launch_ctwg<T, 256, 128, 1, 128, 64>(a, st);     // wider variants: 128 x 64 blocks over grid.z
    if (cl == 512 && cu == 256) return launch_ctwg<T, 512, 256, 1, 128, 64>(a, st);
    if (cl == 1024 && cu == 512) return launch_ctwg<T, 1024, 512, 1, 128, 64>(a, st);
    *handled = false;
    return 0;
}

}  // namespace

// dBias [Cu] (optional) += sum of the up half over all pixels, folded into the gradient staging.
// dWt [Cl][Cu][2][2] += correlation of the activated low-resolution producer with the up half (channels 0..Cu of a
// [N,H,W,stride] fp32 tensor) of the concat gradient.  16-bit storage, LightweightUNet(features_start=8) channel pairs.
int convt_wgrad_tc_launch(int dtype, const float* dCat, int stride, const void* raw_low, const double* stats, const float* gamma,
                          const float* beta, float* dWt, float* dBias, int N, int H, int W, int Cl, int Cu, int groups, float eps,
                          cudaStream_t st, bool* handled) {
    *handled = false;
    if (dtype != DG_F16 && dtype != DG_BF16) return 0;
    if ((reinterpret_cast<uintptr_t>(dCat) & 15) || (stride & 3) || (reinterpret_cast<uintptr_t>(raw_low) & 15) || ((H | W) & 1)) return 0;
    CtWgArgs a{raw_low, stats, gamma, beta, groups, dCat, stride, dWt, dBias, N, H / 2, W / 2, eps, 0, 0};
    if (dtype == DG_F16) return dispatch_ctwg<__half>(a, Cl, Cu, st, handled);
    return dispatch_ctwg<__nv_bfloat16>(a, Cl, Cu, st, handled);
}

namespace {
}  // namespace

// Sources as dg_conv3x3_fused describes them, except that a ConvTranspose source must already be MATERIALISED: src[0] =
// identity 16-bit NHWC `up` (stats == NULL, silu == 0), src[1] = the skip.  dW element (tap, ci, co) lives at
// dW[tap*s_tap + ci*s_ci + co*s_co] and is accumulated atomically (zero it first).
int conv3x3_wgrad_tc_launch(const dg_conv3x3_args& a, const float* dR, float* dW, int s_tap, int s_ci, int s_co,
                            cudaStream_t st, bool* handled, const void* dR_bf16, bool dry) {
    *handled = false;
    if (a.dtype != DG_F16 && a.dtype != DG_BF16) return 0;
    if (a.N < 1 || (reinterpret_cast<uintptr_t>(dR) & 15)) return 0;
    WgArgs w;
    memset(&w, 0, sizeof(w));
    int mode, ci;
    const dg_src& s0 = a.src[0];
    if (a.nsrc == 1) {
        if (s0.stats == nullptr || !s0.silu || s0.scale || s0.coef) return 0;
        if (s0.xform == DG_X_SAME) mode = WG_SAME;
        else if (s0.xform == DG_X_POOL2) mode = WG_POOL;
        else return 0;
        ci = s0.channels;
        w.src0 = s0.raw; w.st0 = s0.stats; w.g0 = s0.gamma; w.b0 = s0.beta; w.groups0 = s0.groups;
        if (reinterpret_cast<uintptr_t>(s0.raw) & 15) return 0;
    } else if (a.nsrc == 2) {
        const dg_src& s1 = a.src[1];
        if (s0.xform != DG_X_SAME || s0.stats != nullptr || s0.silu || s0.scale) return 0;   // materialised up
        if (s1.xform != DG_X_SAME || s1.stats == nullptr || !s1.silu || s1.scale || s1.coef) return 0;
        if (s0.channels != s1.channels) return 0;
        mode = WG_CAT2;
        ci = 2 * s0.channels;
        w.src0 = s0.raw;
        w.src1 = s1.raw; w.st1 = s1.stats; w.g1 = s1.gamma; w.b1 = s1.beta; w.groups1 = s1.groups;
        if ((reinterpret_cast<uintptr_t>(s0.raw) | reinterpret_cast<uintptr_t>(s1.raw)) & 15) return 0;
    } else {
        return 0;
    }
    if (dR_bf16 != nullptr && (reinterpret_cast<uintptr_t>(dR_bf16) & 15)) return 0;
    w.dR = dR; w.dW = dW; w.dRb = dR_bf16; w.dry = dry ? 1 : 0; w.N = a.N; w.H = a.H; w.W = a.W;
    w.s_tap = s_tap; w.s_ci = s_ci; w.s_co = s_co; w.eps = a.eps;
    if (a.dtype == DG_F16) return dispatch_wg<__half>(w, ci, a.cout, mode, st, handled);
    return dispatch_wg<__nv_bfloat16>(w, ci, a.cout, mode, st, handled);
}

}  // namespace dg
