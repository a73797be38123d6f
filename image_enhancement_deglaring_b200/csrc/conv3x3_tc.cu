// Tensor-core implicit-GEMM path of dg_conv3x3_fused for 16-bit storage (fp16 / bf16, fp32 accumulate).
//
// One CTA (8 warps) computes a TH x TW output tile of one image for all COUT channels:
//   1. weights (pre-packed B tiles) stream into shared memory with cp.async (resident, or one tap per
//      stage, double buffered, for the deep layers);
//   2. the haloed input tile is staged ONCE into shared memory as 16-bit "channel planes"
//      [CIN/8][(TH+2)*(TW+2)][8] after the consumer-side prologue -- GroupNorm apply + SiLU, and either
//      identity, 2x2 average pool, or (MODE_UPCAT) ConvTranspose2d(2,2)+bias of the activated low-res tile
//      computed on the tensor cores and scattered next to the activated skip tile (torch.cat never exists);
//   3. the 3x3 conv is 9 shifted GEMMs over that tile: A fragments come straight from the planes with
//      ldmatrix (a tap shift is a +16 B/pixel address offset, so no im2col copy), B fragments from the
//      packed weights, mma.sync.m16n8k16 accumulates in fp32 registers;
//   4. the epilogue rounds to the storage type, stores NHWC, and reduces the GroupNorm statistics of the
//      stored values (warp shuffles -> shared atomics -> one double atomic per channel per CTA).
//
// Why mma.sync and not tcgen05 here: for COUT = 8..32 the UMMA A operand (128 pixels x 16 k) must be re-read
// from shared memory for every 8..32 output channels, which is shared-memory-bandwidth bound at ~1/8..1/2 of
// the tensor rate; HMMA keeps A in registers across n-tiles and the measured rate (tools/mma_bench.cu:
// 557 TFLOP/s dense, 990 MAC/clk/SM) is enough to sit under the HBM time of the level-1/2 layers.
//
// Reference semantics: src/model.py:92-99, :35-41, :47-53, :116-128 (see conv3x3_generic.cu).
#include "tc_common.cuh"

namespace dg {

// M_CAT2: torch.cat((up, skip)) where `up` is an already materialised ConvTranspose output (identity source, planes
// [0, C/8)) and `skip` is activated on load -- used for the deep decoder levels, where running the transposed conv as its own
// small GEMM kernel (convt_tc_kernel) beats fusing it (profile r1c: 1 CTA/SM, 65 KB of ConvTranspose weights per CTA).
enum { M_SAME = 0, M_POOL = 1, M_UPCAT = 2, M_CAT2 = 3 };
constexpr int TC_THREADS = 256;

struct TcArgs {
    const void* src0; const double* st0; const float* g0; const float* b0; int groups0;
    const void* src1; const double* st1; const float* g1; const float* b1; int groups1;
    const void* wgt; const void* ctw; const float* ctb;
    void* out; double* out_stats;
    int N, H, W; float eps;
    const float* cf0; const float* cf1;   // optional finished (a, b) of src0 / src1 ([N,C,2]), else computed from st0 / st1
};

// ---- compile-time geometry -------------------------------------------------------------------------
constexpr int pad_plane(int pix, int nc8) {
    // plane stride (in 16-byte pixels) chosen so that the nc8 planes written by one quarter-warp of a
    // pixel-major staging pass land in distinct banks: stride == 8/nc8 (mod 8), or 1 (mod 8) for nc8 >= 8
    const int want = nc8 >= 8 ? 1 : (nc8 <= 1 ? 0 : 8 / nc8);
    if (nc8 <= 1) return pix;
    int p = pix;
    while (p % 8 != want) ++p;
    return p;
}

template <int CIN_, int COUT_, int MODE_, int TH_, int TW_, int WM_, int WN_, bool STREAM_>
struct Geo {
    static constexpr int CIN = CIN_, COUT = COUT_, MODE = MODE_, TH = TH_, TW = TW_, WM = WM_, WN = WN_;
    static constexpr bool STREAM = STREAM_;
    static constexpr int THREADS = 32 * WM * WN;
    // ROLL: the narrow layers are bound by the shared-memory data pipe (profile r1c: l1tex LSU wavefronts at ~70 % of peak,
    // ~3/4 of them the ldmatrix re-reads of the same pixels for the 9 taps).  There a warp owns a COLUMN of consecutive
    // output rows of one 16-pixel segment, loads each (input row, kx) fragment once and feeds it to the three output rows
    // that use it (ky = 0, 1, 2); the weights live in registers.  ldmatrix traffic drops from 9 to ~3.75 reads per pixel.
    static constexpr int RW = TH_ / (WM_ / (TW_ / 16) > 0 ? WM_ / (TW_ / 16) : 1);  // rows per warp in ROLL mode
    static constexpr bool ROLL = !STREAM_ && CIN_ <= 16 && (WM_ % (TW_ / 16)) == 0 && RW * (COUT_ / 8 / WN_) * 4 <= 32;
    static constexpr int PH = TH + 2, PW = TW + 2, NC8 = CIN / 8;
    static constexpr int PLANE = pad_plane(PH * PW, NC8);
    static constexpr int KC = CIN >= 16 ? CIN / 16 : 1;
    static constexpr int NCHUNK = CIN == 8 ? 5 : 9 * KC;
    static constexpr int SEGS = TW / 16, MTILES = TH * SEGS, MPW = MTILES / WM, NT = COUT / 8 / WN;
    // accumulator budget per thread: 32 registers when the weights are resident -- those kernels are latency-bound on the
    // CUDA-core prologue / epilogue, so more resident CTAs beat B-fragment reuse (measured ~10 % on levels 3-4); 64 when the
    // taps stream (a second m-tile group would stream them again: measured 8-15 % slower on the 128-channel layers).
    static constexpr int ACC_REGS = STREAM ? 64 : 32;
    static constexpr int MG = (MPW * NT * 4 <= ACC_REGS) ? MPW : (ACC_REGS / (NT * 4));
    static constexpr int STAGE_CHUNKS = STREAM ? KC : NCHUNK;
    static constexpr int NSTAGE = STREAM ? 9 : 1;
    // MODE_UPCAT: ConvTranspose2d(CIN -> COUT) of the half-res tile, skip has COUT channels
    static constexpr int CU = COUT, CL = CIN, NCL8 = CL / 8;
    static constexpr int LPH = TH / 2 + 2, LPW = TW / 2 + 2, LM = LPH * LPW;
    static constexpr int LPLANE = pad_plane(LM, NCL8);
    static constexpr int LMT = (LM + 15) / 16;
    static constexpr int CT_CHUNKS = CL / 16, CT_N = 4 * CU, CT_NT = CT_N / 8, CT_NTG = CT_NT < 8 ? CT_NT : 8;
    static constexpr int NCOEF = MODE == M_UPCAT ? (CL + CU) : (MODE == M_CAT2 ? COUT : CIN);
    // shared memory carve-up (bytes)
    static constexpr int ACT_BYTES = NC8 * PLANE * 16;
    static constexpr int WGT_BYTES = (STREAM ? 2 : 1) * STAGE_CHUNKS * COUT * 32;
    static constexpr int COEF_BYTES = NCOEF * 8;
    static constexpr int STAT_BYTES = WM * COUT * 2 * 4;  // one float (sum, sumsq) slot per (m-warp, channel)
    static constexpr int LOW_BYTES = MODE == M_UPCAT ? NCL8 * LPLANE * 16 : 0;
    static constexpr int CTW_BYTES = MODE == M_UPCAT ? CT_CHUNKS * 2 * CT_N * 16 : 0;
    static constexpr int CTB_BYTES = MODE == M_UPCAT ? (CU * 4 + ((LM + 15) / 16) * 16) : 0;  // bias + scatter mask table
    static constexpr int OFF_ACT = 0;
    static constexpr int OFF_WGT = OFF_ACT + ACT_BYTES;
    static constexpr int OFF_LOW = OFF_WGT + WGT_BYTES;
    static constexpr int OFF_CTW = OFF_LOW + LOW_BYTES;
    static constexpr int OFF_COEF = OFF_CTW + CTW_BYTES;
    static constexpr int OFF_STAT = OFF_COEF + COEF_BYTES;
    static constexpr int OFF_CTB = OFF_STAT + STAT_BYTES;
    static constexpr int SMEM_BYTES = OFF_CTB + CTB_BYTES;
    // Resident CTAs per SM the register allocator must leave room for (__launch_bounds__): the narrow memory-bound layers
    // live on inter-CTA overlap of their staging / MMA phases (4 CTAs = 64 registers; a 74-register build ran 12 % slower),
    // the compute-heavy ones need ~100 registers for 64 accumulators.
    static constexpr int CTA_TARGET = ((MG * NT * 4 <= 32) ? ((MODE == M_POOL || (ROLL && CIN == 16 && NT == 2)) ? 3 : 4) : 2) * (256 / THREADS);
    static constexpr int CTA_SMEM = (227 * 1024) / (SMEM_BYTES + 1024);
    static constexpr int MIN_CTAS = CTA_SMEM < 1 ? 1 : (CTA_SMEM < CTA_TARGET ? CTA_SMEM : CTA_TARGET);
    static_assert(WM * WN == 8 || WM * WN == 4, "4 or 8 warps");
    static_assert(MTILES % WM == 0 && (COUT / 8) % WN == 0, "tile split");
    static_assert(MPW % MG == 0, "m-tile groups");
    static_assert(!STREAM || CIN >= 16, "streamed weights: one tap per stage");
    static_assert(NT == 1 || NT % 2 == 0, "n-tiles come in ldmatrix.x4 pairs");
    static_assert((MODE != M_UPCAT && MODE != M_CAT2) || CIN == 2 * COUT, "UPCAT/CAT2: (up C, skip C) -> C");
    static_assert(CIN % 8 == 0 && COUT % 8 == 0 && TW % 16 == 0 && TH % 2 == 0, "shape");
};

// Stage a same-resolution (or 2x2-average-pooled) activated source into planes [plane0, plane0 + C/8).
// Items are (pixel, 8-channel chunk), pixel-major so a warp's global loads are contiguous; 256 % (C/8) == 0, so a
// thread always owns the same chunk and keeps its coefficients in registers.  The item slots of a thread are split into
// ITERS batches of BATCH; all loads of a batch are issued before any math, the slot count is matched to the tile, the
// (row, column) of a slot advances incrementally, and tiles whose halo lies inside the image skip every bounds test
// (profiles r1b/r1c: addressing was ~1/3 of the instructions).  `src` points at image n; offsets are 32-bit.
// SYNC_FIRST: the GroupNorm coefficients `cfs` are still being written by other threads when this is called; the CTA barrier
// that publishes them is taken here, AFTER the first batch of global loads has been issued, so the coefficient chain
// (statistics load -> double math -> shared memory) and the first tile loads overlap instead of running back to back.
template <typename T, typename G, int C, bool POOL, bool IDENT = false, bool SYNC_FIRST = false>
__device__ __forceinline__ void stage_planes(unsigned char* act, const unsigned char* __restrict__ src,
                                             const float2* __restrict__ cfs, int plane0, int y0, int x0, int H, int W) {
    constexpr int NC = C / 8;
    constexpr int NPIX = G::PH * G::PW;
    constexpr int PSTRIDE = G::THREADS / NC;                       // pixels between two slots of a thread
    constexpr int NSLOT = (NPIX + PSTRIDE - 1) / PSTRIDE;
    constexpr int MAXB = POOL ? 2 : 5;
    constexpr int ITERS = (NSLOT + MAXB - 1) / MAXB;
    constexpr int BATCH = (NSLOT + ITERS - 1) / ITERS;
    constexpr int DR = PSTRIDE / G::PW, DC = PSTRIDE % G::PW;      // slot-to-slot advance of (row, column)
    static_assert(G::THREADS % NC == 0, "chunk ownership");
    const int c8 = threadIdx.x % NC;
    const int p0 = threadIdx.x / NC;
    float2 cf[8];
    auto read_coefs = [&]() {
#pragma unroll
        for (int k = 0; k < 8; ++k) cf[k] = cfs[c8 * 8 + k];
    };
    if constexpr (!SYNC_FIRST && !IDENT) read_coefs();
    unsigned char* dst = act + (size_t)(plane0 + c8) * G::PLANE * 16;
    const uint32_t rowb = (uint32_t)(POOL ? 2 * W : W) * C * 2;    // source row pitch in bytes
    const unsigned char* srcc = src + c8 * 16;
    const bool interior = y0 >= 1 && x0 >= 1 && y0 + G::TH + 1 <= H && x0 + G::TW + 1 <= W;

    auto run = [&](auto interior_c) {
        constexpr bool INTERIOR = decltype(interior_c)::value;
        int r = p0 / G::PW, c = p0 - (p0 / G::PW) * G::PW;
        int pix = p0;
#pragma unroll 1
        for (int it = 0; it < ITERS; ++it) {
            uint4 q[BATCH][POOL ? 4 : 1];
            int pixs[BATCH];
            bool ok[BATCH];
#pragma unroll
            for (int b = 0; b < BATCH; ++b) {
                const int gy = y0 + r - 1, gx = x0 + c - 1;
                pixs[b] = pix;
                ok[b] = pix < NPIX && (INTERIOR || ((unsigned)gy < (unsigned)H && (unsigned)gx < (unsigned)W));
                if (ok[b]) {
                    if constexpr (POOL) {
                        const unsigned char* base = srcc + ((uint32_t)(2 * gy) * rowb + (uint32_t)(2 * gx) * (C * 2));
                        q[b][0] = __ldg(reinterpret_cast<const uint4*>(base));
                        q[b][1] = __ldg(reinterpret_cast<const uint4*>(base + C * 2));
                        q[b][2] = __ldg(reinterpret_cast<const uint4*>(base + rowb));
                        q[b][3] = __ldg(reinterpret_cast<const uint4*>(base + rowb + C * 2));
                    } else {
                        q[b][0] = __ldg(reinterpret_cast<const uint4*>(srcc + ((uint32_t)gy * rowb + (uint32_t)gx * (C * 2))));
                    }
                }
                pix += PSTRIDE;
                r += DR;
                c += DC;
                if (c >= G::PW) { c -= G::PW; r += 1; }
            }
            if constexpr (SYNC_FIRST) {
                if (it == 0) {
                    __syncthreads();   // coefficients published (uniform: every thread runs the same ITERS)
                    read_coefs();
                }
            }
#pragma unroll
            for (int b = 0; b < BATCH; ++b) {
                if (pixs[b] >= NPIX) continue;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (ok[b]) {
                    if constexpr (IDENT) {
                        o = q[b][0];  // already-final values (materialised ConvTranspose output): plain copy
                    } else {
                        float y[8];
                        act8<T>(q[b][0], cf, y);
                        if constexpr (POOL) {
                            float t[8];
#pragma unroll
                            for (int j = 1; j < 4; ++j) {
                                act8<T>(q[b][j], cf, t);
#pragma unroll
                                for (int k = 0; k < 8; ++k) y[k] += t[k];
                            }
#pragma unroll
                            for (int k = 0; k < 8; ++k) y[k] *= 0.25f;
                        }
                        o = pack8<T>(y);
                    }
                }
                *reinterpret_cast<uint4*>(dst + (uint32_t)pixs[b] * 16) = o;
            }
        }
    };
    if (interior) run(std::true_type{});
    else run(std::false_type{});
}

template <typename T, typename G>
__global__ void __launch_bounds__(G::THREADS, G::MIN_CTAS) conv3x3_tc_kernel(const TcArgs p) {
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char* act = smem + G::OFF_ACT;
    unsigned char* wgt = smem + G::OFF_WGT;
    float2* coef = reinterpret_cast<float2*>(smem + G::OFF_COEF);
    float* statf = reinterpret_cast<float*>(smem + G::OFF_STAT);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int wm = warp % G::WM, wn = warp / G::WM;
    const int n = blockIdx.z;
    const int y0 = blockIdx.y * G::TH, x0 = blockIdx.x * G::TW;
    const int H = p.H, W = p.W;

    pdl_launch_dependents();
    // ---- (0) start the weight traffic ----------------------------------------------------------------
    auto load_stage = [&](int stage, int buf) {
        constexpr int BYTES = G::STAGE_CHUNKS * G::COUT * 32;
        const unsigned char* src = reinterpret_cast<const unsigned char*>(p.wgt) + (size_t)stage * BYTES;
        const uint32_t dst = smem_u32(wgt) + buf * BYTES;
        for (int i = tid * 16; i < BYTES; i += G::THREADS * 16) cp_async16(dst + i, src + i);
    };
    load_stage(0, 0);
    if constexpr (G::MODE == M_UPCAT) {
        const unsigned char* src = reinterpret_cast<const unsigned char*>(p.ctw);
        const uint32_t dst = smem_u32(smem + G::OFF_CTW);
        for (int i = tid * 16; i < G::CTW_BYTES; i += G::THREADS * 16) cp_async16(dst + i, src + i);
    }
    cp_async_commit();

    pdl_wait();  // everything above overlapped the producer's tail; its activations / statistics are complete from here on
    // ---- (1) GroupNorm coefficients (a, b) per source channel ---------------------------------------
    if constexpr (G::MODE == M_UPCAT) {
        for (int c = tid; c < G::CL + G::CU; c += G::THREADS) {
            float a, b;
            if (c < G::CL) {
                if (p.cf0) { a = __ldg(p.cf0 + (size_t)(n * G::CL + c) * 2); b = __ldg(p.cf0 + (size_t)(n * G::CL + c) * 2 + 1); }
                else gn_coef(p.st0, p.g0, p.b0, n, G::CL, p.groups0, c, (double)(H / 2) * (W / 2), p.eps, a, b);
            } else {
                const int cc = c - G::CL;
                if (p.cf1) { a = __ldg(p.cf1 + (size_t)(n * G::CU + cc) * 2); b = __ldg(p.cf1 + (size_t)(n * G::CU + cc) * 2 + 1); }
                else gn_coef(p.st1, p.g1, p.b1, n, G::CU, p.groups1, cc, (double)H * W, p.eps, a, b);
            }
            a *= 0.5f; b *= 0.5f;  // silu(y) = h + h*tanh(h), h = y/2
            coef[c] = make_float2(a, b);
        }
        float* ctb = reinterpret_cast<float*>(smem + G::OFF_CTB);
        for (int c = tid; c < G::CU; c += G::THREADS) ctb[c] = p.ctb[c];
        // scatter mask of every low pixel (li, lj): it feeds the 2x2 block at tile (2li-1+a, 2lj-1+b); bit (2a+b) = that
        // position lies inside the staged tile, bit 4+(2a+b) = it also lies inside the image (else the concat is zero there)
        unsigned char* okt = smem + G::OFF_CTB + G::CU * 4;
        for (int lp = tid; lp < G::LM; lp += G::THREADS) {
            const int li = lp / G::LPW, lj = lp - li * G::LPW;
            const int r0 = 2 * li - 1, c0 = 2 * lj - 1;
            uint32_t m = 0;
#pragma unroll
            for (int ab = 0; ab < 4; ++ab) {
                const int r = r0 + (ab >> 1), c = c0 + (ab & 1);
                const bool in_tile = (unsigned)r < (unsigned)G::PH && (unsigned)c < (unsigned)G::PW;
                const bool in_img = (unsigned)(y0 - 1 + r) < (unsigned)H && (unsigned)(x0 - 1 + c) < (unsigned)W;
                m |= (in_tile ? 1u : 0u) << ab;
                m |= ((in_tile && in_img) ? 1u : 0u) << (4 + ab);
            }
            okt[lp] = (unsigned char)m;
        }
    } else if constexpr (G::MODE == M_CAT2) {
        for (int c = tid; c < G::COUT; c += G::THREADS) {
            float a, b;
            if (p.cf1) { a = __ldg(p.cf1 + (size_t)(n * G::COUT + c) * 2); b = __ldg(p.cf1 + (size_t)(n * G::COUT + c) * 2 + 1); }
            else gn_coef(p.st1, p.g1, p.b1, n, G::COUT, p.groups1, c, (double)H * W, p.eps, a, b);
            a *= 0.5f; b *= 0.5f;
            coef[c] = make_float2(a, b);
        }
    } else {
        const double plane = G::MODE == M_POOL ? (double)(2 * H) * (2 * W) : (double)H * W;
        for (int c = tid; c < G::CIN; c += G::THREADS) {
            float a, b;
            if (p.cf0) { a = __ldg(p.cf0 + (size_t)(n * G::CIN + c) * 2); b = __ldg(p.cf0 + (size_t)(n * G::CIN + c) * 2 + 1); }
            else gn_coef(p.st0, p.g0, p.b0, n, G::CIN, p.groups0, c, plane, p.eps, a, b);
            a *= 0.5f; b *= 0.5f;
            coef[c] = make_float2(a, b);
        }
    }
    // the barrier that publishes the coefficients is taken inside the first stage_planes call that needs them (SYNC_FIRST)

    // ---- (2) stage the activated halo tile ------------------------------------------------------------
    if constexpr (G::MODE == M_SAME) {
        stage_planes<T, G, G::CIN, false, false, true>(act, reinterpret_cast<const unsigned char*>(p.src0) + (size_t)n * H * W * G::CIN * 2,
                                                             coef, 0, y0, x0, H, W);
    } else if constexpr (G::MODE == M_CAT2) {
        stage_planes<T, G, G::COUT, false, true>(act, reinterpret_cast<const unsigned char*>(p.src0) + (size_t)n * H * W * G::COUT * 2,
                                                      coef, 0, y0, x0, H, W);
        stage_planes<T, G, G::COUT, false, false, true>(act, reinterpret_cast<const unsigned char*>(p.src1) + (size_t)n * H * W * G::COUT * 2,
                                                              coef, G::COUT / 8, y0, x0, H, W);
    } else if constexpr (G::MODE == M_POOL) {
        stage_planes<T, G, G::CIN, true, false, true>(act, reinterpret_cast<const unsigned char*>(p.src0) + (size_t)n * H * W * G::CIN * 8,
                                                            coef, 0, y0, x0, H, W);
    } else {
        // skip -> planes [CU/8, 2CU/8)
        stage_planes<T, G, G::CU, false, false, true>(act, reinterpret_cast<const unsigned char*>(p.src1) + (size_t)n * H * W * G::CU * 2,
                                                            coef + G::CL, G::CU / 8, y0, x0, H, W);
        // activated low-res tile -> low planes
        unsigned char* low = smem + G::OFF_LOW;
        const T* raw = reinterpret_cast<const T*>(p.src0);
        const int Hl = H / 2, Wl = W / 2;
        const int li0 = (y0 >> 1) - 1, lj0 = (x0 >> 1) - 1;
        {
            static_assert(G::THREADS % G::NCL8 == 0, "chunk ownership");
            const int c8 = tid % G::NCL8;
            float2 cf[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) cf[k] = coef[c8 * 8 + k];
            constexpr int LITEMS = G::LM * G::NCL8;
            constexpr int LSLOTS = (LITEMS + G::THREADS - 1) / G::THREADS;
            constexpr int LB = LSLOTS < 4 ? LSLOTS : 4;  // loads in flight per thread
            const unsigned char* rawn = reinterpret_cast<const unsigned char*>(raw) + (size_t)n * Hl * Wl * G::CL * 2 + c8 * 16;
#pragma unroll 1
            for (int idx0 = tid; idx0 < LITEMS; idx0 += G::THREADS * LB) {
                uint4 q[LB];
                bool ok[LB];
#pragma unroll
                for (int b = 0; b < LB; ++b) {
                    const int lp = (idx0 + b * G::THREADS) / G::NCL8;
                    const int li = lp / G::LPW;
                    const int gi = li0 + li, gj = lj0 + lp - li * G::LPW;
                    ok[b] = lp < G::LM && (unsigned)gi < (unsigned)Hl && (unsigned)gj < (unsigned)Wl;
                    if (ok[b]) q[b] = __ldg(reinterpret_cast<const uint4*>(rawn + (uint32_t)(gi * Wl + gj) * (G::CL * 2)));
                }
#pragma unroll
                for (int b = 0; b < LB; ++b) {
                    const int lp = (idx0 + b * G::THREADS) / G::NCL8;
                    if (lp >= G::LM) continue;
                    uint4 o = make_uint4(0u, 0u, 0u, 0u);
                    if (ok[b]) {
                        float y[8];
                        act8<T>(q[b], cf, y);
                        o = pack8<T>(y);
                    }
                    *reinterpret_cast<uint4*>(low + ((size_t)c8 * G::LPLANE + lp) * 16) = o;
                }
            }
        }
        cp_async_wait<0>();  // ConvTranspose weights (and conv stage 0) have landed
        __syncthreads();
        // ---- (2b) ConvTranspose2d(2,2) on the tensor cores: [low pixels x CL] x [CL x 4*CU] -------------
        const uint32_t low_u = smem_u32(low);
        const uint32_t ctw_u = smem_u32(smem + G::OFF_CTW);
        const float* ctb = reinterpret_cast<const float*>(smem + G::OFF_CTB);
        constexpr int NG = G::CT_NT / G::CT_NTG;  // work item = (16 low pixels, CT_NTG n-tiles), round-robin over warps
#pragma unroll 1
        for (int item = warp; item < G::LMT * NG; item += G::WM * G::WN) {
            const int mt = item / NG;
            const int ng = (item % NG) * G::CT_NTG;
            int lp_lane = mt * 16 + (lane & 15);
            if (lp_lane > G::LM - 1) lp_lane = G::LM - 1;
            {
                float acc[G::CT_NTG][4];
#pragma unroll
                for (int i = 0; i < G::CT_NTG; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
#pragma unroll
                for (int ch = 0; ch < G::CT_CHUNKS; ++ch) {
                    uint32_t a0, a1, a2, a3;
                    ldsm_x4(low_u + (uint32_t)(((2 * ch + (lane >> 4)) * G::LPLANE + lp_lane) * 16), a0, a1, a2, a3);
#pragma unroll
                    for (int np = 0; np < G::CT_NTG / 2; ++np) {
                        uint32_t b0, b1, b2, b3;
                        const int nrow = (ng + 2 * np + (lane >> 4)) * 8 + (lane & 7);
                        ldsm_x4(ctw_u + (uint32_t)(((ch * 2 + ((lane >> 3) & 1)) * G::CT_N + nrow) * 16), b0, b1, b2, b3);
                        mma16816<T>(acc[2 * np], a0, a1, a2, a3, b0, b1);
                        mma16816<T>(acc[2 * np + 1], a0, a1, a2, a3, b2, b3);
                    }
                }
                // scatter (+bias) into the up planes [0, CU/8); outside the image the concat is zero-padded.
                // (Measured and rejected: re-mapping the m-tiles so that the interior TH/2 x TW/2 low pixels form mask-free
                // m-tiles and the border ring is handled separately -- .319 -> .330 ms on up1+dec1.0: the ring's strided
                // ldmatrix rows and the index arithmetic cost more than the mask tests save.)
                // Geometry of the two accumulator rows is n-tile independent: low pixel (li, lj) feeds the 2x2 block at
                // tile (2li-1+a, 2lj-1+b); bit (2a+b) of `okm` = inside the staged tile, bit 4+(2a+b) = inside the image.
                uint32_t boff[2], okm[2];
                const unsigned char* okt = smem + G::OFF_CTB + G::CU * 4;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const int lp = mt * 16 + (lane >> 2) + 8 * hf;
                    const int li = lp / G::LPW, lj = lp - li * G::LPW;
                    boff[hf] = (uint32_t)(((2 * li - 1) * G::PW + (2 * lj - 1)) * 16);
                    okm[hf] = lp < G::LM ? (uint32_t)okt[lp] : 0u;
                }
#pragma unroll
                for (int i = 0; i < G::CT_NTG; ++i) {
                    const int nn = (ng + i) * 8 + 2 * (lane & 3);
                    const int pos = nn / G::CU, co = nn % G::CU;
                    const float bias0 = ctb[co], bias1 = ctb[co + 1];
                    const uint32_t poff = (uint32_t)((((pos >> 1) * G::PW + (pos & 1)) + (co >> 3) * G::PLANE) * 16 + (co & 7) * 2);
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        if ((okm[hf] >> pos) & 1u) {
                            const uint32_t v = ((okm[hf] >> (4 + pos)) & 1u)
                                                   ? pack2<T>(acc[i][2 * hf] + bias0, acc[i][2 * hf + 1] + bias1) : 0u;
                            *reinterpret_cast<uint32_t*>(act + boff[hf] + poff) = v;
                        }
                    }
                }
            }
        }
    }

    // ---- (3) main loop: 9 shifted GEMMs ------------------------------------------------------------------
    const uint32_t act_u = smem_u32(act);
    const uint32_t wgt_u = smem_u32(wgt);
    const int nt0 = wn * G::NT;
    // per-lane B row offset inside a chunk (bytes): matrix = lane>>3 -> (k-half, n-tile of the pair)
    const uint32_t b_lane = G::NT == 1 ? (uint32_t)(((((lane >> 3) & 1) * G::COUT) + nt0 * 8 + (lane & 7)) * 16)
                                       : (uint32_t)(((((lane >> 3) & 1) * G::COUT) + (nt0 + (lane >> 4)) * 8 + (lane & 7)) * 16);
    float s1[G::NT][2], s2[G::NT][2];
#pragma unroll
    for (int i = 0; i < G::NT; ++i) s1[i][0] = s1[i][1] = s2[i][0] = s2[i][1] = 0.f;
    T* outp = reinterpret_cast<T*>(p.out);

    if constexpr (G::ROLL) {
        static_assert(G::RW * (G::WM / G::SEGS) == G::TH && G::RW * G::NT * 4 <= 32, "ROLL: rows per warp / accumulator budget");
        cp_async_wait<0>();
        __syncthreads();  // weights + staged tile visible to every warp
        // B fragments of all 9 taps in registers: b[tap][nt][kh] = W[tap][ci = 8*kh + 2*(lane&3) (+1)][co = nt*8 + lane>>2]
        constexpr int KH = G::CIN == 8 ? 1 : 2;
        uint32_t bw[9][G::NT][KH];
#pragma unroll
        for (int t = 0; t < 9; ++t)
#pragma unroll
            for (int i = 0; i < G::NT; ++i)
#pragma unroll
                for (int kh = 0; kh < KH; ++kh) {
                    const int chunk = G::CIN == 8 ? t / 2 : t, khh = G::CIN == 8 ? (t & 1) : kh;
                    bw[t][i][kh] = *reinterpret_cast<const uint32_t*>(
                        wgt + ((size_t)(chunk * 2 + khh) * G::COUT + (nt0 + i) * 8 + (lane >> 2)) * 16 + (lane & 3) * 4);
                }
        const int seg = wm % G::SEGS, rb = wm / G::SEGS;
        float acc[G::RW][G::NT][4];
#pragma unroll
        for (int y = 0; y < G::RW; ++y)
#pragma unroll
            for (int i = 0; i < G::NT; ++i) acc[y][i][0] = acc[y][i][1] = acc[y][i][2] = acc[y][i][3] = 0.f;
        // lane's pixel of the m-tile in the haloed tile, input row 0 of this warp's block, kx = 0
        const uint32_t a_base = act_u + (uint32_t)(((rb * G::RW) * G::PW + seg * 16 + (lane & 15)) * 16);
#pragma unroll
        for (int r = 0; r < G::RW + 2; ++r) {  // input row r of the block feeds output rows r-2 .. r (ky = r - y)
            const uint32_t a_row = a_base + (uint32_t)(r * G::PW * 16);
            if constexpr (G::CIN == 8) {
                uint32_t f0, f1, f2, f3, g0, g1;
                ldsm_x4(a_row + (lane >> 4) * 16, f0, f1, f2, f3);   // lanes 0-15: kx = 0, lanes 16-31: kx = 1 (next pixel)
                ldsm_x2(a_row + 32, g0, g1);                          // kx = 2
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    const int y = r - ky;
                    if (y < 0 || y >= G::RW) continue;
#pragma unroll
                    for (int i = 0; i < G::NT; ++i) {
                        mma16816<T>(acc[y][i], f0, f1, f2, f3, bw[ky * 3][i][0], bw[ky * 3 + 1][i][0]);
                        mma16808<T>(acc[y][i], g0, g1, bw[ky * 3 + 2][i][0]);
                    }
                }
            } else {
                uint32_t f[3][4];
#pragma unroll
                for (int kx = 0; kx < 3; ++kx)   // lanes 0-15: channels 0-7 (plane 0), lanes 16-31: channels 8-15 (plane 1)
                    ldsm_x4(a_row + kx * 16 + (lane >> 4) * (G::PLANE * 16), f[kx][0], f[kx][1], f[kx][2], f[kx][3]);
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    const int y = r - ky;
                    if (y < 0 || y >= G::RW) continue;
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx)
#pragma unroll
                        for (int i = 0; i < G::NT; ++i)
                            mma16816<T>(acc[y][i], f[kx][0], f[kx][1], f[kx][2], f[kx][3], bw[ky * 3 + kx][i][0], bw[ky * 3 + kx][i][KH - 1]);
                }
            }
        }
        // epilogue: this warp's RW consecutive rows of one 16-pixel segment
        const bool full = (y0 + G::TH <= H) && (x0 + G::TW <= W);
        const int gx = x0 + seg * 16 + (lane >> 2);
        const uint32_t orow = (uint32_t)W * G::COUT;
        T* obase = outp + ((size_t)(n * H + y0 + rb * G::RW) * W + gx) * G::COUT + nt0 * 8 + 2 * (lane & 3);
        auto epilogue = [&](auto full_c) {
            constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
            for (int y = 0; y < G::RW; ++y) {
                const int gy = y0 + rb * G::RW + y;
                T* o = obase + (uint32_t)y * orow;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool ok = FULL || (gy < H && gx + 8 * hf < W);
#pragma unroll
                    for (int i = 0; i < G::NT; ++i) {
                        const float v0 = ok ? acc[y][i][2 * hf] : 0.f, v1 = ok ? acc[y][i][2 * hf + 1] : 0.f;
                        if (ok) *reinterpret_cast<uint32_t*>(o + hf * 8 * G::COUT + i * 8) = pack2<T>(v0, v1);
                        s1[i][0] += v0; s2[i][0] = fmaf(v0, v0, s2[i][0]);
                        s1[i][1] += v1; s2[i][1] = fmaf(v1, v1, s2[i][1]);
                    }
                }
            }
        };
        if (full) epilogue(std::true_type{});
        else epilogue(std::false_type{});
    } else {  // (braces: a bare `else` followed by `#pragma unroll` made nvcc drop the statement after the loop)
#pragma unroll 1
    for (int g = 0; g < G::MPW; g += G::MG) {
        float acc[G::MG][G::NT][4];
        uint32_t a_pix[G::MG];  // byte offset of this lane's A row (pixel) for each m-tile, tap (0,0), plane 0
#pragma unroll
        for (int m = 0; m < G::MG; ++m) {
            const int mt = wm + G::WM * (g + m);
            const int row = mt / G::SEGS, seg = mt % G::SEGS;
            a_pix[m] = (uint32_t)((row * G::PW + seg * 16 + (lane & 15)) * 16);
#pragma unroll
            for (int i = 0; i < G::NT; ++i) acc[m][i][0] = acc[m][i][1] = acc[m][i][2] = acc[m][i][3] = 0.f;
        }
        if constexpr (G::STREAM) {
            if (g > 0) {  // next group of m-tiles: stream the taps again (the trailing barrier of the last stage freed buffer 0)
                load_stage(0, 0);
                cp_async_commit();
            }
        }
#pragma unroll 1
        for (int stage = 0; stage < G::NSTAGE; ++stage) {
            if constexpr (G::STREAM) {
                if (stage + 1 < G::NSTAGE) {
                    load_stage(stage + 1, (stage + 1) & 1);
                    cp_async_commit();
                    cp_async_wait<1>();
                } else {
                    cp_async_wait<0>();
                }
                __syncthreads();
            } else {
                if (g == 0) {
                    cp_async_wait<0>();
                    __syncthreads();  // weights + staged tile visible to every warp
                }
            }
            const uint32_t wbuf = wgt_u + (G::STREAM ? (uint32_t)((stage & 1) * G::STAGE_CHUNKS * G::COUT * 32) : 0u);
#pragma unroll
            for (int j = 0; j < G::STAGE_CHUNKS; ++j) {
                // A offsets of this chunk: lanes 0-15 feed k 0..7, lanes 16-31 feed k 8..15
                uint32_t a_off;
                if constexpr (G::CIN == 8) {
                    const int t_lo = 2 * j, t_hi = (2 * j + 1 < 9) ? 2 * j + 1 : 8;
                    const int o_lo = ((t_lo / 3) * G::PW + (t_lo % 3)) * 16, o_hi = ((t_hi / 3) * G::PW + (t_hi % 3)) * 16;
                    a_off = (uint32_t)(o_lo + (lane >> 4) * (o_hi - o_lo));
                } else {
                    const int tap = G::STREAM ? stage : j / G::KC;
                    const int cp = G::STREAM ? j : j % G::KC;
                    a_off = (uint32_t)((((2 * cp + (lane >> 4)) * G::PLANE) + (tap / 3) * G::PW + (tap % 3)) * 16);
                }
                uint32_t bf[G::NT][2];
                if constexpr (G::NT == 1) {
                    ldsm_x2(wbuf + (uint32_t)(j * 2 * G::COUT * 16) + b_lane, bf[0][0], bf[0][1]);
                } else {
#pragma unroll
                    for (int np = 0; np < G::NT / 2; ++np)
                        ldsm_x4(wbuf + (uint32_t)((j * 2 * G::COUT + np * 16) * 16) + b_lane, bf[2 * np][0], bf[2 * np][1],
                                bf[2 * np + 1][0], bf[2 * np + 1][1]);
                }
#pragma unroll
                for (int m = 0; m < G::MG; ++m) {
                    uint32_t a0, a1, a2, a3;
                    ldsm_x4(act_u + a_pix[m] + a_off, a0, a1, a2, a3);
#pragma unroll
                    for (int i = 0; i < G::NT; ++i) mma16816<T>(acc[m][i], a0, a1, a2, a3, bf[i][0], bf[i][1]);
                }
            }
            if constexpr (G::STREAM) __syncthreads();  // everyone is done with this buffer before it is refilled
        }
        // ---- (4) epilogue for this group of m-tiles ------------------------------------------------------
        // Statistics come from the fp32 accumulators (the 16-bit rounding of the stored copy changes the plane sums
        // by ~2^-12/sqrt(n) relative -- far below the rounding noise itself) so no unpack is needed; full tiles
        // take a branch-free path with one address computation per m-tile.
        const bool full = (y0 + G::TH <= H) && (x0 + G::TW <= W);
        constexpr int RSTEP = G::WM / G::SEGS;
        static_assert(G::WM % G::SEGS == 0, "a warp's m-tiles share one 16-pixel segment");
        const int gx = x0 + (wm % G::SEGS) * 16 + (lane >> 2);
        const uint32_t orow = (uint32_t)W * G::COUT;  // elements per output row
        T* obase = outp + ((size_t)(n * H + y0 + wm / G::SEGS) * W + gx) * G::COUT + nt0 * 8 + 2 * (lane & 3);
        auto epilogue = [&](auto full_c) {
            constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
            for (int m = 0; m < G::MG; ++m) {
                // m-tile wm + WM*k sits RSTEP*k rows below the warp's first one, same 16-pixel segment
                const int gy = y0 + wm / G::SEGS + RSTEP * (g + m);
                T* o = obase + (uint32_t)((g + m) * RSTEP) * orow;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool ok = FULL || (gy < H && gx + 8 * hf < W);
#pragma unroll
                    for (int i = 0; i < G::NT; ++i) {
                        const float v0 = ok ? acc[m][i][2 * hf] : 0.f, v1 = ok ? acc[m][i][2 * hf + 1] : 0.f;
                        if (ok) *reinterpret_cast<uint32_t*>(o + hf * 8 * G::COUT + i * 8) = pack2<T>(v0, v1);
                        s1[i][0] += v0; s2[i][0] = fmaf(v0, v0, s2[i][0]);
                        s1[i][1] += v1; s2[i][1] = fmaf(v1, v1, s2[i][1]);
                    }
                }
            }
        };
        if (full) epilogue(std::true_type{});
        else epilogue(std::false_type{});
    }
    }
    // ---- (5) GroupNorm statistics: lanes with equal lane&3 hold the same channels -------------------------
#pragma unroll
    for (int i = 0; i < G::NT; ++i)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            float a = s1[i][k], b = s2[i][k];
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                a += __shfl_xor_sync(0xffffffffu, a, o);
                b += __shfl_xor_sync(0xffffffffu, b, o);
            }
            if (lane < 4) {
                // one slot per (m-warp, channel): no shared atomics, and the cross-warp sum below has a fixed order
                const int ch = (nt0 + i) * 8 + 2 * lane + k;
                statf[(wm * G::COUT + ch) * 2] = a;
                statf[(wm * G::COUT + ch) * 2 + 1] = b;
            }
        }
    __syncthreads();
    if (p.out_stats != nullptr)
        for (int c = tid; c < 2 * G::COUT; c += G::THREADS) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < G::WM; ++w) t += (double)statf[w * G::COUT * 2 + c];
            atomicAdd(p.out_stats + (size_t)n * G::COUT * 2 + c, t);
        }
}

// ---- weight packing kernels ------------------------------------------------------------------------------
template <typename T>
__global__ void pack_conv3x3_tc_kernel(const float* __restrict__ w, T* __restrict__ out, int cin, int cout, int nchunk) {
    // out[chunk][kh][co][8]
    const int total = nchunk * 2 * cout * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7;
        const int co = (i >> 3) % cout;
        const int kh = (i / (8 * cout)) & 1;
        const int chunk = i / (16 * cout);
        int tap, ci;
        if (cin == 8) {
            tap = 2 * chunk + kh;
            ci = e;
        } else {
            const int kc = cin / 16;
            tap = chunk / kc;
            ci = (chunk % kc) * 16 + kh * 8 + e;
        }
        const float v = tap < 9 ? w[((size_t)tap * cin + ci) * cout + co] : 0.f;
        out[i] = Store<T>::from_f(v);
    }
}

template <typename T>
__global__ void pack_convt_tc_kernel(const float* __restrict__ w, T* __restrict__ out, int cl, int cu) {
    // w [2][2][cl][cu] -> out[chunk = ci/16][kh][n = pos*cu + co][8]
    const int ctn = 4 * cu;
    const int total = (cl / 16) * 2 * ctn * 8;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int e = i & 7;
        const int nn = (i >> 3) % ctn;
        const int kh = (i / (8 * ctn)) & 1;
        const int chunk = i / (16 * ctn);
        const int ci = chunk * 16 + kh * 8 + e;
        const int pos = nn / cu, co = nn % cu;
        out[i] = Store<T>::from_f(w[((size_t)pos * cl + ci) * cu + co]);
    }
}

static int tc_nchunk(int cin) { return cin == 8 ? 5 : 9 * (cin / 16); }

int tc_conv3x3_bytes(int cin, int cout, size_t* bytes) {
    if (cin < 8 || (cin != 8 && cin % 16) || cout % 8) { set_error("tc packing: unsupported %d -> %d", cin, cout); return 3; }
    *bytes = (size_t)tc_nchunk(cin) * cout * 32;
    return 0;
}
int tc_convt_bytes(int cl, int cu, size_t* bytes) {
    if (cl % 16 || cu % 8) { set_error("tc convT packing: unsupported %d -> %d", cl, cu); return 3; }
    *bytes = (size_t)cl * 4 * cu * 2;
    return 0;
}
int pack_conv3x3_tc(const float* w, void* out, int cin, int cout, int dtype, cudaStream_t st) {
    size_t bytes;
    int rc = tc_conv3x3_bytes(cin, cout, &bytes);
    if (rc) return rc;
    const int total = (int)(bytes / 2);
    const int blocks = (total + 255) / 256;
    if (dtype == DG_F16) pack_conv3x3_tc_kernel<__half><<<blocks, 256, 0, st>>>(w, (__half*)out, cin, cout, tc_nchunk(cin));
    else if (dtype == DG_BF16) pack_conv3x3_tc_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(w, (__nv_bfloat16*)out, cin, cout, tc_nchunk(cin));
    else { set_error("tc packing needs a 16-bit dtype"); return 2; }
    count_launch();
    return check_launch("pack_conv3x3_tc");
}
int pack_convt_tc(const float* w, void* out, int cl, int cu, int dtype, cudaStream_t st) {
    size_t bytes;
    int rc = tc_convt_bytes(cl, cu, &bytes);
    if (rc) return rc;
    const int total = (int)(bytes / 2);
    const int blocks = (total + 255) / 256;
    if (dtype == DG_F16) pack_convt_tc_kernel<__half><<<blocks, 256, 0, st>>>(w, (__half*)out, cl, cu);
    else if (dtype == DG_BF16) pack_convt_tc_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(w, (__nv_bfloat16*)out, cl, cu);
    else { set_error("tc packing needs a 16-bit dtype"); return 2; }
    count_launch();
    return check_launch("pack_convt_tc");
}

// ---- dispatch -----------------------------------------------------------------------------------------------
template <typename T, typename G>
static int launch_geo(const TcArgs& t, cudaStream_t st) {
    auto kern = conv3x3_tc_kernel<T, G>;
    static bool attr_done = false;  // per instantiation
    if (!attr_done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, G::SMEM_BYTES);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%d B): %s", G::SMEM_BYTES, cudaGetErrorString(e)); return 4; }
        attr_done = true;
    }
    dim3 grid((t.W + G::TW - 1) / G::TW, (t.H + G::TH - 1) / G::TH, t.N);
    cudaError_t le = launch_kernel(kern, grid, dim3(G::THREADS), (size_t)G::SMEM_BYTES, st, t);
    if (le != cudaSuccess) { set_error("conv3x3_tc launch: %s", cudaGetErrorString(le)); return 10; }
    count_launch();
    return check_launch("conv3x3_tc");
}

template <typename T>
static int dispatch(const dg_conv3x3_args& a, const TcArgs& t, int mode, int cin, cudaStream_t st, bool* handled) {
    *handled = true;
    const int cout = a.cout;
#define DG_TC(CI, CO, MD, TH, TW, WM, WN, ST) \
    if (cin == CI && cout == CO && mode == MD) return launch_geo<T, Geo<CI, CO, MD, TH, TW, WM, WN, ST>>(t, st);
    DG_TC(8, 8, M_SAME, 16, 32, 4, 1, false)      // enc1.3, dec1.3 (128-thread CTAs: 8 independent phase streams per SM)
    DG_TC(8, 16, M_POOL, 16, 64, 8, 1, false)     // enc2.0 (ROLL measured slower: .135 vs .112 ms, pooled staging wants the wide tile)
    DG_TC(16, 16, M_SAME, 16, 64, 8, 1, false)    // enc2.3, dec2.3 (ROLL at 16x32 measured slower: .117 vs .099 ms)
    DG_TC(16, 32, M_POOL, 16, 32, 8, 1, false)    // enc3.0
    DG_TC(32, 32, M_SAME, 16, 32, 8, 1, false)    // enc3.3, dec3.3
    DG_TC(32, 64, M_POOL, 8, 32, 4, 2, false)     // enc4.0 (WM=8 WN=1 measured: .062 vs .054 ms)
    DG_TC(64, 64, M_SAME, 8, 32, 4, 2, true)      // enc4.3, dec4.3 (WM=8 WN=1 measured: .0775 vs .0741 ms)
    DG_TC(64, 128, M_POOL, 4, 32, 2, 4, true)     // bottleneck.0
    DG_TC(128, 128, M_SAME, 4, 32, 2, 4, true)    // bottleneck.3 (WM=4 WN=2 measured: .086 vs .084 ms)
    DG_TC(128, 64, M_CAT2, 8, 16, 4, 2, true)     // dec4.0 on a materialised upconv4 (8x32 tile, WM=8 WN=1 measured: .190 vs .175 ms)
    DG_TC(64, 32, M_CAT2, 8, 32, 8, 1, true)      // dec3.0 on a materialised upconv3 (WM=8 WN=1: four n-tiles per A fragment, .201 -> .185 ms)
    DG_TC(32, 16, M_CAT2, 8, 64, 8, 1, false)     // dec2.0 on a materialised upconv2
    DG_TC(128, 64, M_UPCAT, 8, 16, 4, 2, true)    // upconv4 + dec4.0
    DG_TC(64, 32, M_UPCAT, 8, 32, 4, 2, true)     // upconv3 + dec3.0
    DG_TC(32, 16, M_UPCAT, 16, 32, 8, 1, false)   // upconv2 + dec2.0 (16x32 tile: smaller low-res halo than 8x64, .236 -> .229 ms)
    DG_TC(16, 8, M_UPCAT, 16, 64, 8, 1, false)    // upconv1 + dec1.0 (16x32 tile with 4 warps measured: .335 vs .319 ms)
#undef DG_TC
    *handled = false;
    return 0;
}

int conv3x3_tc_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled) {
    *handled = false;
    if (a.dtype != DG_F16 && a.dtype != DG_BF16) return 0;
    if (a.weight_tc == nullptr || a.act_sum != nullptr) return 0;
    const dg_src& s0 = a.src[0];
    TcArgs t;
    memset(&t, 0, sizeof(t));
    int mode, cin;
    if (a.nsrc == 1 && (s0.xform == DG_X_SAME || s0.xform == DG_X_POOL2)) {
        if (s0.stats == nullptr || !s0.silu || s0.scale != nullptr) return 0;
        mode = s0.xform == DG_X_SAME ? M_SAME : M_POOL;
        cin = s0.channels;
    } else if (a.nsrc == 2 && s0.xform == DG_X_SAME && a.src[1].xform == DG_X_SAME && s0.stats == nullptr && !s0.silu &&
               s0.scale == nullptr) {
        const dg_src& s1 = a.src[1];
        if (s1.stats == nullptr || !s1.silu || s1.scale || s0.channels != a.cout || s1.channels != a.cout) return 0;
        mode = M_CAT2;
        cin = 2 * a.cout;
        t.src1 = s1.raw; t.st1 = s1.stats; t.g1 = s1.gamma; t.b1 = s1.beta; t.groups1 = s1.groups;
    } else if (a.nsrc == 2 && s0.xform == DG_X_CONVT2 && a.src[1].xform == DG_X_SAME) {
        const dg_src& s1 = a.src[1];
        if (s0.stats == nullptr || s1.stats == nullptr || !s0.silu || !s1.silu || s0.scale || s1.scale) return 0;
        if (s0.ct_w_tc == nullptr || s0.ct_cout != a.cout || s1.channels != a.cout || s0.channels != 2 * a.cout) return 0;
        if ((a.H | a.W) & 1) return 0;
        mode = M_UPCAT;
        cin = s0.channels;
        t.src1 = s1.raw; t.st1 = s1.stats; t.g1 = s1.gamma; t.b1 = s1.beta; t.groups1 = s1.groups;
        t.ctw = s0.ct_w_tc; t.ctb = s0.ct_b;
    } else {
        return 0;
    }
    // 128-bit loads need 16-byte aligned bases
    if ((reinterpret_cast<uintptr_t>(s0.raw) | reinterpret_cast<uintptr_t>(a.out) | reinterpret_cast<uintptr_t>(a.weight_tc) |
         reinterpret_cast<uintptr_t>(t.src1) | reinterpret_cast<uintptr_t>(t.ctw)) & 15)
        return 0;
    if (a.N > 65535) return 0;
    t.src0 = s0.raw; t.st0 = s0.stats; t.g0 = s0.gamma; t.b0 = s0.beta; t.groups0 = s0.groups;
    t.cf0 = s0.coef;
    if (a.nsrc == 2) t.cf1 = a.src[1].coef;
    t.wgt = a.weight_tc;
    t.out = a.out; t.out_stats = a.out_stats;
    t.N = a.N; t.H = a.H; t.W = a.W; t.eps = a.eps;
    if (a.dtype == DG_F16) return dispatch<__half>(a, t, mode, cin, stream, handled);
    return dispatch<__nv_bfloat16>(a, t, mode, cin, stream, handled);
}

}  // namespace dg
