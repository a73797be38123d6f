// Warp-specialised tcgen05 implicit-GEMM 3x3 conv (sm_100a) for every layer with C_out >= 32: the deep levels of the shipped
// LightweightUNet(features_start=8) and ALL of the wide variant (features_start=64, BASELINE.json configs[4]).  Same fusion
// contract as conv3x3_tc.cu -- GroupNorm apply + SiLU [+ AvgPool2d | identity `up` half of torch.cat] on load, raw NHWC
// output + GroupNorm statistics of the stored values in the epilogue (src/model.py:92-99, :35-41, :116-128).
//
// Roles of one persistent CTA (one per SM, 14 warps), coupled only by mbarriers -- there is no CTA-wide barrier in the loop:
//   warps 0-3   epilogue: tcgen05.ld -> round to the storage type -> 128-bit NHWC stores; the GroupNorm statistics are
//               column sums of the stored tile, taken through a padded per-warp shared-memory transpose;
//   warps 4-19  stagers: raw NHWC -> GroupNorm affine + SiLU (+ 2x2 mean | plain copy of `up`) -> 16-bit channel planes;
//   warp 20     weight producer: one thread streams [tap][KC ci][NB co] weight tiles into a shared-memory ring with
//               cp.async.bulk (TMA bulk copy, completes on the ring's `full` mbarrier);
//   warps 21-22 MMA issuers (M-tiles of a work item interleaved between them): one thread issues tcgen05.mma (M = 128 pixels, N = NB <= 128 output channels, K = 16) with the
//               accumulators in tensor memory, and releases ring slots / publishes accumulators with tcgen05.commit.
// While the tensor core runs work item i, the stagers already build the A operand of item i+1 and the epilogue drains
// item i-1 from the other TMEM stage.
//
// Implicit GEMM without im2col, "q-stream" tiling: the zero-padded image is the 1-D pixel stream q' = r'*(W+2) + c'
// (r', c' = haloed coordinates).  Output pixel q = y*(W+2) + x reads input q + ky*(W+2) + kx for tap (ky, kx), so with the
// activated stream in shared memory as 16-bit channel planes [KC/8][pixels][8 ch] (8 consecutive pixels of a plane = one
// 128-byte core matrix of the no-swizzle K-major UMMA layout: LBO = plane stride, SBO = 128 B) EVERY tap, horizontal ones
// included, is a pure start-address offset of the A descriptor.  An M-tile is any 128 consecutive q; the two halo columns
// per row produce accumulator rows that are simply not stored (2/(W+2) of the MMA work).  One staged copy of the tile
// serves all 9 taps -- the round-1 UMMA kernel needed three kx-shifted copies.  A work item is `mt` consecutive M-tiles
// of one image times one block of NB output channels; K is walked in chunks of KC input channels (A ring) x 9 taps (B ring).
#include <cstdio>
#include <cstdlib>

#include "tc_common.cuh"

namespace dg {

namespace {

enum { T5_SAME = 0, T5_POOL = 1, T5_CAT2 = 3, T5_CONVT = 4, T5_IDENT = 6 };   // T5_CONVT: ConvTranspose2d(2,2)+bias as a 1-tap GEMM with N = 4*C_up
// T5_IDENT: the conv DATA GRADIENT of the wide layers (dgrad = a 3x3 conv of dR with the taps-flipped, transposed weights): the one
// source is an identity bf16 tensor (no GroupNorm, no SiLU: chunks are copied), the epilogue stores the fp32 accumulators as fp32
// [N,H,W,cout] and keeps no statistics.
constexpr int T5_STAGE_WARPS = 16;   // staging is dependent-chain bound per warp (measured ~0.1 IPC): it scales with warps, not with ILP
constexpr int T5_STAGE_THREADS = 32 * T5_STAGE_WARPS;
// Warp roles by warp id.  The warp scheduler prefers the HIGHEST warp id among eligible warps (B300_MICROARCH.md, "arbiter
// priority: hi-wid-first"), so the two single-thread control warps sit on top -- measured with the MMA issuer as warp 1 below
// eight FFMA/MUFU-saturated stager warps: ~250 clk per issued MMA against the 56 clk the tensor core needs (tools/umma_rate.cu).
constexpr int T5_EPI_WARP0 = 0;                    // warps 0-3 epilogue (warp % 4 = TMEM lane quarter), 4-11 stagers: the stagers are the
constexpr int T5_STG_WARP0 = 4;                    // throughput-critical CUDA-core role, so they outrank the epilogue at the schedulers
constexpr int T5_TMA_WARP = T5_STG_WARP0 + T5_STAGE_WARPS;   // 20: weight producer
constexpr int T5_MMA_WARP = T5_TMA_WARP + 1;        // 21, 22: MMA issuers (M-tiles interleaved between them); 13 owns the TMEM allocation
constexpr int T5_MMA_WARPS = 2;
constexpr int T5_THREADS = 32 * (T5_MMA_WARP + T5_MMA_WARPS);  // 736 threads: 88 registers each
constexpr int T5_SCR_PITCH = 80;                                      // bytes per pixel row of the statistics transpose (64 + 16)
constexpr int T5_MAX_RING = 8;

struct T5Args {
    const void* src0; const double* st0; const float* g0; const float* b0; const float* cf0; int groups0;
    const void* src1; const double* st1; const float* g1; const float* b1; const float* cf1; int groups1;
    const void* wgt; void* out; double* out_stats;
    int N, H, W; float eps;
    int cin, cout;
    int pitch;        // tw + 2: pixels per row of the q-stream
    int tw, nstrips;  // the image is cut into column strips of tw <= 128 output columns (+ 2 halo columns) so that the two
                      // halo ROWS every work item stages cost 2 (tw + 2) pixels, not 2 (W + 2) (wide variant: W = 512 at level 1)
    int mt;           // M-tiles (128 stream pixels each) per work item
    int mtiles_img;   // M-tiles per image
    int bands_img;    // work items per image and n-block
    int kc, nchunk;   // input channels per A chunk, chunks
    int nb, nnb;      // output channels per block, blocks
    int plane_px;     // pixels per channel plane (padded for conflict-free staging stores)
    int na, nbs, ts;  // ring depths: A chunks, weight tiles, TMEM accumulator stages
    int a_stage_bytes, b_stage_bytes;
    int tmem_cols;
    int off_b, off_coef, off_scr, off_bar;
    int ncoef;
    int ntaps;        // 9, or 1 (T5_CONVT: the centre tap only)
    int cu;           // T5_CONVT: channels of the full-resolution output (GEMM N = cout = 4 * cu)
    const float* bias;   // T5_CONVT: [cu]
    int items;
    long long* trace;   // DG_T5_TRACE=1: per-role clock64 timestamps of CTA 0 (debug aid, see t5_trace_dump)
};

__device__ __forceinline__ uint64_t t5_desc(uint32_t addr, uint32_t lbo, uint32_t sbo) {
    return (uint64_t)((addr & 0x3FFFF) >> 4) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
           ((uint64_t)1 << 46);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// Bounded wait: a protocol error must abort the launch, not hang the GPU.  try_wait suspends the thread in hardware (up to the
// hint) and is woken by the completing arrive, so waiting warps do not take issue slots from the working ones; the clock is
// only looked at every 64 wake-ups.
__device__ __forceinline__ bool mbar_try(uint32_t bar, uint32_t parity) {
    uint32_t done;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    return done != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    for (uint32_t spin = 1;; ++spin) {
        if (mbar_try(bar, parity)) return;
        if ((spin & 63u) == 0 && clock64() - t0 > 8000000000LL) __trap();
    }
}
// Waits that are a whole pipeline stage ahead of the critical path (stagers, epilogue, weight producer) back off between polls,
// so that idle roles do not take issue slots from the working ones.
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) {
    if (mbar_try(bar, parity)) return;
    const long long t0 = clock64();
    for (uint32_t spin = 1;; ++spin) {
        __nanosleep(64);
        if (mbar_try(bar, parity)) return;
        if ((spin & 63u) == 0 && clock64() - t0 > 8000000000LL) __trap();
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}" : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void stager_bar() { asm volatile("bar.sync 1, %0;" ::"n"(T5_STAGE_THREADS) : "memory"); }

// trace slots: [role 0..3][event index], 512 events per role
#define T5_TRACE(role, idx) do { if (p.trace != nullptr && blockIdx.x == 0 && (idx) < 512) p.trace[(role) * 512 + (idx)] = clock64(); } while (0)

// All MMAs one issuer warp owes to one tap: `count` M-tiles (every T5_MMA_WARPS-th of the work item) x KS K-steps, from ONE asm
// block whose loop runs warp-uniformly; the elected lane's guard predicate issues.  (C++ loops around a per-MMA asm compiled to
// ~70 SASS instructions of R2UR / predicate shuffling per M-tile = ~300 clk against the 56 clk an N = 32 MMA needs.)
template <int KS>
__device__ __forceinline__ void t5_issue_tap(uint32_t dc, uint64_t da, uint64_t db, uint32_t idesc, uint64_t dA, uint64_t dB,
                                             uint32_t accumulate, int count, uint32_t dc_step) {
    if constexpr (KS == 1) {
        asm volatile(
            "{\n\t"
            ".reg .pred pel, pacc, ploop;\n\t.reg .b64 da;\n\t.reg .b32 dc, m;\n\t"
            "elect.sync _|pel, 0xffffffff;\n\t"
            "setp.ne.b32 pacc, %6, 0;\n\t"
            "mov.b64 da, %1;\n\tmov.b32 dc, %0;\n\tmov.b32 m, %7;\n"
            "T5_L1:\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], da, %2, %3, pacc;\n\t"
            "add.u64 da, da, %9;\n\tadd.u32 dc, dc, %8;\n\tsub.u32 m, m, 1;\n\t"
            "setp.ne.b32 ploop, m, 0;\n\t@ploop bra.uni T5_L1;\n\t"
            "}"
            ::"r"(dc), "l"(da), "l"(db), "r"(idesc), "l"(dA), "l"(dB), "r"(accumulate), "r"(count), "r"(dc_step),
              "l"((uint64_t)(128 * T5_MMA_WARPS)));
    } else if constexpr (KS == 2) {
        asm volatile(
            "{\n\t"
            ".reg .pred pel, pacc, ptrue, ploop;\n\t.reg .b64 da, a1, b1;\n\t.reg .b32 dc, m;\n\t"
            "elect.sync _|pel, 0xffffffff;\n\t"
            "setp.ne.b32 pacc, %6, 0;\n\tsetp.eq.b32 ptrue, 0, 0;\n\t"
            "add.u64 b1, %2, %5;\n\t"
            "mov.b64 da, %1;\n\tmov.b32 dc, %0;\n\tmov.b32 m, %7;\n"
            "T5_L2:\n\t"
            "add.u64 a1, da, %4;\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], da, %2, %3, pacc;\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], a1, b1, %3, ptrue;\n\t"
            "add.u64 da, da, %9;\n\tadd.u32 dc, dc, %8;\n\tsub.u32 m, m, 1;\n\t"
            "setp.ne.b32 ploop, m, 0;\n\t@ploop bra.uni T5_L2;\n\t"
            "}"
            ::"r"(dc), "l"(da), "l"(db), "r"(idesc), "l"(dA), "l"(dB), "r"(accumulate), "r"(count), "r"(dc_step),
              "l"((uint64_t)(128 * T5_MMA_WARPS)));
    } else {
        asm volatile(
            "{\n\t"
            ".reg .pred pel, pacc, ptrue, ploop;\n\t.reg .b64 da, a1, a2, a3, b1, b2, b3;\n\t.reg .b32 dc, m;\n\t"
            "elect.sync _|pel, 0xffffffff;\n\t"
            "setp.ne.b32 pacc, %6, 0;\n\tsetp.eq.b32 ptrue, 0, 0;\n\t"
            "add.u64 b1, %2, %5;\n\tadd.u64 b2, b1, %5;\n\tadd.u64 b3, b2, %5;\n\t"
            "mov.b64 da, %1;\n\tmov.b32 dc, %0;\n\tmov.b32 m, %7;\n"
            "T5_L4:\n\t"
            "add.u64 a1, da, %4;\n\tadd.u64 a2, a1, %4;\n\tadd.u64 a3, a2, %4;\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], da, %2, %3, pacc;\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], a1, b1, %3, ptrue;\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], a2, b2, %3, ptrue;\n\t"
            "@pel tcgen05.mma.cta_group::1.kind::f16 [dc], a3, b3, %3, ptrue;\n\t"
            "add.u64 da, da, %9;\n\tadd.u32 dc, dc, %8;\n\tsub.u32 m, m, 1;\n\t"
            "setp.ne.b32 ploop, m, 0;\n\t@ploop bra.uni T5_L4;\n\t"
            "}"
            ::"r"(dc), "l"(da), "l"(db), "r"(idesc), "l"(dA), "l"(dB), "r"(accumulate), "r"(count), "r"(dc_step),
              "l"((uint64_t)(128 * T5_MMA_WARPS)));
    }
}

struct T5Item { int n, m0, mt_cur, nbk, xs; };
__device__ __forceinline__ T5Item t5_item(const T5Args& p, int item) {
    T5Item it;
    it.nbk = item % p.nnb;
    const int rest = item / p.nnb;
    const int sn = rest / p.bands_img;            // (image, strip)
    const int band = rest - sn * p.bands_img;
    it.n = sn / p.nstrips;
    it.xs = (sn - it.n * p.nstrips) * p.tw;       // first output column of the strip
    it.m0 = band * p.mt;
    const int left = p.mtiles_img - it.m0;
    it.mt_cur = left < p.mt ? left : p.mt;
    return it;
}

template <typename T, int MODE>
__global__ void __launch_bounds__(T5_THREADS, 1) conv3x3_t5_kernel(const __grid_constant__ T5Args p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + p.off_bar);
    // barrier table: a_full[R] a_empty[R] b_full[R] b_empty[R] t_full[2] t_empty[2], R = T5_MAX_RING
    const uint32_t bar0 = smem_u32(bars);
    auto A_FULL = [&](int s) { return bar0 + 8u * s; };
    auto A_EMPTY = [&](int s) { return bar0 + 8u * (T5_MAX_RING + s); };
    auto B_FULL = [&](int s) { return bar0 + 8u * (2 * T5_MAX_RING + s); };
    auto B_EMPTY = [&](int s) { return bar0 + 8u * (3 * T5_MAX_RING + s); };
    auto T_FULL = [&](int s) { return bar0 + 8u * (4 * T5_MAX_RING + s); };
    auto T_EMPTY = [&](int s) { return bar0 + 8u * (4 * T5_MAX_RING + 2 + s); };
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + p.off_bar + 8 * (4 * T5_MAX_RING + 4));

    pdl_launch_dependents();
    if (tid == 0) {
        for (int s = 0; s < T5_MAX_RING; ++s) {
            mbar_init(A_FULL(s), T5_STAGE_THREADS);
            mbar_init(A_EMPTY(s), T5_MMA_WARPS);
            mbar_init(B_FULL(s), 1);
            mbar_init(B_EMPTY(s), T5_MMA_WARPS);
        }
        for (int s = 0; s < 2; ++s) {
            mbar_init(T_FULL(s), T5_MMA_WARPS);
            mbar_init(T_EMPTY(s), 128);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == T5_MMA_WARP) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(p.tmem_cols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t taddr = *tmem_slot;

    // contiguous range of work items of this CTA (few image changes -> few statistics flushes / coefficient rebuilds)
    const int it0 = (int)((long long)p.items * blockIdx.x / gridDim.x);
    const int it1 = (int)((long long)p.items * (blockIdx.x + 1) / gridDim.x);
    const int ksteps = p.kc >> 4;
    const uint32_t plane_bytes = (uint32_t)p.plane_px * 16u;
    const uint32_t a_base = smem_u32(smem);
    const uint32_t b_base = smem_u32(smem + p.off_b);

    if (warp == T5_TMA_WARP) {
        // ================= weight producer (TMA bulk copies) =================
        if (lane == 0) {
            int sb = 0; uint32_t pb = 0;
            const unsigned char* wg = reinterpret_cast<const unsigned char*>(p.wgt);
            const int kst_tot = p.cin >> 4;
            for (int item = it0; item < it1; ++item) {
                const int nbk = item % p.nnb;
                for (int ch = 0; ch < p.nchunk; ++ch)
                    for (int tap = 0; tap < p.ntaps; ++tap) {
                        mbar_wait_relaxed(B_EMPTY(sb), pb ^ 1u);
                        if (ch == 0 && (tap == 0 || tap == 8)) T5_TRACE(3, 2 * (item - it0) + (tap ? 1 : 0));
                        mbar_expect_tx(B_FULL(sb), (uint32_t)p.b_stage_bytes);
                        const uint32_t dst = b_base + (uint32_t)sb * p.b_stage_bytes;
                        const size_t ck = (size_t)tap * kst_tot + (size_t)ch * ksteps;   // first 16-channel weight chunk
                        if (p.nnb == 1) {
                            bulk_g2s(dst, wg + ck * p.cout * 32, (uint32_t)p.b_stage_bytes, B_FULL(sb));
                        } else {
                            for (int j = 0; j < 2 * ksteps; ++j)   // (k-step, k-half) slices of NB output channels
                                bulk_g2s(dst + (uint32_t)j * p.nb * 16, wg + (ck * 2 + j) * p.cout * 16 + (size_t)nbk * p.nb * 16,
                                         (uint32_t)p.nb * 16, B_FULL(sb));
                        }
                        if (++sb == p.nbs) { sb = 0; pb ^= 1u; }
                    }
            }
        }
    } else if (warp >= T5_MMA_WARP) {
        // ================= MMA issuers =================
        // The WHOLE warp walks the loop nest (uniform control flow, so every descriptor lives in uniform registers and an MMA
        // costs ~6 issue slots); one elected lane issues.  Measured with a single-lane loop: ~35 SASS instructions per MMA incl.
        // a R2UR waterfall = 150-190 clk per MMA against the 56-64 clk the tensor core needs (tools/umma_rate.cu).
        {
            const uint32_t idesc = (1u << 4) | ((std::is_same<T, __half>::value ? 0u : 1u) << 7) |
                                   ((std::is_same<T, __half>::value ? 0u : 1u) << 10) | ((uint32_t)(p.nb >> 3) << 17) |
                                   ((uint32_t)(128 >> 4) << 24);
            const uint64_t dA = 2u * (uint32_t)p.plane_px, dB = 2u * (uint32_t)p.nb;   // descriptor advance per K step (16-byte units)
            const int mw = warp - T5_MMA_WARP;   // this warp issues M-tiles mw, mw + T5_MMA_WARPS, ...
            int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
            int k = 0;
            for (int item = it0; item < it1; ++item, ++k) {
                const T5Item it = t5_item(p, item);
                const int tsg = p.ts == 2 ? (k & 1) : 0;
                const uint32_t tph = p.ts == 2 ? ((k >> 1) & 1) : (k & 1);
                mbar_wait_relaxed(T_EMPTY(tsg), tph ^ 1u);   // long waits back off: a spinning issuer warp (highest scheduler
                tc_fence_after();                           // priority) would starve the stagers it is waiting for
                if (lane == 0 && mw == 0) T5_TRACE(0, 4 * k);
                const int cnt = it.mt_cur > mw ? (it.mt_cur - mw + T5_MMA_WARPS - 1) / T5_MMA_WARPS : 0;
                const uint32_t dcol = taddr + (uint32_t)(tsg * p.mt * p.nb);
                for (int ch = 0; ch < p.nchunk; ++ch) {
                    mbar_wait_relaxed(A_FULL(sa), pa);
                    tc_fence_after();
                    if (ch == 0 && lane == 0 && mw == 0) T5_TRACE(0, 4 * k + 1);
                    const uint64_t da_chunk = t5_desc(a_base + (uint32_t)sa * p.a_stage_bytes, plane_bytes, 128);
                    for (int tap = 0; tap < p.ntaps; ++tap) {
                        mbar_wait(B_FULL(sb), pb);
                        tc_fence_after();
                        const int ky = p.ntaps == 1 ? 1 : tap / 3, kx = p.ntaps == 1 ? 1 : tap - ky * 3;
                        const uint64_t da = da_chunk + (uint32_t)(ky * p.pitch + kx);
                        const uint64_t db = t5_desc(b_base + (uint32_t)sb * p.b_stage_bytes, (uint32_t)p.nb * 16u, 128);
                        if (cnt > 0) {
                            const uint32_t acc = (ch | tap) ? 1u : 0u;
                            const uint32_t dc0 = dcol + (uint32_t)(mw * p.nb);
                            const uint64_t da0 = da + (uint32_t)(mw * 128);
                            if (ksteps == 4) t5_issue_tap<4>(dc0, da0, db, idesc, dA, dB, acc, cnt, (uint32_t)(T5_MMA_WARPS * p.nb));
                            else if (ksteps == 2) t5_issue_tap<2>(dc0, da0, db, idesc, dA, dB, acc, cnt, (uint32_t)(T5_MMA_WARPS * p.nb));
                            else t5_issue_tap<1>(dc0, da0, db, idesc, dA, dB, acc, cnt, (uint32_t)(T5_MMA_WARPS * p.nb));
                        }
                        __syncwarp();
                        if (elect_one()) umma_commit(B_EMPTY(sb));
                        if (++sb == p.nbs) { sb = 0; pb ^= 1u; }
                    }
                    if (elect_one()) umma_commit(A_EMPTY(sa));
                    if (++sa == p.na) { sa = 0; pa ^= 1u; }
                }
                if (elect_one()) umma_commit(T_FULL(tsg));
                if (lane == 0 && mw == 0) T5_TRACE(0, 4 * k + 2);
            }
        }
    } else if (warp < T5_STG_WARP0) {
        // ================= epilogue: TMEM -> HBM + GroupNorm statistics =================
        pdl_wait();   // the output buffer / statistics may still be read by the kernels before the producer of our inputs
        const int wq = warp & 3;   // TMEM lane quarter this warp may access
        unsigned char* scr = smem + p.off_scr + (warp - T5_EPI_WARP0) * (32 * T5_SCR_PITCH);
        const int half = lane >> 4, pr = lane & 15;
        // fp32 partial sums cover 16 pixels of ONE M-tile (fixed order); everything above that is accumulated in double, so the
        // statistics -- and with them the network output -- do not depend on how work items are spread over CTAs / batch sizes
        double s1[4][2], s2[4][2];
#pragma unroll
        for (int c = 0; c < 4; ++c) s1[c][0] = s1[c][1] = s2[c][0] = s2[c][1] = 0.0;
        int stats_n = -1, stats_nbk = 0;
        const int ncc = p.nb >> 5;
        auto flush = [&]() {
            if (stats_n < 0 || p.out_stats == nullptr) return;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                if (c < ncc) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        const double a = s1[c][e] + __shfl_xor_sync(0xffffffffu, s1[c][e], 16);
                        const double b = s2[c][e] + __shfl_xor_sync(0xffffffffu, s2[c][e], 16);
                        if (half == 0) {
                            const int col = stats_nbk * p.nb + c * 32 + 2 * pr + e;
                            double* d = p.out_stats + ((size_t)stats_n * p.cout + col) * 2;
                            atomicAdd(d, a);
                            atomicAdd(d + 1, b);
                        }
                    }
                }
                s1[c][0] = s1[c][1] = s2[c][0] = s2[c][1] = 0.0;
            }
        };
        int k = 0;
        for (int item = it0; item < it1; ++item, ++k) {
            const T5Item it = t5_item(p, item);
            if (it.n != stats_n || it.nbk != stats_nbk) {
                flush();
                stats_n = it.n;
                stats_nbk = it.nbk;
            }
            const int tsg = p.ts == 2 ? (k & 1) : 0;
            const uint32_t tph = p.ts == 2 ? ((k >> 1) & 1) : (k & 1);
            mbar_wait_relaxed(T_FULL(tsg), tph);
            tc_fence_after();
            if (warp == T5_EPI_WARP0 && lane == 0) T5_TRACE(1, 2 * k);
            for (int m = 0; m < it.mt_cur; ++m) {
                const int q = (it.m0 + m) * 128 + wq * 32 + lane;
                const int y = q / p.pitch, xl = q - y * p.pitch, x = it.xs + xl;
                const bool valid = xl < p.tw && x < p.W && y < p.H;
                T* o = reinterpret_cast<T*>(p.out) + ((size_t)(it.n * p.H + y) * p.W + x) * p.cout + it.nbk * p.nb;
                const uint32_t trow = taddr + ((uint32_t)(wq * 32) << 16) + (uint32_t)((tsg * p.mt + m) * p.nb);
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    if (c < ncc) {
                        uint32_t r[32];
                        asm volatile(
                            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                            "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                              "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                              "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                              "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                            : "r"(trow + (uint32_t)(c * 32)));
                        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                        if constexpr (MODE == T5_IDENT) {
                            // data gradient: fp32 out, 32 consecutive channels of this lane's pixel = eight 128-bit stores
                            if (valid) {
                                float4* of = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) +
                                                                       ((size_t)(it.n * p.H + y) * p.W + x) * p.cout + it.nbk * p.nb + c * 32);
#pragma unroll
                                for (int j = 0; j < 8; ++j)
                                    of[j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                                                        __uint_as_float(r[4 * j + 3]));
                            }
                        } else if constexpr (MODE == T5_CONVT) {
                            // ConvTranspose2d(2,2): column n = pos * cu + co of low pixel (y, x) is channel co of output pixel
                            // (2y + pos/2, 2x + pos%2); + bias, no statistics (the consumer treats `up` as an identity source)
                            const int n0 = it.nbk * p.nb + c * 32;
                            const int pos = n0 / p.cu, co0 = n0 - pos * p.cu;
                            if (valid) {
                                T* ou = reinterpret_cast<T*>(p.out) +
                                        ((size_t)(it.n * 2 * p.H + 2 * y + (pos >> 1)) * (2 * p.W) + 2 * x + (pos & 1)) * p.cu + co0;
                                const float4* bp = reinterpret_cast<const float4*>(p.bias + co0);
#pragma unroll
                                for (int j = 0; j < 4; ++j) {
                                    const float4 b0 = __ldg(bp + 2 * j), b1 = __ldg(bp + 2 * j + 1);
                                    *reinterpret_cast<uint4*>(ou + j * 8) = make_uint4(
                                        pack2<T>(__uint_as_float(r[8 * j]) + b0.x, __uint_as_float(r[8 * j + 1]) + b0.y),
                                        pack2<T>(__uint_as_float(r[8 * j + 2]) + b0.z, __uint_as_float(r[8 * j + 3]) + b0.w),
                                        pack2<T>(__uint_as_float(r[8 * j + 4]) + b1.x, __uint_as_float(r[8 * j + 5]) + b1.y),
                                        pack2<T>(__uint_as_float(r[8 * j + 6]) + b1.z, __uint_as_float(r[8 * j + 7]) + b1.w));
                                }
                            }
                        } else {
                            uint32_t pk[16];
#pragma unroll
                            for (int j = 0; j < 16; ++j)
                                pk[j] = valid ? pack2<T>(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])) : 0u;
                            if (valid) {
#pragma unroll
                                for (int j = 0; j < 4; ++j)
                                    *reinterpret_cast<uint4*>(o + c * 32 + j * 8) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                            }
                            // statistics of the STORED values: transpose through shared memory, lane = (pixel half, channel pair)
                            __syncwarp();
#pragma unroll
                            for (int j = 0; j < 4; ++j)
                                *reinterpret_cast<uint4*>(scr + lane * T5_SCR_PITCH + j * 16) = make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
                            __syncwarp();
                            float a0 = 0.f, a1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
                            for (int i = 0; i < 16; ++i) {
                                const int row = half * 16 + ((i + 4 * half) & 15);   // the two halves hit disjoint banks
                                const float2 v = unpack2<T>(*reinterpret_cast<const uint32_t*>(scr + row * T5_SCR_PITCH + pr * 4));
                                a0 += v.x; q0 = fmaf(v.x, v.x, q0);
                                a1 += v.y; q1 = fmaf(v.y, v.y, q1);
                            }
                            s1[c][0] += (double)a0; s2[c][0] += (double)q0;
                            s1[c][1] += (double)a1; s2[c][1] += (double)q1;
                        }
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(T_EMPTY(tsg));
            if (warp == T5_EPI_WARP0 && lane == 0) T5_TRACE(1, 2 * k + 1);
        }
        flush();
    } else {
        // ================= stagers: raw -> activated channel planes =================
        // A thread owns the same (pixel, 8-channel chunk) slots in every job (job = one A-ring stage = one K chunk of one work
        // item).  SAME / CAT2: the raw 16-byte chunks go global -> shared with cp.async straight into their final position in the
        // channel planes (zero-filled outside the image), one whole job ahead of the arithmetic, so HBM latency is paid by the
        // copy engine and not by a register-staged load -> use chain; the GroupNorm affine + SiLU then runs IN PLACE on the
        // thread's own chunks (no cross-thread hand-over until the stage's `full` barrier).  POOL: the 2x2 mean shrinks the data
        // four-fold, so it keeps register staging (8 loads in flight per thread).
        pdl_wait();   // the producer's activations / statistics are complete from here on
        const int ts_ = tid - 32 * T5_STG_WARP0;
        const int nc8 = p.kc >> 3;
        const int l2 = nc8 == 8 ? 3 : (nc8 == 4 ? 2 : 1);
        const int c8 = ts_ & (nc8 - 1), p0 = ts_ >> l2, pstr = T5_STAGE_THREADS >> l2;
        const int DR = pstr / p.pitch, DC = pstr - DR * p.pitch;
        float2* coef = reinterpret_cast<float2*>(smem + p.off_coef);
        const int H = p.H, W = p.W;
        const int Hs = MODE == T5_POOL ? 2 * H : H, Ws = MODE == T5_POOL ? 2 * W : W;
        const int Cs = MODE == T5_CAT2 ? p.cout : p.cin;           // channels of one source tensor
        const uint32_t rowb = (uint32_t)Ws * Cs * 2;
        const int njobs = (it1 - it0) * p.nchunk;

        struct Job { int n, apix, r0, c0, cs, xs; bool ident; const unsigned char* src; };
        auto job_of = [&](int j) {
            Job jb;
            const int item = it0 + j / p.nchunk, ch = j - (j / p.nchunk) * p.nchunk;
            const T5Item it = t5_item(p, item);
            jb.n = it.n;
            jb.xs = it.xs;
            jb.apix = 128 * it.mt_cur + 2 * p.pitch + 2;
            const int q0 = it.m0 * 128 + p0;
            jb.r0 = q0 / p.pitch;
            jb.c0 = q0 - jb.r0 * p.pitch;
            const int cg = ch * p.kc + c8 * 8;                         // first of this thread's 8 input channels
            jb.ident = (MODE == T5_CAT2 && cg < p.cout) || MODE == T5_IDENT;   // `up` half of the concat / a gradient tensor: plain copy
            jb.cs = (MODE == T5_CAT2 && !jb.ident) ? cg - p.cout : cg;
            jb.src = reinterpret_cast<const unsigned char*>((MODE == T5_CAT2 && !jb.ident) ? p.src1 : p.src0) +
                     (size_t)it.n * Hs * Ws * Cs * 2 + (size_t)jb.cs * 2;
            return jb;
        };
        auto stage_ptr = [&](int sa) { return smem + (size_t)sa * p.a_stage_bytes + (size_t)c8 * plane_bytes; };
        // One batch = B slots of this thread, loaded into registers before any of them is processed; two batches alternate, so
        // B..2B 16-byte loads per thread (8 warps: 32-64 KB per SM) are in flight while the previous batch is activated and
        // stored.  The activated chunk goes to shared memory exactly once: UMMA operand reads already use ~85 % of the 128 B/clk
        // shared-memory bandwidth on the N = 32 layers, and a cp.async -> in-place variant (three shared-memory passes per
        // element) measured 2x slower staging for that reason.
        constexpr int B = MODE == T5_POOL ? 1 : 2;   // x 2 alternating batches x 512 threads: 32 KB of loads in flight per SM
        constexpr int NL = MODE == T5_POOL ? 4 : 1;
        struct Batch { uint4 v[B][NL]; int ss[B]; bool ok[B]; };
        struct Cursor { int s, r, c; };
        auto load_batch = [&](const Job& jb, Cursor& cu, Batch& q) {
#pragma unroll
            for (int b = 0; b < B; ++b) {
                const int gy = cu.r - 1, gx = jb.xs + cu.c - 1;
                q.ss[b] = cu.s;
                q.ok[b] = cu.s < jb.apix && (unsigned)gy < (unsigned)H && (unsigned)gx < (unsigned)W;
                if (q.ok[b]) {
                    if constexpr (MODE == T5_POOL) {
                        const unsigned char* base = jb.src + ((size_t)(2 * gy) * rowb + (size_t)(2 * gx) * (Cs * 2));
                        q.v[b][0] = __ldg(reinterpret_cast<const uint4*>(base));
                        q.v[b][1] = __ldg(reinterpret_cast<const uint4*>(base + Cs * 2));
                        q.v[b][2] = __ldg(reinterpret_cast<const uint4*>(base + rowb));
                        q.v[b][3] = __ldg(reinterpret_cast<const uint4*>(base + rowb + Cs * 2));
                    } else {
                        q.v[b][0] = __ldg(reinterpret_cast<const uint4*>(jb.src + ((size_t)gy * rowb + (size_t)gx * (Cs * 2))));
                    }
                }
                cu.s += pstr; cu.r += DR; cu.c += DC;
                if (cu.c >= p.pitch) { cu.c -= p.pitch; cu.r += 1; }
            }
        };
        float2 cf[8];
        auto load_coefs = [&](const Job& jb) {
            if (jb.ident) return;
#pragma unroll
            for (int e = 0; e < 8; ++e) cf[e] = coef[jb.cs + e];
        };
        auto proc_batch = [&](const Job& jb, const Batch& q, unsigned char* dst) {
#pragma unroll
            for (int b = 0; b < B; ++b) {
                if (q.ss[b] >= jb.apix) continue;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (q.ok[b]) {
                    if (jb.ident) {
                        o = q.v[b][0];
                    } else {
                        float yv[8];
                        act8<T>(q.v[b][0], cf, yv);
                        if constexpr (MODE == T5_POOL) {
                            float t[8];
#pragma unroll
                            for (int j = 1; j < 4; ++j) {
                                act8<T>(q.v[b][j], cf, t);
#pragma unroll
                                for (int e = 0; e < 8; ++e) yv[e] += t[e];
                            }
#pragma unroll
                            for (int e = 0; e < 8; ++e) yv[e] *= 0.25f;
                        }
                        o = pack8<T>(yv);
                    }
                }
                *reinterpret_cast<uint4*>(dst + (size_t)q.ss[b] * 16) = o;
            }
        };
        auto ensure_coefs = [&](int n, int& coef_n) {
            if constexpr (MODE == T5_IDENT) return;   // nothing to normalise
            if (n == coef_n) return;
            stager_bar();   // every stager is done with the previous image's coefficients
            const double plane = (double)Hs * Ws;
            for (int c = ts_; c < p.ncoef; c += T5_STAGE_THREADS) {
                float a, b;
                if (MODE == T5_CAT2) {
                    if (p.cf1) { a = __ldg(p.cf1 + (size_t)(n * p.ncoef + c) * 2); b = __ldg(p.cf1 + (size_t)(n * p.ncoef + c) * 2 + 1); }
                    else gn_coef(p.st1, p.g1, p.b1, n, p.ncoef, p.groups1, c, plane, p.eps, a, b);
                } else {
                    if (p.cf0) { a = __ldg(p.cf0 + (size_t)(n * p.ncoef + c) * 2); b = __ldg(p.cf0 + (size_t)(n * p.ncoef + c) * 2 + 1); }
                    else gn_coef(p.st0, p.g0, p.b0, n, p.ncoef, p.groups0, c, plane, p.eps, a, b);
                }
                a *= 0.5f; b *= 0.5f;
                coef[c] = make_float2(a, b);
            }
            coef_n = n;
            stager_bar();
        };

        int coef_n = -1;
        int sa = 0; uint32_t pa = 0;
        for (int j = 0; j < njobs; ++j) {
            if (ts_ == 0) T5_TRACE(2, 4 * j);
            const Job jb = job_of(j);
            Cursor cu{p0, jb.r0, jb.c0};
            Batch q0, q1;
            load_batch(jb, cu, q0);                 // the first loads fly while we wait for the ring stage
            ensure_coefs(jb.n, coef_n);
            load_coefs(jb);
            mbar_wait_relaxed(A_EMPTY(sa), pa ^ 1u);
            if (ts_ == 0) T5_TRACE(2, 4 * j + 1);
            unsigned char* dst = stage_ptr(sa);
#pragma unroll 1
            while (true) {
                const bool m1 = cu.s < jb.apix;
                if (m1) load_batch(jb, cu, q1);
                proc_batch(jb, q0, dst);
                if (!m1) break;
                const bool m0 = cu.s < jb.apix;
                if (m0) load_batch(jb, cu, q0);
                proc_batch(jb, q1, dst);
                if (!m0) break;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the UMMA reads
            mbar_arrive(A_FULL(sa));
            if (ts_ == 0) T5_TRACE(2, 4 * j + 2);
            if (++sa == p.na) { sa = 0; pa ^= 1u; }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == T5_MMA_WARP) {
        __syncwarp();
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(p.tmem_cols));
    }
}

int t5_sm_count() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    return sms;
}

// Geometry / shared-memory plan.  Returns false when the configuration does not fit (caller falls back to mma.sync).
bool t5_plan(T5Args& t, int mode, int ntaps = 0) {
    const int cin = t.cin, cout = t.cout;
    if (cin < 16 || cin % 16 || cout < 32 || cout % 32) return false;
    t.nb = cout <= 128 ? cout : 128;
    if (cout % t.nb || (t.nb != 32 && t.nb != 64 && t.nb != 128 && t.nb != 96)) return false;
    if (t.nb == 96) return false;   // keep N a power of two (TMEM stage arithmetic)
    t.nnb = cout / t.nb;
    const int csrc = mode == T5_CAT2 ? cout : cin;   // channels of one source tensor
    t.ntaps = ntaps ? ntaps : (mode == T5_CONVT ? 1 : 9);   // ntaps = 1 with T5_IDENT: a plain GEMM over pixels (centre tap)
    t.kc = csrc >= 64 ? 64 : csrc;
    if (t.kc != 16 && t.kc != 32 && t.kc != 64) return false;
    if (csrc % t.kc || cin % t.kc) return false;
    t.nchunk = cin / t.kc;
    t.ncoef = csrc;
    t.tw = t.W <= 128 ? t.W : 126;                 // pitch 128 for wide images; one strip = the whole width up to 128 columns
    t.nstrips = (t.W + t.tw - 1) / t.tw;
    t.pitch = t.tw + 2;
    const long long stream_px = (long long)(t.H - 1) * t.pitch + t.tw;
    t.mtiles_img = (int)((stream_px + 127) / 128);
    const int ksteps_total = t.ntaps * (cin / 16);
    // accumulators: double-buffered in TMEM unless K is so long that the epilogue is negligible and M reuse of the streamed
    // weights matters more (wide variant)
    t.ts = ksteps_total >= 576 ? 1 : 2;
    int mt_max = 512 / (t.ts * t.nb);
    for (;; ) {
        if (mt_max < 1) return false;
        const int bands = (t.mtiles_img + mt_max - 1) / mt_max;
        t.mt = (t.mtiles_img + bands - 1) / bands;
        t.bands_img = (t.mtiles_img + t.mt - 1) / t.mt;
        const int apix = 128 * t.mt + 2 * t.pitch + 2;
        const int nc8 = t.kc / 8;
        const int want = nc8 >= 8 ? 1 : 8 / nc8;
        int px = apix;
        while (px % 8 != want) ++px;
        t.plane_px = px;
        t.a_stage_bytes = nc8 * px * 16;
        t.b_stage_bytes = (t.kc / 16) * t.nb * 32;
        const int fixed = t.ncoef * 8 + 4 * 32 * T5_SCR_PITCH + 8 * (4 * T5_MAX_RING + 4) + 16 + 1024;
        // ring depths: at least 2 A chunks and 3 weight tiles, more while shared memory lasts
        int budget = 227 * 1024 - fixed;
        t.na = 2; t.nbs = 3;
        if (t.na * t.a_stage_bytes + t.nbs * t.b_stage_bytes > budget) {
            // first give up channels per chunk (the K loop just gets more, shorter chunks), then M-tiles per item: fewer M-tiles
            // means the two halo rows are staged for fewer output pixels (mt = 2 at pitch 128: 2x staging, mt = 4: 1.5x)
            if (t.kc > 32 && csrc % (t.kc / 2) == 0) { t.kc /= 2; t.nchunk = cin / t.kc; continue; }
            if (mt_max > 1) { mt_max /= 2; t.kc = csrc >= 64 ? 64 : csrc; t.nchunk = cin / t.kc; continue; }
            return false;
        }
        budget -= t.na * t.a_stage_bytes + t.nbs * t.b_stage_bytes;
        while (t.nbs < T5_MAX_RING && t.nbs < 6 && budget >= t.b_stage_bytes) { ++t.nbs; budget -= t.b_stage_bytes; }
        if (t.nchunk > 2 && budget >= t.a_stage_bytes && t.na < T5_MAX_RING) { ++t.na; budget -= t.a_stage_bytes; }
        break;
    }
    int cols = t.ts * t.mt * t.nb, pw = 32;
    while (pw < cols) pw <<= 1;
    if (pw > 512) return false;
    t.tmem_cols = pw;
    t.off_b = (t.na * t.a_stage_bytes + 127) / 128 * 128;
    t.off_coef = t.off_b + t.nbs * t.b_stage_bytes;
    t.off_scr = (t.off_coef + t.ncoef * 8 + 15) / 16 * 16;
    t.off_bar = t.off_scr + 4 * 32 * T5_SCR_PITCH;
    const long long items = (long long)t.N * t.nstrips * t.bands_img * t.nnb;
    if (items > 0x7fffffffLL) return false;
    t.items = (int)items;
    return true;
}

int t5_smem_bytes(const T5Args& t) { return t.off_bar + 8 * (4 * T5_MAX_RING + 4) + 16; }

void t5_trace_dump(const T5Args& t, long long* dev, cudaStream_t st) {
    cudaStreamSynchronize(st);
    static long long h[4 * 512];
    cudaMemcpy(h, dev, sizeof(h), cudaMemcpyDeviceToHost);
    const int items = (int)(((long long)t.items + 0) / (t.items < t5_sm_count() ? t.items : t5_sm_count()));
    long long t0 = h[0];
    for (int i = 0; i < 4 * 512; ++i) if (h[i] && h[i] < t0) t0 = h[i];
    fprintf(stderr, "[t5 trace] cin %d cout %d HxW %dx%d N %d: mt %d nb %d kc %d na %d nbs %d ts %d items %d (~%d per CTA)\n", t.cin, t.cout, t.H, t.W,
            t.N, t.mt, t.nb, t.kc, t.na, t.nbs, t.ts, t.items, items);
    for (int k = 0; k < items + 1 && k < 12; ++k)
        fprintf(stderr, "  item %2d  mma: tmem_free %7lld a_full %7lld done_issue %7lld | epi: t_full %7lld done %7lld | stage: start %7lld loaded %7lld arrived %7lld next %7lld | tma: tap0 %7lld tap8 %7lld\n",
                k, h[4 * k] - t0, h[4 * k + 1] - t0, h[4 * k + 2] - t0, h[512 + 2 * k] - t0, h[512 + 2 * k + 1] - t0, h[1024 + 4 * k] - t0,
                h[1024 + 4 * k + 1] - t0, h[1024 + 4 * k + 2] - t0, h[1024 + 4 * k + 3] - t0, h[1536 + 2 * k] - t0, h[1536 + 2 * k + 1] - t0);
}

template <typename T, int MODE>
int launch_t5(const T5Args& t, cudaStream_t st) {
    auto kern = conv3x3_t5_kernel<T, MODE>;
    static bool done = false;
    if (!done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) { set_error("conv3x3 t5: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return 4; }
        done = true;
    }
    const int sms = t5_sm_count();
    const int grid = t.items < sms ? t.items : sms;
    static long long* trace_buf = nullptr;
    static const bool tracing = getenv("DG_T5_TRACE") != nullptr;
    T5Args tt = t;
    if (tracing) {
        if (trace_buf == nullptr) cudaMalloc(&trace_buf, 4 * 512 * sizeof(long long));
        cudaMemsetAsync(trace_buf, 0, 4 * 512 * sizeof(long long), st);
        tt.trace = trace_buf;
    }
    cudaError_t le = launch_kernel(kern, dim3(grid), dim3(T5_THREADS), (size_t)t5_smem_bytes(t), st, tt);
    if (le != cudaSuccess) { set_error("conv3x3 t5 launch: %s", cudaGetErrorString(le)); return 10; }
    count_launch();
    if (tracing) t5_trace_dump(tt, trace_buf, st);
    return check_launch("conv3x3_t5");
}

template <typename T>
int dispatch_t5(const T5Args& t, int mode, cudaStream_t st) {
    if (mode == T5_SAME) return launch_t5<T, T5_SAME>(t, st);
    if (mode == T5_POOL) return launch_t5<T, T5_POOL>(t, st);
    if (mode == T5_CONVT) return launch_t5<T, T5_CONVT>(t, st);
    return launch_t5<T, T5_CAT2>(t, st);
}
}  // namespace

// path bit 7 (128): do not use this kernel; bit 8 (256): the caller insists on it (tests) -- unsupported is then an error.
int conv3x3_t5_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled) {
    *handled = false;
    const bool forced = (a.path & 256) != 0;
    auto decline = [&](const char* why) {
        if (forced) { set_error("conv3x3 t5: %s", why); return 3; }
        return 0;
    };
    if (a.path & 128) return 0;
    if (a.dtype != DG_F16 && a.dtype != DG_BF16) return decline("needs 16-bit storage");
    const dg_src& s0 = a.src[0];
    if (a.weight_tc == nullptr || a.act_sum != nullptr) return decline("needs the tensor-core weight packing and no act_sum");
    T5Args t;
    memset(&t, 0, sizeof(t));
    int mode;
    if (a.nsrc == 1 && (s0.xform == DG_X_SAME || s0.xform == DG_X_POOL2)) {
        if (s0.stats == nullptr || !s0.silu || s0.scale != nullptr) return decline("source must be GroupNorm + SiLU");
        mode = s0.xform == DG_X_SAME ? T5_SAME : T5_POOL;
        t.cin = s0.channels;
    } else if (a.nsrc == 2 && s0.xform == DG_X_SAME && a.src[1].xform == DG_X_SAME && s0.stats == nullptr && !s0.silu &&
               s0.scale == nullptr) {
        const dg_src& s1 = a.src[1];
        if (s1.stats == nullptr || !s1.silu || s1.scale || s0.channels != a.cout || s1.channels != a.cout)
            return decline("concat must be (identity up C, GroupNorm+SiLU skip C) -> C");
        mode = T5_CAT2;
        t.cin = 2 * a.cout;
        t.src1 = s1.raw; t.st1 = s1.stats; t.g1 = s1.gamma; t.b1 = s1.beta; t.cf1 = s1.coef; t.groups1 = s1.groups;
    } else {
        return decline("source combination not covered");
    }
    if ((reinterpret_cast<uintptr_t>(s0.raw) | reinterpret_cast<uintptr_t>(a.out) | reinterpret_cast<uintptr_t>(a.weight_tc) |
         reinterpret_cast<uintptr_t>(t.src1)) & 15)
        return decline("pointers must be 16-byte aligned");
    t.src0 = s0.raw; t.st0 = s0.stats; t.g0 = s0.gamma; t.b0 = s0.beta; t.cf0 = s0.coef; t.groups0 = s0.groups;
    t.wgt = a.weight_tc;
    t.out = a.out; t.out_stats = a.out_stats;
    t.N = a.N; t.H = a.H; t.W = a.W; t.eps = a.eps;
    t.cout = a.cout;
    // N = 32 with a single-source prologue: a UMMA re-reads its 4 KB A tile for only 32 output channels, and the mma.sync kernel
    // measured on par or faster (enc3.0 0.071 vs 0.100 ms, enc3.3 0.079 vs 0.083 ms at batch 64); the concat conv (K = 576) wins here
    if (!forced && a.cout == 32 && mode != T5_CAT2) return 0;
    if (!t5_plan(t, mode)) return decline("shape does not fit the tcgen05 plan");
    *handled = true;
    return a.dtype == DG_F16 ? dispatch_t5<__half>(t, mode, stream) : dispatch_t5<__nv_bfloat16>(t, mode, stream);
}


// Stand-alone ConvTranspose2d(2,2)+bias of the activated low-resolution source on the tcgen05 kernel (C_up >= 32, any C_low % 16):
// the wide variant's up-convolutions (1024 -> 512 ... 128 -> 64) and upconv4 / upconv3 of the shipped model.  H, W = OUTPUT size.
int convt_t5_launch(const dg_src& s, int dtype, int N, int H, int W, void* out, float eps, int path, cudaStream_t st, bool* handled) {
    *handled = false;
    if (path & 128) return 0;
    if (dtype != DG_F16 && dtype != DG_BF16) return 0;
    if (s.xform != DG_X_CONVT2 || s.ct_w_tc == nullptr || s.ct_b == nullptr || s.stats == nullptr || !s.silu || s.scale) return 0;
    if ((H | W) & 1) return 0;
    if (s.ct_cout < 32 || s.ct_cout % 32 || (4 * s.ct_cout) % 128) return 0;
    if ((reinterpret_cast<uintptr_t>(s.raw) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(s.ct_w_tc) |
         reinterpret_cast<uintptr_t>(s.ct_b)) & 15)
        return 0;
    T5Args t;
    memset(&t, 0, sizeof(t));
    t.src0 = s.raw; t.st0 = s.stats; t.g0 = s.gamma; t.b0 = s.beta; t.cf0 = s.coef; t.groups0 = s.groups;
    t.wgt = s.ct_w_tc; t.bias = s.ct_b;
    t.out = out; t.out_stats = nullptr;
    t.N = N; t.H = H / 2; t.W = W / 2; t.eps = eps;
    t.cin = s.channels;
    t.cout = 4 * s.ct_cout;
    t.cu = s.ct_cout;
    if (!t5_plan(t, T5_CONVT)) return 0;
    *handled = true;
    return dtype == DG_F16 ? dispatch_t5<__half>(t, T5_CONVT, st) : dispatch_t5<__nv_bfloat16>(t, T5_CONVT, st);
}


// ---- data gradient of a 3x3 conv on the tcgen05 kernel (wide variant, BASELINE.json configs[4]) ----------------------------------------
//   dX[n,y,x,ci] = sum_{ky,kx,co} dR[n, y+1-ky, x+1-kx, co] * W[co][ci][ky][kx]   (autograd of src/model.py:93,96 w.r.t. the conv input)
// = conv3x3(dR, flipped / transposed W): ck = channels of dR (GEMM K side), cn = channels of dX (N side, >= 32), wflip_tc_bf16 =
// dg_pack_conv3x3_tc of the fp32 [3][3][ck][cn] taps-flipped weights in DG_BF16.  dR comes as fp32 (converted into `scratch_bf16`,
// N*H*W*ck bf16, by one element-wise kernel) or already as bf16 (dR_bf16, e.g. gn_bwd_apply's second output form).
namespace {
__global__ void __launch_bounds__(256) cvt_f32_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n8) {
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n8; i += (size_t)gridDim.x * 256) {
        const float4 a = __ldg(reinterpret_cast<const float4*>(in) + 2 * i), b = __ldg(reinterpret_cast<const float4*>(in) + 2 * i + 1);
        reinterpret_cast<uint4*>(out)[i] = make_uint4(pack2<__nv_bfloat16>(a.x, a.y), pack2<__nv_bfloat16>(a.z, a.w),
                                                      pack2<__nv_bfloat16>(b.x, b.y), pack2<__nv_bfloat16>(b.z, b.w));
    }
}
}  // namespace

// ---- data gradient of ConvTranspose2d(k=2, s=2) on the tcgen05 kernel (wide variant) -------------------------------------------------
//   dLow[n,i,j,ci] = sum_{a,b,co} dUp[n, 2i+a, 2j+b, co] * Wt[ci][co][a][b]     (autograd of src/model.py:47-53 w.r.t. its input)
// = a plain GEMM over low-resolution pixels with K = (position, co) = 4 Cu and N = ci: the up half of the concat gradient is gathered
// per position into a bf16 tensor D [N,Hl,Wl,4 Cu] (one element-wise kernel), then T5_IDENT with ONE tap.  w2_tc_bf16 = the [4 Cu][Cl]
// matrix W2[(2a+b) Cu + co][ci] = Wt[ci][co][a][b] in the [K/16][k-half][N][8] packing (dg_pack_convt2x2_tc of its re-blocked view).
namespace {
__global__ void __launch_bounds__(256) up_half_pos_bf16_kernel(const float* __restrict__ dCat, int stride, __nv_bfloat16* __restrict__ D,
                                                               int N, int Hl, int Wl, int Cu) {
    const int c8n = Cu >> 3;
    const size_t items = (size_t)N * Hl * Wl * 4 * c8n;
    for (size_t e = (size_t)blockIdx.x * 256 + threadIdx.x; e < items; e += (size_t)gridDim.x * 256) {
        const int c8 = (int)(e % c8n);
        const size_t r = e / c8n;
        const int pos = (int)(r & 3);
        const size_t pix = r >> 2;                  // (n*Hl + i)*Wl + j
        const int j = (int)(pix % Wl);
        const size_t row = pix / Wl;                // n*Hl + i
        const int i = (int)(row % Hl);
        const size_t n = row / Hl;
        const float* q = dCat + ((n * (2 * Hl) + 2 * i + (pos >> 1)) * (size_t)(2 * Wl) + 2 * j + (pos & 1)) * stride + c8 * 8;
        const float4 a = __ldg(reinterpret_cast<const float4*>(q)), b = __ldg(reinterpret_cast<const float4*>(q) + 1);
        *reinterpret_cast<uint4*>(D + (pix * 4 + pos) * Cu + c8 * 8) =
            make_uint4(pack2<__nv_bfloat16>(a.x, a.y), pack2<__nv_bfloat16>(a.z, a.w), pack2<__nv_bfloat16>(b.x, b.y), pack2<__nv_bfloat16>(b.z, b.w));
    }
}
}  // namespace

int convt_dgrad_t5_launch(const float* dCat, int stride, void* scratch_bf16, const void* w2_tc_bf16, float* dLow, int N, int H, int W,
                          int Cl, int Cu, cudaStream_t st, bool* handled) {
    *handled = false;
    if (dCat == nullptr || scratch_bf16 == nullptr || w2_tc_bf16 == nullptr || dLow == nullptr || ((H | W) & 1)) return 0;
    if ((Cu & 7) || (stride & 3) ||
        ((reinterpret_cast<uintptr_t>(dCat) | reinterpret_cast<uintptr_t>(scratch_bf16) | reinterpret_cast<uintptr_t>(w2_tc_bf16) |
          reinterpret_cast<uintptr_t>(dLow)) & 15))
        return 0;
    T5Args t;
    memset(&t, 0, sizeof(t));
    t.src0 = scratch_bf16;
    t.wgt = w2_tc_bf16;
    t.out = dLow; t.out_stats = nullptr;
    t.N = N; t.H = H / 2; t.W = W / 2; t.eps = 1e-5f;
    t.cin = 4 * Cu;
    t.cout = Cl;
    if (!t5_plan(t, T5_IDENT, 1)) return 0;
    const size_t items = (size_t)N * (H / 2) * (W / 2) * 4 * (Cu / 8);
    size_t blocks = (items + 255) / 256;
    if (blocks > 148 * 8) blocks = 148 * 8;
    up_half_pos_bf16_kernel<<<(unsigned)blocks, 256, 0, st>>>(dCat, stride, static_cast<__nv_bfloat16*>(scratch_bf16), N, H / 2, W / 2, Cu);
    count_launch();
    int rc = check_launch("up_half_pos_bf16");
    if (rc) return rc;
    *handled = true;
    return launch_t5<__nv_bfloat16, T5_IDENT>(t, st);
}

int conv3x3_dgrad_t5_launch(const float* dR, const void* dR_bf16, void* scratch_bf16, const void* wflip_tc_bf16, float* out, int N,
                            int H, int W, int ck, int cn, cudaStream_t st, bool* handled) {
    *handled = false;
    if (wflip_tc_bf16 == nullptr || out == nullptr || (dR_bf16 == nullptr && (dR == nullptr || scratch_bf16 == nullptr))) return 0;
    const void* src = dR_bf16 != nullptr ? dR_bf16 : scratch_bf16;
    if ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(wflip_tc_bf16) |
         reinterpret_cast<uintptr_t>(dR)) & 15)
        return 0;
    T5Args t;
    memset(&t, 0, sizeof(t));
    t.src0 = src;
    t.wgt = wflip_tc_bf16;
    t.out = out; t.out_stats = nullptr;
    t.N = N; t.H = H; t.W = W; t.eps = 1e-5f;
    t.cin = ck;
    t.cout = cn;
    if (!t5_plan(t, T5_IDENT)) return 0;
    if (dR_bf16 == nullptr) {
        const size_t n8 = (size_t)N * H * W * ck / 8;   // ck % 16 == 0 (t5_plan)
        size_t blocks = (n8 + 255) / 256;
        if (blocks > 148 * 8) blocks = 148 * 8;
        cvt_f32_bf16_kernel<<<(unsigned)blocks, 256, 0, st>>>(dR, static_cast<__nv_bfloat16*>(scratch_bf16), n8);
        count_launch();
        int rc = check_launch("cvt_f32_bf16");
        if (rc) return rc;
    }
    *handled = true;
    return launch_t5<__nv_bfloat16, T5_IDENT>(t, st);
}

}  // namespace dg
