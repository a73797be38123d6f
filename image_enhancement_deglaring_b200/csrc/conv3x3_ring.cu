// Persistent, TMA-fed 3x3 conv for the level-1 layers of LightweightUNet(features_start=8): 8 -> 8 channels at full resolution
// (enc1.3, dec1.3; src/model.py:96 with the GroupNorm + SiLU of :94-95 applied on load) -- 16 bytes per pixel in and out, the
// layers that hold most of the network's HBM bytes.
//
// What changes against conv3x3_tc.cu (one CTA per tile, LDG -> registers -> activate -> shared memory, 4-8 CTAs per SM hiding
// each other's load latency; ncu: 53 % issue utilisation, top stall `barrier`):
//   * one persistent CTA walks a contiguous range of 16 x 64 tiles; GroupNorm coefficients are rebuilt once per image and the
//     tap weights (B fragments) live in registers for the CTA's whole life instead of once per tile;
//   * the RAW halo tile (18 x 66 pixels x 16 B) is fetched by TMA -- one cp.async.bulk.tensor per tile, issued by one thread two
//     tiles ahead into a 3-stage shared-memory ring, completion on an mbarrier, out-of-image pixels zero-filled by the copy
//     engine -- so no thread computes a load address or tests a bound, and HBM latency never sits in a warp's dependency chain;
//   * the tile lands in shared memory already in the 16-byte-per-pixel plane layout ldmatrix reads, so GroupNorm affine + SiLU
//     run IN PLACE (LDS.128 -> FFMA / MUFU.TANH -> STS.128), one __syncthreads per tile;
//   * the tensor-core part is the ROLL scheme of conv3x3_tc.cu (a warp owns 8 consecutive output rows of a 16-pixel segment,
//     A fragments loaded once per input row and fed to the three output rows that use them), statistics accumulate in
//     registers across the tiles of an image and are flushed once per image per CTA.
#include "tc_common.cuh"
#include "tma.cuh"

namespace dg {

namespace {

constexpr int RG_TH = 16, RG_TW = 64, RG_PH = RG_TH + 2, RG_PW = RG_TW + 2;
constexpr int RG_THREADS = 256, RG_WARPS = 8, RG_NS = 3;
constexpr int RG_TILE_BYTES = RG_PH * RG_PW * 16;                    // 19008
constexpr int RG_STAGE_BYTES = (RG_TILE_BYTES + 127) / 128 * 128;    // 19072
constexpr int RG_C = 8;
constexpr int RG_RW = 8;     // output rows per warp: warp = (segment 0..3, row block 0..1)
constexpr int RG_OFF_COEF = RG_NS * RG_STAGE_BYTES;
constexpr int RG_OFF_STAT = RG_OFF_COEF + RG_C * 8;
constexpr int RG_OFF_BAR = RG_OFF_STAT + RG_WARPS * RG_C * 2 * 8;
constexpr int RG_SMEM = RG_OFF_BAR + RG_NS * 8 + 64;

struct RingArgs {
    CUtensorMap tmap;
    const double* st; const float* g; const float* b; const float* cf; int groups;
    const void* wgt; void* out; double* out_stats;
    int N, H, W; float eps;
    int tiles_x, tiles_y, total;
};

__device__ __forceinline__ void rg_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void rg_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rg_mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done = 0;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) return;
    const long long t0 = clock64();
    for (uint32_t spin = 1; !done; ++spin) {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if ((spin & 255u) == 0 && clock64() - t0 > 8000000000LL) __trap();   // a protocol error must not hang the GPU
    }
}

template <typename T>
__global__ void __launch_bounds__(RG_THREADS, 3) conv8_ring_kernel(const __grid_constant__ RingArgs p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    float2* coef = reinterpret_cast<float2*>(smem + RG_OFF_COEF);
    double* statd = reinterpret_cast<double*>(smem + RG_OFF_STAT);
    const uint32_t bar0 = smem_u32(smem + RG_OFF_BAR);
    const uint32_t act0 = smem_u32(smem);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int seg = warp & 3, rb = warp >> 2;
    const int H = p.H, W = p.W;

    pdl_launch_dependents();
    if (tid == 0) {
        for (int s = 0; s < RG_NS; ++s) rg_mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        tma_prefetch_desc(&p.tmap);
    }
    // tap weights as B fragments, for the whole life of the CTA: bw[tap] = W[tap][ci = 2 (lane & 3) (+1)][co = lane >> 2]
    uint32_t bw[9];
    {
        const unsigned char* wg = reinterpret_cast<const unsigned char*>(p.wgt);
#pragma unroll
        for (int t = 0; t < 9; ++t)
            bw[t] = __ldg(reinterpret_cast<const uint32_t*>(wg + ((size_t)((t >> 1) * 2 + (t & 1)) * RG_C + (lane >> 2)) * 16 + (lane & 3) * 4));
    }
    __syncthreads();

    const int t0 = (int)((long long)p.total * blockIdx.x / gridDim.x);
    const int t1 = (int)((long long)p.total * (blockIdx.x + 1) / gridDim.x);
    const int per_img = p.tiles_x * p.tiles_y;
    auto tile_pos = [&](int tile, int& n, int& y0, int& x0) {
        n = tile / per_img;
        const int r = tile - n * per_img;
        const int ty = r / p.tiles_x;
        y0 = ty * RG_TH;
        x0 = (r - ty * p.tiles_x) * RG_TW;
    };
    auto issue = [&](int tile, int stage) {   // one thread: arm the barrier, start the tensor copy of the raw halo tile
        int n, y0, x0;
        tile_pos(tile, n, y0, x0);
        rg_mbar_expect_tx(bar0 + 8 * stage, RG_TILE_BYTES);
        tma_load_3d(act0 + stage * RG_STAGE_BYTES, &p.tmap, 2 * (x0 - 1), y0 - 1, n, bar0 + 8 * stage);
    };

    pdl_wait();   // the producer's activations / statistics are complete from here on
    if (tid == 0)
        for (int k = 0; k < RG_NS && t0 + k < t1; ++k) issue(t0 + k, k);

    // Statistics: fp32 partial sums over ONE tile per thread (a fixed order, so they depend on the tile only), accumulated in
    // double across the CTA's tiles of an image -- the result is independent of how tiles are distributed over CTAs / batches up
    // to double rounding, which keeps the network's output batch-invariant (tests: tiled == per-tile forward, bit for bit).
    double d1[2] = {0.0, 0.0}, d2[2] = {0.0, 0.0};
    int cur_n = -1;
    auto flush_stats = [&](int n) {
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            double a = d1[k], b = d2[k];
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                a += __shfl_xor_sync(0xffffffffu, a, o);
                b += __shfl_xor_sync(0xffffffffu, b, o);
            }
            if (lane < 4) {
                statd[(warp * RG_C + 2 * lane + k) * 2] = a;
                statd[(warp * RG_C + 2 * lane + k) * 2 + 1] = b;
            }
            d1[k] = d2[k] = 0.0;
        }
        __syncthreads();
        if (tid < 2 * RG_C && p.out_stats != nullptr) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < RG_WARPS; ++w) t += statd[w * RG_C * 2 + tid];
            atomicAdd(p.out_stats + (size_t)n * RG_C * 2 + tid, t);
        }
        __syncthreads();
    };

    T* outp = reinterpret_cast<T*>(p.out);
    for (int k = 0; t0 + k < t1; ++k) {
        const int tile = t0 + k, stage = k % RG_NS;
        int n, y0, x0;
        tile_pos(tile, n, y0, x0);
        if (n != cur_n) {
            if (cur_n >= 0) flush_stats(cur_n);
            if (tid < RG_C) {
                float a, b;
                if (p.cf) { a = __ldg(p.cf + (size_t)(n * RG_C + tid) * 2); b = __ldg(p.cf + (size_t)(n * RG_C + tid) * 2 + 1); }
                else gn_coef(p.st, p.g, p.b, n, RG_C, p.groups, tid, (double)H * W, p.eps, a, b);
                a *= 0.5f; b *= 0.5f;
                coef[tid] = make_float2(a, b);
            }
            cur_n = n;
            __syncthreads();
        }
        // ---- (1) the raw tile has landed: GroupNorm affine + SiLU in place ----------------------------------------------------
        rg_mbar_wait(bar0 + 8 * stage, (uint32_t)((k / RG_NS) & 1));
        unsigned char* act = smem + stage * RG_STAGE_BYTES;
        {
            float2 cf[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) cf[e] = coef[e];
            const bool interior = y0 >= 1 && x0 >= 1 && y0 + RG_TH + 1 <= H && x0 + RG_TW + 1 <= W;
            constexpr int NPIX = RG_PH * RG_PW;
            constexpr int SLOTS = (NPIX + RG_THREADS - 1) / RG_THREADS;   // 5
            uint4 q[SLOTS];
#pragma unroll
            for (int i = 0; i < SLOTS; ++i) {
                const int px = tid + i * RG_THREADS;
                if (px < NPIX) q[i] = *reinterpret_cast<const uint4*>(act + px * 16);
            }
#pragma unroll
            for (int i = 0; i < SLOTS; ++i) {
                const int px = tid + i * RG_THREADS;
                if (px >= NPIX) continue;
                bool ok = true;
                if (!interior) {   // the conv zero-pads the ACTIVATED tensor: out-of-image pixels must stay exactly zero
                    const int r = px / RG_PW, c = px - r * RG_PW;
                    ok = (unsigned)(y0 - 1 + r) < (unsigned)H && (unsigned)(x0 - 1 + c) < (unsigned)W;
                }
                if (ok) {
                    float yv[8];
                    act8<T>(q[i], cf, yv);
                    *reinterpret_cast<uint4*>(act + px * 16) = pack8<T>(yv);
                }
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // our generic-proxy writes vs the TMA refill of this stage later on
        __syncthreads();   // activated tile visible; every warp is also done with the previous tile's MMAs ...
        if (tid == 0 && k >= 1 && tile - 1 + RG_NS < t1) issue(tile - 1 + RG_NS, (k - 1) % RG_NS);   // ... so its stage can be refilled

        // ---- (2) 9 shifted GEMMs, ROLL: input row r of the warp's block feeds output rows r-2 .. r ---------------------------
        float acc[RG_RW][4];
#pragma unroll
        for (int y = 0; y < RG_RW; ++y) acc[y][0] = acc[y][1] = acc[y][2] = acc[y][3] = 0.f;
        const uint32_t a_base = act0 + stage * RG_STAGE_BYTES + (uint32_t)(((rb * RG_RW) * RG_PW + seg * 16 + (lane & 15)) * 16);
#pragma unroll
        for (int r = 0; r < RG_RW + 2; ++r) {
            const uint32_t a_row = a_base + (uint32_t)(r * RG_PW * 16);
            uint32_t f0, f1, f2, f3, g0, g1;
            ldsm_x4(a_row + (lane >> 4) * 16, f0, f1, f2, f3);   // lanes 0-15: kx = 0, lanes 16-31: kx = 1 (next pixel)
            ldsm_x2(a_row + 32, g0, g1);                          // kx = 2
#pragma unroll
            for (int ky = 0; ky < 3; ++ky) {
                const int y = r - ky;
                if (y < 0 || y >= RG_RW) continue;
                mma16816<T>(acc[y], f0, f1, f2, f3, bw[ky * 3], bw[ky * 3 + 1]);
                mma16808<T>(acc[y], g0, g1, bw[ky * 3 + 2]);
            }
        }
        // ---- (3) epilogue: round, store NHWC, statistics from the fp32 accumulators ------------------------------------------
        float s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f};
        const bool full = (y0 + RG_TH <= H) && (x0 + RG_TW <= W);
        const int gx = x0 + seg * 16 + (lane >> 2);
        const uint32_t orow = (uint32_t)W * RG_C;
        T* obase = outp + ((size_t)(n * H + y0 + rb * RG_RW) * W + gx) * RG_C + 2 * (lane & 3);
        auto epilogue = [&](auto full_c) {
            constexpr bool FULL = decltype(full_c)::value;
#pragma unroll
            for (int y = 0; y < RG_RW; ++y) {
                const int gy = y0 + rb * RG_RW + y;
                T* o = obase + (uint32_t)y * orow;
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool ok = FULL || (gy < H && gx + 8 * hf < W);
                    const float v0 = ok ? acc[y][2 * hf] : 0.f, v1 = ok ? acc[y][2 * hf + 1] : 0.f;
                    if (ok) *reinterpret_cast<uint32_t*>(o + hf * 8 * RG_C) = pack2<T>(v0, v1);
                    s1[0] += v0; s2[0] = fmaf(v0, v0, s2[0]);
                    s1[1] += v1; s2[1] = fmaf(v1, v1, s2[1]);
                }
            }
        };
        if (full) epilogue(std::true_type{});
        else epilogue(std::false_type{});
        d1[0] += (double)s1[0]; d1[1] += (double)s1[1];
        d2[0] += (double)s2[0]; d2[1] += (double)s2[1];
    }
    if (cur_n >= 0) flush_stats(cur_n);
}

template <typename T>
int launch_ring(const RingArgs& a, cudaStream_t st) {
    auto kern = conv8_ring_kernel<T>;
    static bool done = false;
    if (!done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, RG_SMEM);
        if (e != cudaSuccess) { set_error("conv8 ring: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return 4; }
        done = true;
    }
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    int grid = 3 * sms;
    if (grid > a.total) grid = a.total;
    cudaError_t le = launch_kernel(kern, dim3(grid), dim3(RG_THREADS), (size_t)RG_SMEM, st, a);
    if (le != cudaSuccess) { set_error("conv8 ring launch: %s", cudaGetErrorString(le)); return 10; }
    count_launch();
    return check_launch("conv8_ring");
}

}  // namespace

// path bit 9 (512): do not use this kernel (A/B against conv3x3_tc.cu)
int conv3x3_ring_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled) {
    *handled = false;
    if (a.path & 512) return 0;
    if (a.dtype != DG_F16 && a.dtype != DG_BF16) return 0;
    if (a.weight_tc == nullptr || a.act_sum != nullptr || a.nsrc != 1 || a.cout != RG_C) return 0;
    const dg_src& s0 = a.src[0];
    if (s0.xform != DG_X_SAME || s0.channels != RG_C || s0.stats == nullptr || !s0.silu || s0.scale != nullptr) return 0;
    if ((reinterpret_cast<uintptr_t>(s0.raw) | reinterpret_cast<uintptr_t>(a.out) | reinterpret_cast<uintptr_t>(a.weight_tc)) & 15) return 0;
    RingArgs r;
    memset(&r, 0, sizeof(r));
    if (!tma_map_nhwc16(&r.tmap, s0.raw, a.N, a.H, a.W, RG_PW, RG_PH)) return 0;   // no driver entry point: per-tile kernel
    r.st = s0.stats; r.g = s0.gamma; r.b = s0.beta; r.cf = s0.coef; r.groups = s0.groups;
    r.wgt = a.weight_tc; r.out = a.out; r.out_stats = a.out_stats;
    r.N = a.N; r.H = a.H; r.W = a.W; r.eps = a.eps;
    r.tiles_x = (a.W + RG_TW - 1) / RG_TW;
    r.tiles_y = (a.H + RG_TH - 1) / RG_TH;
    const long long total = (long long)r.tiles_x * r.tiles_y * a.N;
    if (total > 0x7fffffffLL) return 0;
    r.total = (int)total;
    *handled = true;
    return a.dtype == DG_F16 ? launch_ring<__half>(r, stream) : launch_ring<__nv_bfloat16>(r, stream);
}

}  // namespace dg
