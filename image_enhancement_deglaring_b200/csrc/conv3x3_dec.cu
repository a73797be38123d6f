// up1 + dec1.0 of LightweightUNet(features_start=8) as ONE persistent TMA-fed kernel with the ConvTranspose folded into the conv:
//     y = Conv3x3( cat( ConvTranspose2d(16 -> 8, k=2, s=2)(act(low)) + b , act(skip) ) )        src/model.py:47-53, :116-128, :93
// (act = GroupNorm affine + SiLU of the producing blocks, applied on load).
//
// The transposed conv is linear and has stride 2 = kernel 2, so every up-sampled pixel depends on exactly ONE low-resolution pixel:
//     up[2i+a, 2j+b, co] = b[co] + sum_ci low[i, j, ci] Wt[ci, co, a, b].
// Substituting it into the 3x3 conv, an output pixel of parity class (py, px) = (y & 1, x & 1) sees its 3x3 window of `up` as a
// 2x2 window of LOW-resolution pixels, with composite weights
//     Wc[py][px][ti][tj][ci][o] = sum over the taps (ky, kx) that land on low pixel (i + ti - 1 + py, j + tj - 1 + px)
//                                 of sum_co Wt[ci, co, a(ky), b(kx)] W3[o, co, ky, kx],
// i.e. the `up` half of the concat conv is four 16-channel taps (K = 64) instead of nine 8-channel taps on a tensor that would
// first have to be computed, scattered into shared memory and padded.  Neither `up` nor the concat exists anywhere -- not in HBM
// and not in shared memory; the round-1 kernel (conv3x3_tc.cu MODE_UPCAT) spent more instructions on the transposed-conv GEMM,
// its masked scatter and the extra barrier than on the conv itself (178.8 M warp instructions, 6 % of them HMMA).
// The ConvTranspose bias contributes sum over the taps INSIDE the image of sum_co W3[o, co, ky, kx] b[co]: a constant per output
// channel in the interior (accumulator initial value), corrected on the one-pixel image border.  The zero padding of the concat
// falls out of the zero-filled low-resolution halo (outside pixels stay exactly zero after the masked activation).
//
// Structure as in conv3x3_ring.cu: persistent CTAs over 16 x 64 output tiles, raw halo tiles of BOTH sources fetched by TMA into a
// 2-stage ring (one mbarrier per stage), activation into two small plane buffers (skip: de-interleaved by column parity so that
// the stride-2 pixel sets of a parity class are contiguous ldmatrix rows), mma.sync m16n8k16 with all weights in registers,
// statistics per tile in fp32 and across tiles in double.
#include "tc_common.cuh"
#include "tma.cuh"

namespace dg {

namespace {

constexpr int DC_TH = 16, DC_TW = 64, DC_PH = DC_TH + 2, DC_PW = DC_TW + 2;        // skip halo tile 18 x 66
constexpr int DC_LH = DC_TH / 2 + 2, DC_LW = DC_TW / 2 + 2;                        // low halo tile 10 x 34
constexpr int DC_THREADS = 256, DC_WARPS = 8, DC_NS = 2;
constexpr int DC_CU = 8, DC_CL = 16;
constexpr int DC_SRAW = DC_PH * DC_PW * 16;                                        // 19008
constexpr int DC_LRAW = DC_LH * DC_LW * 32;                                        // 10880
constexpr int DC_OFF_LRAW = (DC_SRAW + 127) / 128 * 128;                           // 19072
constexpr int DC_STAGE = DC_OFF_LRAW + DC_LRAW;                                    // 29952
constexpr int DC_SW = 34;                                                          // half-columns per row of a parity plane
constexpr int DC_SPLANE = DC_PH * DC_SW * 16;                                      // 9792 == 64 (mod 128): the two planes fill all banks
constexpr int DC_LPLANE = DC_LH * DC_LW * 16;                                      // 5440
constexpr int DC_OFF_SACT = DC_NS * DC_STAGE;
constexpr int DC_OFF_LACT = DC_OFF_SACT + 2 * DC_SPLANE;
constexpr int DC_OFF_COEF = DC_OFF_LACT + 2 * DC_LPLANE;
constexpr int DC_OFF_BK = DC_OFF_COEF + (DC_CL + DC_CU) * 8;
constexpr int DC_OFF_BC = DC_OFF_BK + 9 * DC_CU * 4;                                // border corrections [8 kinds][CU]
constexpr int DC_OFF_STAT = DC_OFF_BC + 8 * DC_CU * 4;
constexpr int DC_OFF_BAR = DC_OFF_STAT + DC_WARPS * DC_CU * 2 * 8;
constexpr int DC_SMEM = DC_OFF_BAR + DC_NS * 8 + 64;
// packed weight blob (dg_pack_dec_composite): composite B tiles, skip B tiles, bias-per-tap table
constexpr int DC_COMP_BYTES = 16 * 2 * DC_CU * 16;     // [class*4 + tap][k-half][o][8 ci]
constexpr int DC_SKIPW_BYTES = 9 * DC_CU * 16;         // [tap][o][8 cs]
constexpr int DC_BLOB_BYTES = DC_COMP_BYTES + DC_SKIPW_BYTES + 9 * DC_CU * 4;

struct DecArgs {
    CUtensorMap tmap_skip, tmap_low;
    const double* st_l; const float* g_l; const float* b_l; int groups_l;
    const double* st_s; const float* g_s; const float* b_s; int groups_s;
    const void* blob; void* out; double* out_stats;
    int N, H, W; float eps;
    int tiles_x, tiles_y, total;
};

__device__ __forceinline__ void dc_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void dc_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void dc_mbar_wait(uint32_t bar, uint32_t parity) {
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
__global__ void __launch_bounds__(DC_THREADS, 2) dec8_ring_kernel(const __grid_constant__ DecArgs p) {
    extern __shared__ __align__(1024) unsigned char smem[];
    unsigned char* sact = smem + DC_OFF_SACT;
    unsigned char* lact = smem + DC_OFF_LACT;
    float2* coef = reinterpret_cast<float2*>(smem + DC_OFF_COEF);      // [0, 16): low channels, [16, 24): skip channels
    float* bk = reinterpret_cast<float*>(smem + DC_OFF_BK);            // [ky*3 + kx][o]
    float* bcorr = reinterpret_cast<float*>(smem + DC_OFF_BC);         // bias of the taps a border pixel loses: rows, columns, corners
    double* statd = reinterpret_cast<double*>(smem + DC_OFF_STAT);
    const uint32_t bar0 = smem_u32(smem + DC_OFF_BAR);
    const uint32_t smem0 = smem_u32(smem);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cb = warp & 1, rb = warp >> 1;      // warp tile: output rows 4 rb .. 4 rb + 3, columns 32 cb .. 32 cb + 31
    const int H = p.H, W = p.W, Hl = H >> 1, Wl = W >> 1;

    pdl_launch_dependents();
    if (tid == 0) {
        for (int s = 0; s < DC_NS; ++s) dc_mbar_init(bar0 + 8 * s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        tma_prefetch_desc(&p.tmap_skip);
        tma_prefetch_desc(&p.tmap_low);
    }
    // ---- weights in registers for the life of the CTA ---------------------------------------------------------------------
    // composite taps: bc[class = py*2 + px][tap = ti*2 + tj][k-half] = Wc[..][ci = 8*kh + 2 (lane & 3) (+1)][o = lane >> 2]
    uint32_t bc[4][4][2], bs[9];
    {
        const unsigned char* blob = reinterpret_cast<const unsigned char*>(p.blob);
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
                for (int kh = 0; kh < 2; ++kh)
                    bc[c][t][kh] = __ldg(reinterpret_cast<const uint32_t*>(blob + ((size_t)(((c * 4 + t) * 2 + kh) * DC_CU + (lane >> 2))) * 16 + (lane & 3) * 4));
#pragma unroll
        for (int t = 0; t < 9; ++t)
            bs[t] = __ldg(reinterpret_cast<const uint32_t*>(blob + DC_COMP_BYTES + ((size_t)(t * DC_CU + (lane >> 2))) * 16 + (lane & 3) * 4));
        if (tid < 9 * DC_CU) bk[tid] = __ldg(reinterpret_cast<const float*>(blob + DC_COMP_BYTES + DC_SKIPW_BYTES) + tid);
    }
    __syncthreads();
    if (tid < 8 * DC_CU) {
        const int kind = tid / DC_CU, o = tid - kind * DC_CU;
        float v;
        if (kind == 0) v = bk[0 * DC_CU + o] + bk[1 * DC_CU + o] + bk[2 * DC_CU + o];          // top row of taps (ky = 0)
        else if (kind == 1) v = bk[6 * DC_CU + o] + bk[7 * DC_CU + o] + bk[8 * DC_CU + o];     // bottom row (ky = 2)
        else if (kind == 2) v = bk[0 * DC_CU + o] + bk[3 * DC_CU + o] + bk[6 * DC_CU + o];     // left column (kx = 0)
        else if (kind == 3) v = bk[2 * DC_CU + o] + bk[5 * DC_CU + o] + bk[8 * DC_CU + o];     // right column (kx = 2)
        else v = bk[(kind == 4 ? 0 : kind == 5 ? 2 : kind == 6 ? 6 : 8) * DC_CU + o];          // corners, counted twice above
        bcorr[tid] = v;
    }
    __syncthreads();
    // ConvTranspose bias through all nine taps: the interior value of the accumulator's initial state (channels 2 (lane&3), +1)
    float btot[2] = {0.f, 0.f};
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        btot[0] += bk[t * DC_CU + 2 * (lane & 3)];
        btot[1] += bk[t * DC_CU + 2 * (lane & 3) + 1];
    }

    const int t0 = (int)((long long)p.total * blockIdx.x / gridDim.x);
    const int t1 = (int)((long long)p.total * (blockIdx.x + 1) / gridDim.x);
    const int per_img = p.tiles_x * p.tiles_y;
    auto tile_pos = [&](int tile, int& n, int& y0, int& x0) {
        n = tile / per_img;
        const int r = tile - n * per_img;
        const int ty = r / p.tiles_x;
        y0 = ty * DC_TH;
        x0 = (r - ty * p.tiles_x) * DC_TW;
    };
    auto issue = [&](int tile, int stage) {   // one thread: both raw halo tiles of a work item, one barrier
        int n, y0, x0;
        tile_pos(tile, n, y0, x0);
        dc_mbar_expect_tx(bar0 + 8 * stage, DC_SRAW + DC_LRAW);
        tma_load_3d(smem0 + stage * DC_STAGE, &p.tmap_skip, 2 * (x0 - 1), y0 - 1, n, bar0 + 8 * stage);
        tma_load_3d(smem0 + stage * DC_STAGE + DC_OFF_LRAW, &p.tmap_low, 4 * ((x0 >> 1) - 1), (y0 >> 1) - 1, n, bar0 + 8 * stage);
    };

    pdl_wait();   // the producers' activations / statistics are complete from here on
    if (tid == 0)
        for (int k = 0; k < DC_NS && t0 + k < t1; ++k) issue(t0 + k, k);

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
                statd[(warp * DC_CU + 2 * lane + k) * 2] = a;
                statd[(warp * DC_CU + 2 * lane + k) * 2 + 1] = b;
            }
            d1[k] = d2[k] = 0.0;
        }
        __syncthreads();
        if (tid < 2 * DC_CU && p.out_stats != nullptr) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < DC_WARPS; ++w) t += statd[w * DC_CU * 2 + tid];
            atomicAdd(p.out_stats + (size_t)n * DC_CU * 2 + tid, t);
        }
        __syncthreads();
    };

    T* outp = reinterpret_cast<T*>(p.out);
    const uint32_t sact_u = smem_u32(sact), lact_u = smem_u32(lact);
    for (int k = 0; t0 + k < t1; ++k) {
        const int tile = t0 + k, stage = k % DC_NS;
        int n, y0, x0;
        tile_pos(tile, n, y0, x0);
        if (n != cur_n) {
            if (cur_n >= 0) flush_stats(cur_n);
            if (tid < DC_CL + DC_CU) {
                float a, b;
                if (tid < DC_CL) gn_coef(p.st_l, p.g_l, p.b_l, n, DC_CL, p.groups_l, tid, (double)Hl * Wl, p.eps, a, b);
                else gn_coef(p.st_s, p.g_s, p.b_s, n, DC_CU, p.groups_s, tid - DC_CL, (double)H * W, p.eps, a, b);
                a *= 0.5f; b *= 0.5f;
                coef[tid] = make_float2(a, b);
            }
            cur_n = n;
            __syncthreads();
        }
        // ---- (1) raw tiles have landed: activate into the plane buffers -------------------------------------------------------
        dc_mbar_wait(bar0 + 8 * stage, (uint32_t)((k / DC_NS) & 1));
        const unsigned char* sraw = smem + stage * DC_STAGE;
        const unsigned char* lraw = sraw + DC_OFF_LRAW;
        const bool interior = y0 >= 2 && x0 >= 2 && y0 + DC_TH + 2 <= H && x0 + DC_TW + 2 <= W;
        {   // skip: 18 x 66 pixels, de-interleaved by column parity (global x = x0 - 1 + c; x0 is even)
            float2 cf[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) cf[e] = coef[DC_CL + e];
            constexpr int NPIX = DC_PH * DC_PW;
            constexpr int SLOTS = (NPIX + DC_THREADS - 1) / DC_THREADS;   // 5
            uint4 q[SLOTS];
#pragma unroll
            for (int i = 0; i < SLOTS; ++i) {
                const int px = tid + i * DC_THREADS;
                if (px < NPIX) q[i] = *reinterpret_cast<const uint4*>(sraw + px * 16);
            }
#pragma unroll
            for (int i = 0; i < SLOTS; ++i) {
                const int px = tid + i * DC_THREADS;
                if (px >= NPIX) continue;
                const int r = px / DC_PW, c = px - r * DC_PW;
                bool ok = true;
                if (!interior) ok = (unsigned)(y0 - 1 + r) < (unsigned)H && (unsigned)(x0 - 1 + c) < (unsigned)W;
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (ok) {
                    float yv[8];
                    act8<T>(q[i], cf, yv);
                    o = pack8<T>(yv);
                }
                *reinterpret_cast<uint4*>(sact + ((c & 1) ^ 1) * DC_SPLANE + (r * DC_SW + ((c + 1) >> 1)) * 16) = o;
            }
        }
        {   // low: 10 x 34 pixels x 2 chunks of 8 channels -> two channel planes
            const int c8 = tid & 1;
            float2 cf[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) cf[e] = coef[c8 * 8 + e];
            constexpr int NSL = DC_LH * DC_LW * 2;                          // 680
            constexpr int SLOTS = (NSL + DC_THREADS - 1) / DC_THREADS;     // 3
            uint4 q[SLOTS];
#pragma unroll
            for (int i = 0; i < SLOTS; ++i) {
                const int s = tid + i * DC_THREADS;
                if (s < NSL) q[i] = *reinterpret_cast<const uint4*>(lraw + s * 16);
            }
#pragma unroll
            for (int i = 0; i < SLOTS; ++i) {
                const int s = tid + i * DC_THREADS;
                if (s >= NSL) continue;
                const int lp = s >> 1;
                bool ok = true;
                if (!interior) {
                    const int lr = lp / DC_LW, lc = lp - lr * DC_LW;
                    ok = (unsigned)((y0 >> 1) - 1 + lr) < (unsigned)Hl && (unsigned)((x0 >> 1) - 1 + lc) < (unsigned)Wl;
                }
                uint4 o = make_uint4(0u, 0u, 0u, 0u);
                if (ok) {
                    float yv[8];
                    act8<T>(q[i], cf, yv);
                    o = pack8<T>(yv);
                }
                *reinterpret_cast<uint4*>(lact + c8 * DC_LPLANE + lp * 16) = o;
            }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // our reads of the raw stage vs its TMA refill below
        __syncthreads();
        if (tid == 0 && tile + DC_NS < t1) issue(tile + DC_NS, stage);   // the raw stage is consumed: refill it two tiles ahead

        // ---- (2) tensor-core part --------------------------------------------------------------------------------------------
        float acc[4][2][4];
#pragma unroll
        for (int r4 = 0; r4 < 4; ++r4)
#pragma unroll
            for (int px = 0; px < 2; ++px) {
                acc[r4][px][0] = acc[r4][px][2] = btot[0];
                acc[r4][px][1] = acc[r4][px][3] = btot[1];
            }
        // (2a) `up` half through the composite weights: low rows 2 rb + d, d = 0..3; output row r4 of the warp (py = r4 & 1)
        // reads low rows d = (r4 >> 1) + (r4 & 1) + ti.  Column offsets tj + px = 0, 1, 2.
        {
            const uint32_t l_base = lact_u + (uint32_t)((lane >> 4) * DC_LPLANE + ((2 * rb) * DC_LW + 16 * cb + (lane & 15)) * 16);
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                uint32_t f[3][4];
#pragma unroll
                for (int co = 0; co < 3; ++co)
                    ldsm_x4(l_base + (uint32_t)((d * DC_LW + co) * 16), f[co][0], f[co][1], f[co][2], f[co][3]);
#pragma unroll
                for (int r4 = 0; r4 < 4; ++r4) {
                    const int ti = d - (r4 >> 1) - (r4 & 1);
                    if (ti < 0 || ti > 1) continue;
                    const int py = r4 & 1;
#pragma unroll
                    for (int px = 0; px < 2; ++px)
#pragma unroll
                        for (int tj = 0; tj < 2; ++tj)
                            mma16816<T>(acc[r4][px], f[tj + px][0], f[tj + px][1], f[tj + px][2], f[tj + px][3],
                                        bc[py * 2 + px][ti * 2 + tj][0], bc[py * 2 + px][ti * 2 + tj][1]);
                }
            }
        }
        // (2b) skip half: 3x3 over 8 channels on the parity planes.  For output column x = x0 + 2 jj + px the taps kx = 0, 1, 2 read
        // (plane, half-column): px = 0 -> (1, jj), (0, jj+1), (1, jj+1);  px = 1 -> (0, jj+1), (1, jj+1), (0, jj+2).
        {
            const uint32_t s_lane = (uint32_t)((16 * cb + (lane & 15)) * 16);
            const uint32_t x1 = sact_u + s_lane + ((lane >> 4) ? (uint32_t)(16) : (uint32_t)DC_SPLANE);                  // (1, jj) | (0, jj+1)
            const uint32_t x2 = sact_u + s_lane + 16 + ((lane >> 4) ? (uint32_t)DC_SPLANE : 0u);                           // (0, jj+1) | (1, jj+1)
            const uint32_t x3 = sact_u + s_lane + 32;                                                                     // (0, jj+2)
#pragma unroll
            for (int sr = 0; sr < 6; ++sr) {   // skip rows 4 rb + sr of the halo tile feed output rows r4 = sr - ky
                const uint32_t roff = (uint32_t)(((4 * rb + sr) * DC_SW) * 16);
                uint32_t a[4], b[4], c0, c1;
                ldsm_x4(x1 + roff, a[0], a[1], a[2], a[3]);
                ldsm_x4(x2 + roff, b[0], b[1], b[2], b[3]);
                ldsm_x2(x3 + roff, c0, c1);
#pragma unroll
                for (int ky = 0; ky < 3; ++ky) {
                    const int r4 = sr - ky;
                    if (r4 < 0 || r4 > 3) continue;
                    mma16816<T>(acc[r4][0], a[0], a[1], a[2], a[3], bs[ky * 3], bs[ky * 3 + 1]);
                    mma16808<T>(acc[r4][0], b[2], b[3], bs[ky * 3 + 2]);
                    mma16816<T>(acc[r4][1], b[0], b[1], b[2], b[3], bs[ky * 3], bs[ky * 3 + 1]);
                    mma16808<T>(acc[r4][1], c0, c1, bs[ky * 3 + 2]);
                }
            }
        }
        // ---- (3) epilogue ------------------------------------------------------------------------------------------------------
        // accumulator row m = lane >> 2 (+8) of parity px is output column x0 + 32 cb + 2 m + px; columns 2 (lane & 3), +1 = channels
        float s1[2] = {0.f, 0.f}, s2[2] = {0.f, 0.f};
        const bool full = (y0 + DC_TH <= H) && (x0 + DC_TW <= W);
        const bool edge = y0 == 0 || x0 == 0 || y0 + DC_TH >= H || x0 + DC_TW >= W;   // tile touches the image border: bias taps missing
        const int gxb = x0 + 32 * cb + 2 * (lane >> 2);
        const uint32_t orow = (uint32_t)W * DC_CU;
        T* obase = outp + ((size_t)(n * H + y0 + 4 * rb) * W + gxb) * DC_CU + 2 * (lane & 3);
        auto epilogue = [&](auto full_c, auto edge_c) {
            constexpr bool FULL = decltype(full_c)::value, EDGE = decltype(edge_c)::value;
#pragma unroll
            for (int r4 = 0; r4 < 4; ++r4) {
                const int gy = y0 + 4 * rb + r4;
#pragma unroll
                for (int px = 0; px < 2; ++px)
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf) {
                        const int gx = gxb + 16 * hf + px;
                        const bool ok = FULL || (gy < H && gx < W);
                        float v0 = acc[r4][px][2 * hf], v1 = acc[r4][px][2 * hf + 1];
                        if constexpr (EDGE) {
                            // a pixel ON the image border loses the ConvTranspose bias of the taps outside the image (the concat is
                            // zero-padded there): whole tap rows / columns, corners added back once
                            const bool top = gy == 0, bot = gy == H - 1, lef = gx == 0, rig = gx == W - 1;
                            if (top || bot || lef || rig) {
                                const int o = 2 * (lane & 3);
                                float c0 = 0.f, c1 = 0.f;
                                if (top) { c0 += bcorr[0 * DC_CU + o]; c1 += bcorr[0 * DC_CU + o + 1]; }
                                if (bot) { c0 += bcorr[1 * DC_CU + o]; c1 += bcorr[1 * DC_CU + o + 1]; }
                                if (lef) { c0 += bcorr[2 * DC_CU + o]; c1 += bcorr[2 * DC_CU + o + 1]; }
                                if (rig) { c0 += bcorr[3 * DC_CU + o]; c1 += bcorr[3 * DC_CU + o + 1]; }
                                if (top && lef) { c0 -= bcorr[4 * DC_CU + o]; c1 -= bcorr[4 * DC_CU + o + 1]; }
                                if (top && rig) { c0 -= bcorr[5 * DC_CU + o]; c1 -= bcorr[5 * DC_CU + o + 1]; }
                                if (bot && lef) { c0 -= bcorr[6 * DC_CU + o]; c1 -= bcorr[6 * DC_CU + o + 1]; }
                                if (bot && rig) { c0 -= bcorr[7 * DC_CU + o]; c1 -= bcorr[7 * DC_CU + o + 1]; }
                                v0 -= c0; v1 -= c1;
                            }
                        }
                        if (!ok) v0 = v1 = 0.f;
                        if (ok) *reinterpret_cast<uint32_t*>(obase + (uint32_t)r4 * orow + (16 * hf + px) * DC_CU) = pack2<T>(v0, v1);
                        s1[0] += v0; s2[0] = fmaf(v0, v0, s2[0]);
                        s1[1] += v1; s2[1] = fmaf(v1, v1, s2[1]);
                    }
            }
        };
        if (!edge) epilogue(std::true_type{}, std::false_type{});          // interior tiles are always full
        else if (full) epilogue(std::true_type{}, std::true_type{});
        else epilogue(std::false_type{}, std::true_type{});
        d1[0] += (double)s1[0]; d1[1] += (double)s1[1];
        d2[0] += (double)s2[0]; d2[1] += (double)s2[1];
        __syncthreads();   // every warp is done with the plane buffers before the next tile's activation overwrites them
    }
    if (cur_n >= 0) flush_stats(cur_n);
}

// ---- weight packing: composite ConvTranspose o Conv taps, skip taps, bias-per-tap table ------------------------------------------
// ct_w fp32 [2][2][CL][CU] (a, b, ci, co), ct_b [CU], conv_w fp32 [3][3][2 CU][CU] (ky, kx, c, o) with c < CU = up, c >= CU = skip.
template <typename T>
__global__ void pack_dec_composite_kernel(const float* __restrict__ ct_w, const float* __restrict__ ct_b, const float* __restrict__ w3,
                                          unsigned char* __restrict__ blob) {
    constexpr int CL = DC_CL, CU = DC_CU;
    T* comp = reinterpret_cast<T*>(blob);
    T* skw = reinterpret_cast<T*>(blob + DC_COMP_BYTES);
    float* bk = reinterpret_cast<float*>(blob + DC_COMP_BYTES + DC_SKIPW_BYTES);
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    // composite: index = (((cls*4 + tap)*2 + kh)*CU + o)*8 + e, ci = kh*8 + e
    if (tid < 16 * 2 * CU * 8) {
        const int e = tid & 7, o = (tid >> 3) % CU, kh = (tid / (8 * CU)) & 1, ct = tid / (16 * CU);
        const int cls = ct >> 2, tap = ct & 3, py = cls >> 1, px = cls & 1, ti = tap >> 1, tj = tap & 1, ci = kh * 8 + e;
        float s = 0.f;
        for (int ky = 0; ky < 3; ++ky) {
            const int ey = py + ky - 1, dy = ey < 0 ? -1 : ey >> 1, a = ey - 2 * dy;   // up row y + ky - 1 = 2 (i + dy) + a
            if (dy + 1 - py != ti) continue;
            for (int kx = 0; kx < 3; ++kx) {
                const int ex = px + kx - 1, dx = ex < 0 ? -1 : ex >> 1, b = ex - 2 * dx;
                if (dx + 1 - px != tj) continue;
                for (int co = 0; co < CU; ++co)
                    s += ct_w[((a * 2 + b) * CL + ci) * CU + co] * w3[((ky * 3 + kx) * (2 * CU) + co) * CU + o];
            }
        }
        comp[tid] = Store<T>::from_f(s);
    }
    // skip taps: index = (tap*CU + o)*8 + cs
    if (tid < 9 * CU * 8) {
        const int cs = tid & 7, o = (tid >> 3) % CU, tap = tid / (8 * CU);
        skw[tid] = Store<T>::from_f(w3[(tap * (2 * CU) + CU + cs) * CU + o]);
    }
    // bias through tap t: bk[t][o] = sum_co W3[t][co][o] b[co]
    if (tid < 9 * CU) {
        const int o = tid % CU, tap = tid / CU;
        float s = 0.f;
        for (int co = 0; co < CU; ++co) s += w3[(tap * (2 * CU) + co) * CU + o] * ct_b[co];
        bk[tid] = s;
    }
}

template <typename T>
int launch_dec(const DecArgs& a, cudaStream_t st) {
    auto kern = dec8_ring_kernel<T>;
    static bool done = false;
    if (!done) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, DC_SMEM);
        if (e != cudaSuccess) { set_error("dec8 ring: cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return 4; }
        done = true;
    }
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    }
    int grid = 2 * sms;
    if (grid > a.total) grid = a.total;
    cudaError_t le = launch_kernel(kern, dim3(grid), dim3(DC_THREADS), (size_t)DC_SMEM, st, a);
    if (le != cudaSuccess) { set_error("dec8 ring launch: %s", cudaGetErrorString(le)); return 10; }
    count_launch();
    return check_launch("dec8_ring");
}

}  // namespace

int dec_composite_bytes(int cl, int cu, size_t* bytes) {
    if (cl == DC_CL && cu == DC_CU) { *bytes = DC_BLOB_BYTES; return 0; }
    set_error("composite decoder packing: %d -> %d not covered (only (16, 8))", cl, cu);
    return 3;
}

int pack_dec_composite(const float* ct_w, const float* ct_b, const float* conv_w, void* out, int cl, int cu, int dtype, cudaStream_t st) {
    size_t bytes;
    int rc = dec_composite_bytes(cl, cu, &bytes);
    if (rc) return rc;
    if (dtype != DG_F16 && dtype != DG_BF16) { set_error("composite decoder packing needs a 16-bit dtype"); return 2; }
    const int threads = 16 * 2 * DC_CU * 8;
    if (dtype == DG_F16) pack_dec_composite_kernel<__half><<<(threads + 255) / 256, 256, 0, st>>>(ct_w, ct_b, conv_w, (unsigned char*)out);
    else pack_dec_composite_kernel<__nv_bfloat16><<<(threads + 255) / 256, 256, 0, st>>>(ct_w, ct_b, conv_w, (unsigned char*)out);
    count_launch();
    return check_launch("pack_dec_composite");
}

// path bit 10 (1024): do not use this kernel (A/B against conv3x3_tc.cu MODE_UPCAT)
int conv3x3_dec_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled) {
    *handled = false;
    if (a.path & 1024) return 0;
    if (a.dtype != DG_F16 && a.dtype != DG_BF16) return 0;
    if (a.weight_comp == nullptr || a.act_sum != nullptr || a.nsrc != 2 || a.cout != DC_CU) return 0;
    const dg_src& s0 = a.src[0];
    const dg_src& s1 = a.src[1];
    if (s0.xform != DG_X_CONVT2 || s0.channels != DC_CL || s0.ct_cout != DC_CU || s0.stats == nullptr || !s0.silu || s0.scale) return 0;
    if (s1.xform != DG_X_SAME || s1.channels != DC_CU || s1.stats == nullptr || !s1.silu || s1.scale) return 0;
    if (s0.coef != nullptr || s1.coef != nullptr) return 0;
    if ((a.H | a.W) & 1) return 0;
    if ((reinterpret_cast<uintptr_t>(s0.raw) | reinterpret_cast<uintptr_t>(s1.raw) | reinterpret_cast<uintptr_t>(a.out) |
         reinterpret_cast<uintptr_t>(a.weight_comp)) & 15)
        return 0;
    DecArgs r;
    memset(&r, 0, sizeof(r));
    if (!tma_map_nhwc(&r.tmap_skip, s1.raw, a.N, a.H, a.W, 2, DC_PW, DC_PH)) return 0;
    if (!tma_map_nhwc(&r.tmap_low, s0.raw, a.N, a.H / 2, a.W / 2, 4, DC_LW, DC_LH)) return 0;
    r.st_l = s0.stats; r.g_l = s0.gamma; r.b_l = s0.beta; r.groups_l = s0.groups;
    r.st_s = s1.stats; r.g_s = s1.gamma; r.b_s = s1.beta; r.groups_s = s1.groups;
    r.blob = a.weight_comp; r.out = a.out; r.out_stats = a.out_stats;
    r.N = a.N; r.H = a.H; r.W = a.W; r.eps = a.eps;
    r.tiles_x = (a.W + DC_TW - 1) / DC_TW;
    r.tiles_y = (a.H + DC_TH - 1) / DC_TH;
    const long long total = (long long)r.tiles_x * r.tiles_y * a.N;
    if (total > 0x7fffffffLL) return 0;
    r.total = (int)total;
    *handled = true;
    return a.dtype == DG_F16 ? launch_dec<__half>(r, stream) : launch_dec<__nv_bfloat16>(r, stream);
}

}  // namespace dg
