// First layer (enc1.0: Conv2d(1, C, 3, padding=1, bias=False), src/model.py:93 with in_channels=1) for 16-bit
// storage, on the tensor cores.  The layer is memory-bound (20 B/pixel, 72 MAC/pixel for C=8) but on CUDA cores its
// 72 FFMA + 16 statistics instructions per pixel eat the whole issue budget of the HBM roofline, so the 3x3 stencil
// is run as ONE m16n8k16 HMMA per 16 pixels instead: K = 9 taps placed in 12 of the 16 k-slots as horizontally
// adjacent pairs, so that every A register is a single aligned 32-bit shared-memory load from one of two copies of
// the 16-bit input tile (the second copy is shifted by one pixel to make odd columns aligned):
//
//   k-slot pair p (k = 2p, 2p+1)      0        1        2        3         4         5        6,7
//   taps (ky; kx, kx+1)            (0;0,1)  (1;0,1)  (2;0,1)  (0;1,2)*  (1;1,2)*  (2;1,2)*   zero
//                                  (* first weight of the pair is zero -- only kx=2 is taken from it)
//
// The fp32 network input is rounded to the storage type when the tile is staged (the fp32 tier uses the generic
// kernel).  Epilogue and GroupNorm statistics are those of conv3x3_tc.cu.
#include "tc_common.cuh"

namespace dg {

namespace {
constexpr int F_TH = 32, F_TW = 64, F_PH = F_TH + 2, F_PW = F_TW + 2, F_PA = 68;  // PA: even row pitch (elements)
constexpr int F_THREADS = 256;

struct FirstArgs {
    const float* x; const float* w; void* out; double* out_stats;
    int N, H, W;
    int x_u8;  // x points at uint8 pixels, normalised as float32(u) / 255.0f (api/app.py:153) -- IEEE divide, bit-exact
};

__device__ __forceinline__ float u8_norm(unsigned int u) { return __fdiv_rn((float)u, 255.f); }

template <typename T, int NT>
__global__ void __launch_bounds__(F_THREADS) conv_first_tc_kernel(const FirstArgs p) {
    constexpr int COUT = 8 * NT;
    __shared__ __align__(16) T tileA[F_PH * F_PA];
    __shared__ __align__(16) T tileB[F_PH * F_PA];  // tileB[r][c] = tile(r, c + 1)
    __shared__ float statw[8][2 * COUT];  // per-warp (sum, sumsq) slots, summed in a fixed order

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int q = lane & 3, g = lane >> 2;
    const int n = blockIdx.z;
    const int y0 = blockIdx.y * F_TH, x0 = blockIdx.x * F_TW;
    const int H = p.H, W = p.W;

    pdl_launch_dependents();
    pdl_wait();  // the statistics buffer is zeroed by a memset / reused from the previous forward's consumers
    // ---- stage the haloed input tile (fp32 -> T), zero outside the image ------------------------------
    // Per tile row: 16 aligned float4 groups (the 64 interior pixels; tile column = 1 + 4j..4 + 4j) and the two halo
    // columns.  In tileB (shifted copy) a group is one aligned 8-byte store; in tileA it straddles 4-byte words.
    const float* img = p.x + (size_t)n * H * W;
    const unsigned char* img8 = reinterpret_cast<const unsigned char*>(p.x) + (size_t)n * H * W;
    const bool u8 = p.x_u8 != 0;
    const bool vec_ok = (x0 + F_TW <= W) && ((W & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.x) & (u8 ? 3 : 15)) == 0);
    auto px = [&](size_t off) -> float { return u8 ? u8_norm(__ldg(img8 + off)) : __ldg(img + off); };
    for (int idx = tid; idx < F_PH * 18; idx += F_THREADS) {
        const int r = idx / 18, j = idx - r * 18;
        const int gy = y0 + r - 1;
        const bool rowok = (unsigned)gy < (unsigned)H;
        T* ra = tileA + r * F_PA;
        T* rb = tileB + r * F_PA;
        if (j < 16) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            const int gx = x0 + 4 * j;
            if (rowok) {
                if (vec_ok) {
                    if (u8) {
                        const uchar4 q4 = __ldg(reinterpret_cast<const uchar4*>(img8 + (size_t)gy * W + gx));
                        v = make_float4(u8_norm(q4.x), u8_norm(q4.y), u8_norm(q4.z), u8_norm(q4.w));
                    } else {
                        v = __ldg(reinterpret_cast<const float4*>(img + (size_t)gy * W + gx));
                    }
                } else {
                    if (gx < W) v.x = px((size_t)gy * W + gx);
                    if (gx + 1 < W) v.y = px((size_t)gy * W + gx + 1);
                    if (gx + 2 < W) v.z = px((size_t)gy * W + gx + 2);
                    if (gx + 3 < W) v.w = px((size_t)gy * W + gx + 3);
                }
            }
            const uint32_t lo = pack2<T>(v.x, v.y), hi = pack2<T>(v.z, v.w);
            const int c = 1 + 4 * j;                                   // tile column of v.x
            *reinterpret_cast<uint2*>(rb + c - 1) = make_uint2(lo, hi);  // tileB[r][c-1 .. c+2]
            reinterpret_cast<unsigned short*>(ra)[c] = (unsigned short)(lo & 0xffffu);
            *reinterpret_cast<uint32_t*>(ra + c + 1) = (lo >> 16) | (hi << 16);
            reinterpret_cast<unsigned short*>(ra)[c + 3] = (unsigned short)(hi >> 16);
        } else {
            const int c = j == 16 ? 0 : F_PW - 1;
            const int gx = x0 + c - 1;
            float v = 0.f;
            if (rowok && (unsigned)gx < (unsigned)W) v = px((size_t)gy * W + gx);
            const T h = Store<T>::from_f(v);
            ra[c] = h;
            if (c >= 1) rb[c - 1] = h;
        }
    }

    // ---- B fragments: b0 = k-slot pair q, b1 = pair 4+q, column (output channel) g of each n-tile -------
    uint32_t bfr[NT][2];
    {
        // pair -> (tap of first slot or -1, tap of second slot or -1)
        const int t0a = q < 3 ? 3 * q : -1, t0b = q < 3 ? 3 * q + 1 : 2;          // pairs 0..3
        const int t1a = -1, t1b = q == 0 ? 5 : (q == 1 ? 8 : -1);                  // pairs 4..7
#pragma unroll
        for (int i = 0; i < NT; ++i) {
            const int co = i * 8 + g;
            const float w0a = t0a >= 0 ? __ldg(p.w + t0a * COUT + co) : 0.f;
            const float w0b = t0b >= 0 ? __ldg(p.w + t0b * COUT + co) : 0.f;
            const float w1a = t1a >= 0 ? __ldg(p.w + t1a * COUT + co) : 0.f;
            const float w1b = t1b >= 0 ? __ldg(p.w + t1b * COUT + co) : 0.f;
            bfr[i][0] = pack2<T>(w0a, w0b);
            bfr[i][1] = pack2<T>(w1a, w1b);
        }
    }
    // ---- per-thread A addressing: pair -> (ky, first column offset); parity of (g + kxs) picks the copy ---
    // pair q (q<3: ky=q,kxs=0; q==3: ky=0,kxs=1) and pair 4+q (q==0: ky=1,kxs=1; q==1: ky=2,kxs=1; else dummy = pair 0)
    const int ky0 = q < 3 ? q : 0, kx0 = q < 3 ? 0 : 1;
    const int ky1 = q == 0 ? 1 : (q == 1 ? 2 : 0), kx1 = q < 2 ? 1 : 0;
    auto pair_addr = [&](int ky, int kxs) -> uint32_t {
        const int cc = g + kxs;  // column of the pair's first element for pixel g of a segment (segments start even)
        const T* base = (cc & 1) ? tileB : tileA;
        return smem_u32(base + ky * F_PA + (cc & ~1));
    };
    const uint32_t addr0 = pair_addr(ky0, kx0), addr1 = pair_addr(ky1, kx1);
    __syncthreads();

    float s1[NT][2], s2[NT][2];
#pragma unroll
    for (int i = 0; i < NT; ++i) s1[i][0] = s1[i][1] = s2[i][0] = s2[i][1] = 0.f;
    T* outp = reinterpret_cast<T*>(p.out);
    const bool full = (y0 + F_TH <= H) && (x0 + F_TW <= W);

    auto body = [&](auto full_c) {
        constexpr bool FULL = decltype(full_c)::value;
#pragma unroll 2
        for (int mi = 0; mi < (F_TH * (F_TW / 16)) / 8; ++mi) {
            const int mt = warp + 8 * mi;
            const int row = mt >> 2, seg = mt & 3;
            const uint32_t moff = (uint32_t)((row * F_PA + seg * 16) * 2);
            uint32_t a0, a1, a2, a3;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(a0) : "r"(addr0 + moff));
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(a1) : "r"(addr0 + moff + 16));
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(a2) : "r"(addr1 + moff));
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(a3) : "r"(addr1 + moff + 16));
            const int gy = y0 + row, gx = x0 + seg * 16 + g;
            T* o = outp + ((size_t)(n * H + gy) * W + gx) * COUT + 2 * q;
#pragma unroll
            for (int i = 0; i < NT; ++i) {
                float acc[4] = {0.f, 0.f, 0.f, 0.f};
                mma16816<T>(acc, a0, a1, a2, a3, bfr[i][0], bfr[i][1]);
#pragma unroll
                for (int hf = 0; hf < 2; ++hf) {
                    const bool ok = FULL || (gy < H && gx + 8 * hf < W);
                    const float v0 = ok ? acc[2 * hf] : 0.f, v1 = ok ? acc[2 * hf + 1] : 0.f;
                    if (ok) *reinterpret_cast<uint32_t*>(o + hf * 8 * COUT + i * 8) = pack2<T>(v0, v1);
                    s1[i][0] += v0; s2[i][0] = fmaf(v0, v0, s2[i][0]);
                    s1[i][1] += v1; s2[i][1] = fmaf(v1, v1, s2[i][1]);
                }
            }
        }
    };
    if (full) body(std::true_type{});
    else body(std::false_type{});

#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            float a = s1[i][k], b = s2[i][k];
#pragma unroll
            for (int o = 4; o < 32; o <<= 1) {
                a += __shfl_xor_sync(0xffffffffu, a, o);
                b += __shfl_xor_sync(0xffffffffu, b, o);
            }
            if (lane < 4) {
                const int ch = i * 8 + 2 * lane + k;
                statw[warp][2 * ch] = a;
                statw[warp][2 * ch + 1] = b;
            }
        }
    __syncthreads();
    if (p.out_stats != nullptr && tid < 2 * COUT) {
        double t = 0.0;
#pragma unroll
        for (int w8 = 0; w8 < 8; ++w8) t += (double)statw[w8][tid];
        atomicAdd(p.out_stats + (size_t)n * COUT * 2 + tid, t);
    }
}
}  // namespace

int conv_first_tc_launch(const dg_conv3x3_args& a, cudaStream_t stream, bool* handled) {
    *handled = false;
    const dg_src& s = a.src[0];
    if (a.nsrc != 1 || (s.xform != DG_X_IMAGE && s.xform != DG_X_IMAGE_U8) || s.channels != 1 || s.stats != nullptr || s.silu || s.scale) return 0;
    if (a.dtype != DG_F16 && a.dtype != DG_BF16) return 0;
    if (a.cout != 8 && a.cout != 16) return 0;
    if (a.act_sum != nullptr || a.N > 65535) return 0;
    if (reinterpret_cast<uintptr_t>(a.out) & 3) return 0;
    FirstArgs f{reinterpret_cast<const float*>(s.raw), a.weight, a.out, a.out_stats, a.N, a.H, a.W, s.xform == DG_X_IMAGE_U8 ? 1 : 0};
    dim3 grid((a.W + F_TW - 1) / F_TW, (a.H + F_TH - 1) / F_TH, a.N);
    cudaError_t le = cudaSuccess;
    if (a.dtype == DG_F16) {
        if (a.cout == 8) le = launch_kernel(conv_first_tc_kernel<__half, 1>, grid, dim3(F_THREADS), (size_t)0, stream, f);
        else le = launch_kernel(conv_first_tc_kernel<__half, 2>, grid, dim3(F_THREADS), (size_t)0, stream, f);
    } else {
        if (a.cout == 8) le = launch_kernel(conv_first_tc_kernel<__nv_bfloat16, 1>, grid, dim3(F_THREADS), (size_t)0, stream, f);
        else le = launch_kernel(conv_first_tc_kernel<__nv_bfloat16, 2>, grid, dim3(F_THREADS), (size_t)0, stream, f);
    }
    *handled = true;
    if (le != cudaSuccess) { set_error("conv_first_tc launch: %s", cudaGetErrorString(le)); return 10; }
    count_launch();
    return check_launch("conv_first_tc");
}

}  // namespace dg
