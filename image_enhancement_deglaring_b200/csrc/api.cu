// C-ABI entry points + the native LightweightUNet orchestrator (see include/deglare.h).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include <nvtx3/nvToolsExt.h>

#include "common.cuh"

namespace dg {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
static std::atomic<int> g_pdl{1};
bool pdl_enabled() { return g_pdl.load(std::memory_order_relaxed) != 0; }
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
        return 10;
    }
    return 0;
}

// NVTX ranges per fused kernel of the forward / backward (SURVEY section 5: the reference has no tracing at all).  NVTX v3 is
// header-only and a no-op unless a tool (Nsight Systems / Compute) injects itself; DG_NVTX=0 turns the calls off entirely.
static bool nvtx_on() {
    static const bool on = [] { const char* e = getenv("DG_NVTX"); return !(e && e[0] == '0'); }();
    return on;
}
struct NvtxRange {
    bool live;
    explicit NvtxRange(const char* name) : live(nvtx_on()) { if (live) nvtxRangePushA(name); }
    ~NvtxRange() { if (live) nvtxRangePop(); }
};
static const char* const kConvNames[18] = {"enc1.0", "enc1.3", "enc2.0", "enc2.3", "enc3.0", "enc3.3", "enc4.0", "enc4.3", "bottleneck.0",
                                           "bottleneck.3", "up4+dec4.0", "dec4.3", "up3+dec3.0", "dec3.3", "up2+dec2.0", "dec2.3",
                                           "up1+dec1.0", "dec1.3"};

// Path bits 2-6 and 11 selected kernel variants that measured slower and were removed.  A caller that still sets one gets an error
// rather than different kernels than it asked for.
constexpr int32_t kRemovedPathBits = 0x87c;
static int check_path(int32_t path, const char* who) {
    if (path & kRemovedPathBits) {
        set_error("%s: path %d sets bit %d, whose kernel variant was removed", who, path, __builtin_ctz(path & kRemovedPathBits));
        return 2;
    }
    return 0;
}

static int validate_src(const dg_src& s, const char* who) {
    if (s.raw == nullptr) { set_error("%s: null source pointer", who); return 2; }
    if (s.channels < 1) { set_error("%s: bad channel count %d", who, s.channels); return 2; }
    if (s.stats != nullptr) {
        if (s.gamma == nullptr || s.beta == nullptr) { set_error("%s: GroupNorm affine missing", who); return 2; }
        if (s.groups < 1 || s.channels % s.groups != 0) {
            set_error("%s: %d channels not divisible into %d groups", who, s.channels, s.groups);
            return 2;
        }
    }
    if (s.xform == DG_X_CONVT2 && (s.ct_w == nullptr || s.ct_b == nullptr || s.ct_cout < 1)) {
        set_error("%s: ConvTranspose parameters missing", who);
        return 2;
    }
    if (s.xform < DG_X_SAME || s.xform > DG_X_IMAGE_U8) { set_error("%s: bad xform %d", who, s.xform); return 2; }
    return 0;
}

// ---- LightweightUNet plan -----------------------------------------------------------------
constexpr float kGnEps = 1e-5f;   // every GroupNorm of the reference module (nn.GroupNorm's default)

// Kernel tiers of the orchestrator: path & 3 == 1 keeps every op on the CUDA-core kernels; the tensor-core choices made here
// (materialised ConvTranspose, bf16 backward) also need 16-bit storage.
static inline bool generic_only(const dg_lw_params* p) { return (p->path & 3) == 1; }
static inline bool tc16(const dg_lw_params* p) { return p->dtype != DG_F32 && !generic_only(p); }

struct LwPlan {
    int f[5];
    int conv_c[18], conv_h[18], conv_w[18];
    int conv_cin[18];   // input channels: the image, the previous conv, the level above (pooled) or cat(up, skip)
    size_t esz;         // bytes per stored activation element
    size_t raw_off[18], stats_off[18];
    size_t up_off[4];  // scratch for a materialised upconvK output (deep decoder levels, 16-bit storage)
    size_t stats_bytes, total_bytes;  // stats_bytes = the zero-initialised prefix (statistics)

    // workspace slices from image n0 on (every per-image tensor is contiguous over the batch): conv i's output before its
    // GroupNorm, that GroupNorm's statistics, and upconv u's materialised output
    char* raw(char* ws, int i, int n0) const { return ws + raw_off[i] + (size_t)n0 * conv_h[i] * conv_w[i] * conv_c[i] * esz; }
    double* stats(char* ws, int i, int n0) const { return reinterpret_cast<double*>(ws + stats_off[i]) + (size_t)n0 * conv_c[i] * 2; }
    char* up(char* ws, int u, int n0) const {
        const int i = 2 * (u + 5);   // the decoder conv consuming it
        return ws + up_off[u] + (size_t)n0 * conv_h[i] * conv_w[i] * f[3 - u] * esz;
    }
};

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }
static inline size_t dtype_size(int dt) { return dt == DG_F32 ? 4 : 2; }
static inline int block_level(int b) { return b < 5 ? b : 8 - b; }

static int make_plan(const dg_lw_params* p, int N, int H, int W, LwPlan* pl) {
    if (p == nullptr) { set_error("null params"); return 2; }
    if (int rc = check_path(p->path, "lw")) return rc;
    if (N < 1 || H < 16 || W < 16 || (H % 16) || (W % 16)) {
        // 500x500 raises at the first torch.cat in the reference (src/model.py:116); here it is an error too
        set_error("input %dx%dx%d: H and W must be positive multiples of 16", N, H, W);
        return 3;
    }
    if (p->dtype < DG_F32 || p->dtype > DG_BF16) { set_error("bad dtype %d", p->dtype); return 2; }
    if (p->features_start < 1 || p->in_channels < 1 || p->out_channels < 1) { set_error("bad channel configuration"); return 2; }
    for (int l = 0; l < 5; ++l) pl->f[l] = p->features_start << l;
    pl->esz = dtype_size(p->dtype);
    size_t off = 0;
    for (int i = 0; i < 18; ++i) {
        const int b = i / 2, lvl = block_level(b);
        pl->conv_c[i] = pl->f[lvl];
        pl->conv_cin[i] = i == 0 ? p->in_channels : (i % 2 ? pl->f[lvl] : (b < 5 ? pl->f[lvl - 1] : 2 * pl->f[lvl]));
        pl->conv_h[i] = H >> lvl;
        pl->conv_w[i] = W >> lvl;
        pl->stats_off[i] = off;
        off += (size_t)N * pl->conv_c[i] * 2 * sizeof(double);
    }
    pl->stats_bytes = off;
    off = align_up(off, 256);
    for (int i = 0; i < 18; ++i) {
        pl->raw_off[i] = off;
        off += align_up((size_t)N * pl->conv_h[i] * pl->conv_w[i] * pl->conv_c[i] * pl->esz, 256);
    }
    for (int u = 0; u < 4; ++u) {
        const int lvl = 3 - u;
        pl->up_off[u] = off;
        if (p->dtype != DG_F32)   // all four: inference materialises the deep ones, the tensor-core wgrad wants every `up`
            off += align_up((size_t)N * (H >> lvl) * (W >> lvl) * pl->f[lvl] * pl->esz, 256);
    }
    pl->total_bytes = off;
    return 0;
}

// Decoder levels whose ConvTranspose output is materialised by a stand-alone tensor-core GEMM (16-bit tiers) and read by the
// consuming conv as an identity source: every level with C_up >= 32 -- upconv4 / upconv3 of the shipped model, ALL levels of the
// wide variant (features_start = 64).  The concat itself is never stored.
static inline bool lw_up_materialised(const LwPlan& pl, int u) { return pl.f[3 - u] >= 32; }

// conv conv_idx's output through its GroupNorm + SiLU, images from n0 on
static dg_src gn_src(const dg_lw_params* p, const LwPlan& pl, char* ws, int conv_idx, int xform, int n0) {
    dg_src s;
    memset(&s, 0, sizeof(s));
    const int b = conv_idx / 2, j = conv_idx % 2;
    s.raw = pl.raw(ws, conv_idx, n0);
    s.stats = pl.stats(ws, conv_idx, n0);
    s.gamma = p->gn_w[b][j];
    s.beta = p->gn_b[b][j];
    s.channels = pl.conv_c[conv_idx];
    s.groups = p->groups[b];
    s.xform = xform;
    s.silu = 1;
    return s;
}

// a tensor read as it is stored: no GroupNorm, no SiLU
static dg_src ident_src(const void* raw, int channels, int xform = DG_X_SAME) {
    dg_src s;
    memset(&s, 0, sizeof(s));
    s.raw = raw;
    s.channels = channels;
    s.groups = 1;
    s.xform = xform;
    return s;
}

// upconv u's output, materialised in the workspace by the stand-alone tensor-core kernel (convt_tc.cu), as the first source of
// the decoder conv consuming it in place of the fused DG_X_CONVT2 source
static dg_src up_src(const LwPlan& pl, char* ws, int u, int n0) { return ident_src(pl.up(ws, u, n0), pl.f[3 - u]); }

// Conv i's arguments for images [n0, n0 + nn).  The forward launches them; the backward computes the weight gradient from the
// same sources.  x = the whole batch's input image, uint8 when x_u8.
static dg_conv3x3_args conv_args(const dg_lw_params* p, const LwPlan& pl, char* ws, const void* x, bool x_u8, int n0, int nn, int i) {
    const int b = i / 2;
    dg_conv3x3_args a;
    memset(&a, 0, sizeof(a));
    a.dtype = p->dtype;
    a.N = nn; a.H = pl.conv_h[i]; a.W = pl.conv_w[i];
    a.cout = pl.conv_c[i];
    a.weight = p->conv_w[b][i % 2];
    a.weight_tc = p->conv_w_tc[b][i % 2];
    a.out = pl.raw(ws, i, n0);
    a.out_stats = pl.stats(ws, i, n0);
    a.eps = kGnEps;
    a.path = p->path;
    a.nsrc = 1;
    if (i == 0) {
        const size_t img = (size_t)p->in_channels * a.H * a.W * (x_u8 ? 1 : sizeof(float));
        a.src[0] = ident_src(static_cast<const char*>(x) + n0 * img, p->in_channels, x_u8 ? DG_X_IMAGE_U8 : DG_X_IMAGE);
    } else if (i % 2 == 1) {
        a.src[0] = gn_src(p, pl, ws, i - 1, DG_X_SAME, n0);
    } else if (b < 5) {
        a.src[0] = gn_src(p, pl, ws, i - 1, DG_X_POOL2, n0);        // pool1..4, src/model.py:107-112
    } else {
        const int lvl = block_level(b), u = b - 5;
        a.src[0] = gn_src(p, pl, ws, i - 1, DG_X_CONVT2, n0);      // upconv4..1, src/model.py:115-127
        a.src[0].ct_w = p->up_w[u];
        a.src[0].ct_b = p->up_b[u];
        a.src[0].ct_w_tc = p->up_w_tc[u];
        a.src[0].ct_cout = pl.f[lvl];
        a.src[1] = gn_src(p, pl, ws, 2 * lvl + 1, DG_X_SAME, n0);  // skip: torch.cat((up, skip), 1)
        a.nsrc = 2;
        a.weight_comp = p->dec_comp[u];   // read by the forward's composite-tap kernel only (conv3x3_dec.cu)
    }
    return a;
}

// One forward over images [n0, n0 + nn) of a batch whose workspace was laid out for the whole batch (make_plan), on `stream`.
// io: bit 0 = x is uint8 (normalised by 1/255 on load), bit 1 = y is uint8 (clip + quantise in the head)
static int lw_forward_range(const dg_lw_params* p, const LwPlan& pl, char* ws, const void* x, void* y, int n0, int nn, int H, int W,
                            const float* target, double* l1_sum, cudaStream_t stream, cudaEvent_t* evs, int io) {
    int rc = 0;
    if (evs) cudaEventRecord(evs[0], stream);
    for (int i = 0; i < 18; ++i) {
        NvtxRange range(kConvNames[i]);
        dg_conv3x3_args a = conv_args(p, pl, ws, x, io & 1, n0, nn, i);
        const int u = i / 2 - 5;
        // deep levels (upconv4, upconv3): run the transposed conv as its own tensor-core GEMM and
        // feed its output as an identity source -- see convt_tc.cu for why this beats fusing there
        if (a.nsrc == 2 && tc16(p) && lw_up_materialised(pl, u)) {
            bool handled = false;
            rc = convt_tc_launch(a.src[0], p->dtype, nn, a.H, a.W, pl.up(ws, u, n0), kGnEps, p->path, stream, &handled);
            if (rc) return rc;
            if (handled) a.src[0] = up_src(pl, ws, u, n0);
        }
        rc = dg_conv3x3_fused(&a, reinterpret_cast<dg_stream_t>(stream));
        if (rc) return rc;
        if (evs) cudaEventRecord(evs[i + 1], stream);
    }
    NvtxRange head_range("head");
    dg_head_args h;
    memset(&h, 0, sizeof(h));
    h.src = gn_src(p, pl, ws, 17, DG_X_SAME, n0);
    h.dtype = p->dtype;
    h.N = nn; h.H = H; h.W = W;
    h.cout = p->out_channels;
    h.weight = p->head_w;
    h.bias = p->head_b;
    const size_t out_img = (size_t)p->out_channels * H * W;
    h.out = static_cast<char*>(y) + (size_t)n0 * out_img * ((io & 2) ? 1 : sizeof(float));
    h.target = target ? target + (size_t)n0 * out_img : nullptr;
    h.l1_sum = l1_sum;
    h.eps = kGnEps;
    h.out_kind = (io & 2) ? 1 : 0;
    rc = dg_head1x1(&h, reinterpret_cast<dg_stream_t>(stream));
    if (evs) cudaEventRecord(evs[19], stream);
    return rc;
}

// Two halves of a large batch run concurrently on two private streams (forked from / joined to the caller's stream with
// events): images are independent, and the tail of every kernel of one half -- the partial last wave, during which most SMs
// idle until the next kernel may start -- is filled by the other half's kernels.  Measured on B200, batch 64 x 512x512 fp16:
// 2.25 -> 2.09 ms per forward (two streams; four: 2.12); batch 32: 1.20 -> 1.08 ms, batch 16: 0.675 -> 0.599 ms, batch 8: no
// change (hence the default threshold of 16).  Outputs are bit-identical (nothing depends on the batch size).
struct FwdFork {
    static constexpr int MAXF = 2;   // the two halves of a batch
    bool ready = false;
    int device = -1;
    cudaStream_t s[MAXF];
    cudaEvent_t fork, join[MAXF];
};
// slot 0: calls on the caller's stream (dg_lw_forward / dg_lw_backward); slots 1..4: the chunks in flight of the host pipeline,
// which must not share fork streams (that would serialise the chunks again)
static FwdFork g_forks[5];
static std::atomic<int> g_split{16};   // minimum batch for the two-stream split; 0 disables (dg_set_batch_split)

static int fork_init(int slot) {
    FwdFork& g_fork = g_forks[slot];
    int dev = 0;
    cudaGetDevice(&dev);
    if (g_fork.ready && g_fork.device == dev) return 0;
    cudaError_t e = cudaSuccess;
    for (int k = 0; k < FwdFork::MAXF && e == cudaSuccess; ++k) e = cudaStreamCreateWithFlags(&g_fork.s[k], cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g_fork.fork, cudaEventDisableTiming);
    for (int k = 0; k < FwdFork::MAXF && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&g_fork.join[k], cudaEventDisableTiming);
    if (e != cudaSuccess) { set_error("forward fork streams: %s", cudaGetErrorString(e)); return 10; }
    g_fork.ready = true;
    g_fork.device = dev;
    return 0;
}

// range(n0, nn, stream) over the whole batch on st or, from g_split images on, over its two halves on the fork streams of `slot`
template <class Range>
static int run_halves(cudaStream_t st, int slot, int N, Range&& range) {
    const int split = g_split.load();
    if (split <= 0 || N < split || N < 2) return range(0, N, st);
    if (int rc = fork_init(slot)) return rc;
    FwdFork& F = g_forks[slot];
    cudaEventRecord(F.fork, st);
    const int half = N / 2;
    for (int k = 0; k < 2; ++k) {
        cudaStreamWaitEvent(F.s[k], F.fork, 0);
        const int rc = range(k ? half : 0, k ? N - half : half, F.s[k]);
        cudaEventRecord(F.join[k], F.s[k]);
        cudaStreamWaitEvent(st, F.join[k], 0);   // joined even on error, so the caller's stream stays ordered
        if (rc) return rc;
    }
    return 0;
}

static int lw_forward(const dg_lw_params* p, const void* x, void* y, int N, int H, int W, void* workspace,
                      size_t ws_bytes, const float* target, double* l1_sum, cudaStream_t stream,
                      cudaEvent_t* evs = nullptr, int io = 0, int fork_slot = 0) {
    LwPlan pl;
    int rc = make_plan(p, N, H, W, &pl);
    if (rc) return rc;
    if (workspace == nullptr || ws_bytes < pl.total_bytes) {
        set_error("workspace too small: %zu < %zu", ws_bytes, pl.total_bytes);
        return 4;
    }
    if (x == nullptr || y == nullptr) { set_error("null input/output"); return 2; }
    char* ws = static_cast<char*>(workspace);
    cudaError_t e = cudaMemsetAsync(ws, 0, pl.stats_bytes, stream);
    if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return 10; }
    auto range = [&](int n0, int nn, cudaStream_t s) {
        return lw_forward_range(p, pl, ws, x, y, n0, nn, H, W, target, l1_sum, s, evs, io);
    };
    return evs ? range(0, N, stream) : run_halves(stream, fork_slot, N, range);   // per-conv events time one stream
}

// ---- LightweightUNet backward ------------------------------------------------------------------
// Flat gradient layout = the module's parameters() order and the parameters' own memory layouts:
//   per block: conv0.weight [Co][Ci][3][3], gn0.weight, gn0.bias, conv1.weight, gn1.weight, gn1.bias
//   order: enc1..enc4, bottleneck, (upconvK.weight [Ci][Co][2][2], upconvK.bias, decK block) for K=4..1, head w, head b
// The named fields hold a tensor's index k in that order (bit k of dg_lw_bwd_request.param_mask); off[k] is its flat offset and
// pos[k] its forward position x 2: conv i and the GroupNorm after it 2i, upconvK one below the decoder conv consuming it, head 36.
constexpr int kLwTensors = 64;
struct GradLayout {
    int conv_w[9][2], gn_w[9][2], gn_b[9][2], up_w[4], up_b[4], head_w, head_b;
    size_t off[kLwTensors + 1];   // off[kLwTensors] = the total element count
    int pos[kLwTensors];
};

static void make_grad_layout(const dg_lw_params* p, const LwPlan& pl, GradLayout* g) {
    size_t off = 0;
    int k = 0;
    auto add = [&](size_t count, int pos) { g->off[k] = off; g->pos[k] = pos; off += count; return k++; };
    auto block = [&](int b) {
        const int c = pl.f[block_level(b)];
        g->conv_w[b][0] = add((size_t)c * pl.conv_cin[2 * b] * 9, 4 * b);
        g->gn_w[b][0] = add(c, 4 * b);
        g->gn_b[b][0] = add(c, 4 * b);
        g->conv_w[b][1] = add((size_t)c * c * 9, 4 * b + 2);
        g->gn_w[b][1] = add(c, 4 * b + 2);
        g->gn_b[b][1] = add(c, 4 * b + 2);
    };
    for (int b = 0; b < 5; ++b) block(b);
    for (int b = 5; b < 9; ++b) {
        const int lvl = block_level(b), u = b - 5;
        g->up_w[u] = add((size_t)pl.f[lvl + 1] * pl.f[lvl] * 4, 4 * b - 1);
        g->up_b[u] = add(pl.f[lvl], 4 * b - 1);
        block(b);
    }
    g->head_w = add((size_t)p->out_channels * pl.f[0], 36);
    g->head_b = add(p->out_channels, 36);
    g->off[k] = off;
}

// What one backward computes: the parameter tensors of `mask` into `grads`, and dL/dx into grad_x when set.  `low` = the lowest
// requested forward position x 2 (-2 = the input image): conv i's data gradient runs only when low < 2i.
struct BwdRequest {
    float* grads;
    uint64_t mask;
    float* grad_x;
    int low;
};

struct BwdPlan {
    size_t p_off[18], g_off[18], t_off[18], gb_off[18], low_off[4], coef_off, p_bytes, total;   // gb: dR as bf16 (16-bit tiers)
    int maxc;
};

static void make_bwd_plan(const dg_lw_params* p, const LwPlan& pl, int N, BwdPlan* bp) {
    size_t off = 0;
    for (int i = 0; i < 18; ++i) { bp->p_off[i] = off; off += (size_t)N * pl.conv_c[i] * 2 * sizeof(double); }
    bp->p_bytes = off;
    off = align_up(off, 256);
    int maxc = 0;
    for (int i = 0; i < 18; ++i) {
        bp->g_off[i] = off;
        off += align_up((size_t)N * pl.conv_h[i] * pl.conv_w[i] * pl.conv_c[i] * sizeof(float), 256);
        bp->t_off[i] = off;
        if (i > 0) off += align_up((size_t)N * pl.conv_h[i] * pl.conv_w[i] * pl.conv_cin[i] * sizeof(float), 256);
        if (pl.conv_c[i] > maxc) maxc = pl.conv_c[i];
    }
    for (int u = 0; u < 4; ++u) {
        const int lvl = 3 - u;  // upconv4 produces level 3 from level 4
        bp->low_off[u] = off;
        off += align_up((size_t)N * (pl.conv_h[2 * lvl + 2]) * (pl.conv_w[2 * lvl + 2]) * pl.f[lvl + 1] * sizeof(float), 256);
    }
    for (int i = 0; i < 18; ++i) {
        bp->gb_off[i] = off;
        if (i > 0 && p->dtype != DG_F32) off += align_up((size_t)N * pl.conv_h[i] * pl.conv_w[i] * pl.conv_c[i] * 2, 256);
    }
    bp->coef_off = off;
    bp->maxc = maxc;
    off += align_up((size_t)N * maxc * 2 * sizeof(float), 256);
    bp->total = off;
}

// nn.L1Loss backward fused into the head backward: forward output, target, device scalar dLoss (NULL = 1) and 1 / numel
struct L1Seed { const float* y; const float* target; const float* scale; float inv_numel; };

// Backward over images [n0, n0 + N) of a batch of N_total; every buffer was laid out for the whole batch (`N` below is the
// sub-batch size).  Parameter gradients are accumulated atomically, so concurrent sub-batches add up; the input gradient is per
// image.  Tensors outside rq.mask get no kernel work, and the loop ends below the lowest requested position.
static int lw_backward_range(const dg_lw_params* p, const LwPlan& pl, const BwdPlan& bp, const GradLayout& gl, const float* x,
                             const float* grad_y, int n0, int N, int H, int W, char* fw, char* bw, const BwdRequest& rq,
                             cudaStream_t st, const L1Seed* l1) {
    int rc = 0;
    auto gp = [&](int k) { return ((rq.mask >> k) & 1) ? rq.grads + gl.off[k] : nullptr; };
    bool t_split[18] = {};   // decoder conv i: T(i) holds the two halves of the concat gradient as two compact tensors
    auto hwc = [&](int i, int c) { return (size_t)pl.conv_h[i] * pl.conv_w[i] * c; };
    auto G = [&](int i) { return reinterpret_cast<float*>(bw + bp.g_off[i]) + (size_t)n0 * hwc(i, pl.conv_c[i]); };
    auto T = [&](int i) { return reinterpret_cast<float*>(bw + bp.t_off[i]) + (size_t)n0 * hwc(i, pl.conv_cin[i]); };
    auto P = [&](int i) { return reinterpret_cast<double*>(bw + bp.p_off[i]) + (size_t)n0 * pl.conv_c[i] * 2; };
    auto Rb = [&](int i) { return bw + bp.gb_off[i] + (size_t)n0 * hwc(i, pl.conv_c[i]) * 2; };   // dR_i as bf16 (16-bit tiers)
    auto raw = [&](int i) { return pl.raw(fw, i, n0); };
    auto stats = [&](int i) { return pl.stats(fw, i, n0); };
    auto act_bwd = [&](int j, const float* da, int sa, int oa, const float* db, int sb, int ob) {
        return act_bwd_launch(p->dtype, raw(j), stats(j), p->gn_w[j / 2][j % 2], p->gn_b[j / 2][j % 2], da, sa, oa, db, sb, ob, G(j),
                              P(j), N, pl.conv_h[j], pl.conv_w[j], pl.conv_c[j], p->groups[j / 2], kGnEps, st);
    };
    // head: src/model.py:131 backward
    const size_t o0 = (size_t)n0 * p->out_channels * H * W;
    rc = head_bwd_launch(p->dtype, raw(17), stats(17), p->gn_w[8][1], p->gn_b[8][1],
                         grad_y ? grad_y + o0 : nullptr, p->head_w, G(17), P(17),
                         gp(gl.head_w), gp(gl.head_b), N, H, W, pl.conv_c[17], p->out_channels, p->groups[8], kGnEps, st,
                         l1 ? l1->y + o0 : nullptr, l1 ? l1->target + o0 : nullptr, l1 ? l1->scale : nullptr, l1 ? l1->inv_numel : 0.f);
    if (rc) return rc;
    for (int i = 17; i >= 0 && rq.low <= 2 * i; --i) {
        const int b = i / 2, j = i % 2, C = pl.conv_c[i], Cin = pl.conv_cin[i], Hi = pl.conv_h[i], Wi = pl.conv_w[i];
        float* const dW = gp(gl.conv_w[b][j]);   // NULL: frozen, no weight-gradient kernel
        const bool dgrad = rq.low < 2 * i;       // something below conv i wants a gradient (i = 0: the input image)
        char rname[32];
        snprintf(rname, sizeof(rname), "bwd %s", kConvNames[i]);
        NvtxRange range(rname);
        // dW_i: same sources as the forward conv, correlated with dR_i; written in the parameter's [Co][Ci][3][3] layout.  The
        // tensor-core wgrad (wa) reads a decoder conv's ConvTranspose output materialised, the CUDA-core one (a) fuses it.
        const dg_conv3x3_args a = conv_args(p, pl, fw, x, false, n0, N, i);
        dg_conv3x3_args wa = a;
        if (a.nsrc == 2) wa.src[0] = up_src(pl, fw, b - 5, n0);
        // G_i -> dR_i, dgamma / dbeta.  Where BOTH consumers of dR_i are tensor-core kernels (they round it to bf16 anyway) it is
        // written once as bf16 instead of fp32 in place: they read half the bytes and copy the tile instead of converting it.  A
        // skipped weight gradient leaves the data gradient to decide alone.
        void* dRb = nullptr;
        if (i > 0 && (dW != nullptr || dgrad) && tc16(p) && p->conv_w_tc_bf16[b][j] != nullptr) {
            bool wg_ok = dW == nullptr, dgr_ok = false;
            if (dW != nullptr) conv3x3_wgrad_tc_launch(wa, G(i), dW, 1, 9, 9 * Cin, st, &wg_ok, nullptr, /*dry*/ true);
            conv3x3_dgrad_tc_launch(G(i), p->conv_w_tc_bf16[b][j], G(i), N, Hi, Wi, C, Cin, st, &dgr_ok, nullptr, nullptr, true);
            if (wg_ok && dgr_ok) dRb = Rb(i);
        }
        bool dr_bf16 = false;
        rc = gn_bwd_apply_launch(p->dtype, raw(i), stats(i), p->gn_w[b][j], P(i), G(i), gp(gl.gn_w[b][j]), gp(gl.gn_b[b][j]),
                                 N, Hi, Wi, C, p->groups[b], kGnEps, st, dRb, &dr_bf16);
        if (rc) return rc;
        const void* dRb_in = dr_bf16 ? dRb : nullptr;   // when set, G(i) still holds G, NOT dR: only the bf16 copy is valid
        bool wg_done = dW == nullptr;
        if (dW != nullptr && tc16(p) && i > 0) {
            // tensor-core wgrad (wgrad_tc.cu): the forward left the deep levels' ConvTranspose output in the workspace, for the
            // fused levels it is rebuilt here by the same stand-alone kernel
            bool ok = true;
            if (a.nsrc == 2 && !lw_up_materialised(pl, b - 5)) {
                rc = convt_tc_launch(a.src[0], p->dtype, N, Hi, Wi, pl.up(fw, b - 5, n0), kGnEps, p->path, st, &ok);
                if (rc) return rc;
            }
            if (ok) {
                rc = conv3x3_wgrad_tc_launch(wa, G(i), dW, 1, 9, 9 * Cin, st, &wg_done, dRb_in);
                if (rc) return rc;
            }
        }
        if (dW != nullptr && i == 0 && !generic_only(p) && p->in_channels == 1) {   // first conv: dedicated streaming kernel (backward.cu)
            rc = first_wgrad_launch(x + (size_t)n0 * p->in_channels * H * W, G(0), dW, N, Hi, Wi, C, st, &wg_done);
            if (rc) return rc;
        }
        if (!wg_done && dRb_in != nullptr) { set_error("backward: conv %d wgrad probe / launch mismatch", i); return 11; }
        if (!wg_done) {
            rc = conv3x3_wgrad_launch(a, G(i), dW, /*tap*/ 1, /*ci*/ 9, /*co*/ 9 * Cin, st);
            if (rc) return rc;
        }
        if (!dgrad) break;
        if (i == 0)   // dL/dx: dR_0 is fp32 in G(0) in every tier (conv 0 never gets the bf16 copy)
            return first_dgrad_launch(G(0), p->conv_w[0][0], rq.grad_x + (size_t)n0 * p->in_channels * H * W, N, H, W, p->in_channels, C, st);
        // dA_in = conv3x3(dR_i, flipped weights): tensor cores where covered (dgrad_tc.cu) ...
        bool dg_done = false;
        bool act_fused = false;
        if (tc16(p) && p->conv_w_tc_bf16[b][j] != nullptr) {
            if (j == 1) {
                // the second conv of a block: its input is the activated output of the first and nothing else consumes that, so
                // the data gradient goes straight through the producer's SiLU' / statistics sums into G(i-1), P(i-1)
                DgradAct act{raw(i - 1), stats(i - 1), p->gn_w[b][0], p->gn_b[b][0], P(i - 1), p->groups[b], p->dtype, kGnEps};
                rc = conv3x3_dgrad_tc_launch(G(i), p->conv_w_tc_bf16[b][j], G(i - 1), N, Hi, Wi, C, Cin, st, &dg_done, &act, dRb_in);
                if (rc) return rc;
                act_fused = dg_done;
            }
            if (!dg_done && j == 0 && b >= 5) {
                // decoder conv: its input gradient is a concat gradient whose halves go to different consumers -- written as two
                // compact tensors (up half at T(i), skip half right behind it) instead of one interleaved [.., 2C]
                rc = conv3x3_dgrad_tc_launch(G(i), p->conv_w_tc_bf16[b][j], T(i), N, Hi, Wi, C, Cin, st, &dg_done, nullptr, dRb_in,
                                             false, T(i) + (size_t)N * hwc(i, C));
                if (rc) return rc;
                t_split[i] = dg_done;
            }
            if (!dg_done) {
                rc = conv3x3_dgrad_tc_launch(G(i), p->conv_w_tc_bf16[b][j], T(i), N, Hi, Wi, C, Cin, st, &dg_done, nullptr, dRb_in);
                if (rc) return rc;
            }
        }
        // ... the tcgen05 kernel where the mma.sync data gradient has no instance (wider variants): dR rounded to bf16, the
        // taps-flipped weights in the tensor-core packing, fp32 result (conv3x3_t5.cu, T5_IDENT) ...
        if (!dg_done && dRb_in == nullptr && tc16(p) && p->conv_w_flip_tc_bf16[b][j] != nullptr) {
            rc = conv3x3_dgrad_t5_launch(G(i), nullptr, Rb(i), p->conv_w_flip_tc_bf16[b][j], T(i), N, Hi, Wi, C, Cin, st, &dg_done);
            if (rc) return rc;
        }
        // ... else the forward generic kernel on an identity fp32 source
        if (!dg_done && dRb_in != nullptr) { set_error("backward: conv %d dgrad probe / launch mismatch", i); return 11; }
        if (!dg_done) {
            if (p->conv_w_flip[b][j] == nullptr) { set_error("backward: conv %d needs the CUDA-core dgrad but conv_w_flip is NULL", i); return 2; }
            dg_conv3x3_args d;
            memset(&d, 0, sizeof(d));
            d.dtype = DG_F32;
            d.N = N; d.H = Hi; d.W = Wi;
            d.cout = Cin;
            d.weight = p->conv_w_flip[b][j];
            d.out = T(i);
            d.eps = kGnEps;
            d.path = 1;
            d.nsrc = 1;
            d.src[0] = ident_src(G(i), C);
            rc = conv3x3_generic_launch(d, st);
            if (rc) return rc;
        }
        if (j == 1) {
            if (!act_fused) rc = act_bwd(i - 1, T(i), C, 0, nullptr, 0, 0);
        } else if (b < 5) {
            // producer = skip tensor of level b-1: gradient from the decoder's concat (skip half) + this pooled path
            const int lvl = b - 1, dconv = 2 * (8 - lvl);
            if (t_split[dconv]) rc = act_bwd(i - 1, T(dconv) + (size_t)N * hwc(dconv, pl.f[lvl]), pl.f[lvl], 0, T(i), pl.f[lvl], 0);
            else rc = act_bwd(i - 1, T(dconv), 2 * pl.f[lvl], pl.f[lvl], T(i), pl.f[lvl], 0);
        } else {
            const int lvl = block_level(b), u = b - 5;
            float* dlow = reinterpret_cast<float*>(bw + bp.low_off[u]) + (size_t)n0 * (Hi / 2) * (Wi / 2) * pl.f[lvl + 1];
            // the low-resolution producer feeds nothing but this ConvTranspose: with the tensor-core data gradient its activation
            // backward is fused into that kernel's epilogue, which then writes G(i-1) / P(i-1) directly
            // (the ConvTranspose's own data gradient only when something below it, at conv i-1 or lower, is requested)
            const bool low_wanted = rq.low < 2 * i - 1;
            const bool try_fuse = low_wanted && tc16(p) && p->up_w_tc_bf16[u] != nullptr;
            DgradAct lact{raw(i - 1), stats(i - 1), p->gn_w[b - 1][1], p->gn_b[b - 1][1], P(i - 1), p->groups[b - 1], p->dtype, kGnEps};
            bool low_fused = false;
            rc = convt_bwd_launch(p->dtype, T(i), t_split[i] ? pl.f[lvl] : 2 * pl.f[lvl], p->up_w[u], p->up_w_t[u], raw(i - 1), stats(i - 1), p->gn_w[b - 1][1],
                                  p->gn_b[b - 1][1], !low_wanted ? nullptr : try_fuse ? G(i - 1) : dlow, gp(gl.up_w[u]), gp(gl.up_b[u]),
                                  reinterpret_cast<float*>(bw + bp.coef_off) + (size_t)n0 * bp.maxc * 2, N, Hi, Wi, pl.f[lvl + 1], pl.f[lvl],
                                  p->groups[b - 1], kGnEps, st, !generic_only(p) ? p->up_w_tc_bf16[u] : nullptr,
                                  try_fuse ? &lact : nullptr, try_fuse ? &low_fused : nullptr,
                                  !generic_only(p) ? p->up_w_dgrad_tc_bf16[u] : nullptr,
                                  p->dtype != DG_F32 ? Rb(i) : nullptr);   // conv i's bf16 dR scratch is free again
            if (rc) return rc;
            if (!low_wanted) break;
            if (low_fused) continue;   // G(i-1), P(i-1) are done
            if (try_fuse) {            // the kernel declined: G(i-1) holds the plain gradient; act_bwd works in place on it
                rc = act_bwd(i - 1, G(i - 1), pl.f[lvl + 1], 0, nullptr, 0, 0);
                if (rc) return rc;
                continue;
            }
            rc = act_bwd(i - 1, dlow, pl.f[lvl + 1], 0, nullptr, 0, 0);
        }
        if (rc) return rc;
    }
    return 0;
}

// grads / mask / grad_x as in dg_lw_bwd_request; dg_lw_backward and dg_lw_backward_l1 are mask = every tensor, grad_x = NULL
static int lw_backward(const dg_lw_params* p, const float* x, const float* grad_y, int N, int H, int W, void* fwd_ws,
                       size_t fwd_bytes, void* bwd_ws, size_t bwd_bytes, float* grads, uint64_t mask, float* grad_x, cudaStream_t st,
                       const L1Seed* l1 = nullptr) {
    LwPlan pl;
    int rc = make_plan(p, N, H, W, &pl);
    if (rc) return rc;
    BwdPlan bp;
    make_bwd_plan(p, pl, N, &bp);
    GradLayout gl;
    make_grad_layout(p, pl, &gl);
    if (fwd_ws == nullptr || fwd_bytes < pl.total_bytes || bwd_ws == nullptr || bwd_bytes < bp.total) {
        set_error("backward: workspace too small (fwd %zu/%zu, bwd %zu/%zu)", fwd_bytes, pl.total_bytes, bwd_bytes, bp.total);
        return 4;
    }
    if (x == nullptr || (grad_y == nullptr && l1 == nullptr) || (mask != 0 && grads == nullptr)) { set_error("backward: null pointer"); return 2; }
    BwdRequest rq{grads, mask, grad_x, grad_x != nullptr ? -2 : 1 << 30};
    for (int k = 0; k < kLwTensors; ++k)
        if (((mask >> k) & 1) && gl.pos[k] < rq.low) rq.low = gl.pos[k];
    // conv_w_flip / up_w_t feed the CUDA-core data-gradient kernels only: required where a tensor-core packing is absent
    for (int b = 0; b < 9; ++b)
        for (int j = 0; j < 2; ++j)
            if ((2 * b + j) > 0 && p->conv_w_flip[b][j] == nullptr && p->conv_w_tc_bf16[b][j] == nullptr) {
                set_error("backward: neither flipped weights nor a bf16 tensor-core packing for conv %d", 2 * b + j);
                return 2;
            }
    for (int u = 0; u < 4; ++u)
        if (p->up_w_t[u] == nullptr && p->up_w_tc_bf16[u] == nullptr) { set_error("backward: transposed ConvTranspose weights missing"); return 2; }
    char* fw = static_cast<char*>(fwd_ws);
    char* bw = static_cast<char*>(bwd_ws);
    cudaError_t e = cudaMemsetAsync(bw, 0, bp.p_bytes, st);
    for (int k = 0; k < kLwTensors && e == cudaSuccess;) {   // one memset per run of requested tensors; the others stay untouched
        if (!((mask >> k) & 1)) { ++k; continue; }
        int k1 = k;
        while (k1 < kLwTensors && ((mask >> k1) & 1)) ++k1;
        e = cudaMemsetAsync(grads + gl.off[k], 0, (gl.off[k1] - gl.off[k]) * sizeof(float), st);
        k = k1;
    }
    if (e != cudaSuccess) { set_error("memset: %s", cudaGetErrorString(e)); return 10; }
    return run_halves(st, 0, N, [&](int n0, int nn, cudaStream_t s) {   // two concurrent sub-batches, as in lw_forward
        return lw_backward_range(p, pl, bp, gl, x, grad_y, n0, nn, H, W, fw, bw, rq, s, l1);
    });
}

// ---- host-buffer pipeline state --------------------------------------------------------------
struct HostPipe {
    bool ready = false;
    cudaEvent_t start;   // recorded on the CALLER's stream: weight packing etc. enqueued there is ordered before the pipeline
    static constexpr int NS = 4;  // chunks in flight (measured: 4 x 8-image chunks 2.84 ms per 64 images, 8 in flight 2.98, 2 in flight 3.3): compute streams, staging buffers and workspaces
    cudaStream_t s_in, s_cmp[NS], s_out;
    cudaEvent_t in_done[NS], cmp_done[NS], out_done[NS];
    // asynchronous submissions (dg_lw_infer_host_submit / _wait): the chunk counter runs ACROSS calls, so the first chunks of
    // call k+1 are copied in and computed while the last chunks of call k are still computing / being copied out
    static constexpr int NT = 8;  // tickets (calls) that may be outstanding
    unsigned long long seq = 0, tickets = 0;
    cudaEvent_t ticket_done[NT];
    const void* ws_in_flight = nullptr;   // scratch / geometry of the calls in flight: a different one drains the pipeline first
    int chunk_in_flight = 0, h_in_flight = 0, w_in_flight = 0;
};
static HostPipe g_pipes[16];   // one pipeline (streams, events) per device ordinal
static std::mutex g_pipe_mutex;  // the *_host entry points serialise: they share the pipeline and the caller's scratch

static int pipe_init(HostPipe** out) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 16) { set_error("infer_host: device ordinal %d out of range", dev); return 2; }
    HostPipe& g_pipe = g_pipes[dev];
    *out = &g_pipe;
    if (g_pipe.ready) return 0;
    cudaError_t e;
    if ((e = cudaStreamCreateWithFlags(&g_pipe.s_in, cudaStreamNonBlocking)) != cudaSuccess ||
        (e = cudaStreamCreateWithFlags(&g_pipe.s_out, cudaStreamNonBlocking)) != cudaSuccess) {
        set_error("stream create: %s", cudaGetErrorString(e));
        return 10;
    }
    for (int i = 0; i < HostPipe::NS; ++i) {
        if ((e = cudaStreamCreateWithFlags(&g_pipe.s_cmp[i], cudaStreamNonBlocking)) != cudaSuccess) {
            set_error("stream create: %s", cudaGetErrorString(e));
            return 10;
        }
        cudaEventCreateWithFlags(&g_pipe.in_done[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g_pipe.cmp_done[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&g_pipe.out_done[i], cudaEventDisableTiming);
    }
    if ((e = cudaEventCreateWithFlags(&g_pipe.start, cudaEventDisableTiming)) != cudaSuccess) {
        set_error("event create: %s", cudaGetErrorString(e));
        return 10;
    }
    for (int i = 0; i < HostPipe::NT; ++i)
        if ((e = cudaEventCreateWithFlags(&g_pipe.ticket_done[i], cudaEventDisableTiming | cudaEventBlockingSync)) != cudaSuccess) {
            set_error("event create: %s", cudaGetErrorString(e));
            return 10;
        }
    g_pipe.ready = true;
    return 0;
}

}  // namespace dg

using namespace dg;

extern "C" {

const char* dg_last_error_string(void) { return g_err; }
int dg_version(void) { return 100; }
int dg_set_batch_split(int min_batch) {
    const int old = g_split.load();
    g_split.store(min_batch < 0 ? 0 : min_batch);
    return old;
}
int dg_set_pdl(int enabled) {
    const int old = g_pdl.exchange(enabled ? 1 : 0);
    return old;
}
uint64_t dg_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int dg_conv3x3_fused(const dg_conv3x3_args* a, dg_stream_t stream) {
    if (a == nullptr) { set_error("conv3x3: null args"); return 2; }
    if (int rc = check_path(a->path, "conv3x3")) return rc;
    if (a->nsrc < 1 || a->nsrc > 2) { set_error("conv3x3: nsrc %d", a->nsrc); return 2; }
    if (a->N < 1 || a->H < 1 || a->W < 1 || a->cout < 1) { set_error("conv3x3: bad shape"); return 3; }
    if (a->weight == nullptr || a->out == nullptr) { set_error("conv3x3: null weight/out"); return 2; }
    for (int s = 0; s < a->nsrc; ++s) {
        int rc = validate_src(a->src[s], "conv3x3");
        if (rc) return rc;
        const int xf = a->src[s].xform;
        if ((xf == DG_X_UP2 || xf == DG_X_CONVT2) && ((a->H | a->W) & 1)) {
            set_error("conv3x3: up-sampled source needs even H, W (got %dx%d)", a->H, a->W);
            return 3;
        }
    }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if ((a->path & 3) != 1) {
        bool handled = false;
        int rc = conv_first_tc_launch(*a, st, &handled);
        if (rc) return rc;
        if (handled) return 0;
        rc = conv3x3_t5_launch(*a, st, &handled);     // warp-specialised tcgen05 + TMEM kernel: every C_out >= 32 layer
        if (rc) return rc;
        if (handled) return 0;
        rc = conv3x3_dec_launch(*a, st, &handled);    // upconv1 + dec1.0 with the ConvTranspose folded into the conv taps
        if (rc) return rc;
        if (handled) return 0;
        rc = conv3x3_ring_launch(*a, st, &handled);   // persistent TMA-fed kernel for the 8 -> 8 full-resolution layers
        if (rc) return rc;
        if (handled) return 0;
        rc = conv3x3_tc_launch(*a, st, &handled);
        if (rc) return rc;
        if (handled) return 0;
        if ((a->path & 3) == 2) { set_error("conv3x3: tensor-core path does not cover this configuration"); return 3; }
    }
    return conv3x3_generic_launch(*a, st);
}

int dg_conv3x3_wgrad(const dg_conv3x3_args* a, const float* dR, float* dW, int32_t s_tap, int32_t s_ci, int32_t s_co,
                     dg_stream_t stream) {
    if (a == nullptr || dR == nullptr || dW == nullptr) { set_error("wgrad: null pointer"); return 2; }
    if (int rc = check_path(a->path, "wgrad")) return rc;
    if (a->nsrc < 1 || a->nsrc > 2) { set_error("wgrad: nsrc %d", a->nsrc); return 2; }
    for (int s = 0; s < a->nsrc; ++s) {
        int rc = validate_src(a->src[s], "wgrad");
        if (rc) return rc;
    }
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    if ((a->path & 3) != 1) {
        bool handled = false;
        int rc = conv3x3_wgrad_tc_launch(*a, dR, dW, s_tap, s_ci, s_co, st, &handled);
        if (rc || handled) return rc;
        if ((a->path & 3) == 2) { set_error("wgrad: no tensor-core kernel for this configuration"); return 3; }
    }
    return conv3x3_wgrad_launch(*a, dR, dW, s_tap, s_ci, s_co, st);
}

int dg_conv3x3_dgrad(const float* dR, const void* weight_tc_bf16, float* dX, int32_t N, int32_t H, int32_t W, int32_t cin,
                     int32_t cout, dg_stream_t stream) {
    if (dR == nullptr || weight_tc_bf16 == nullptr || dX == nullptr) { set_error("dgrad: null pointer"); return 2; }
    bool handled = false;
    int rc = conv3x3_dgrad_tc_launch(dR, weight_tc_bf16, dX, N, H, W, cout, cin, reinterpret_cast<cudaStream_t>(stream), &handled);
    if (rc == 0 && !handled) { set_error("dgrad: no tensor-core kernel for %d -> %d channels (or unaligned pointers)", cin, cout); return 3; }
    return rc;
}

int dg_convt2x2_dgrad(const float* dCat, int32_t stride, const void* ct_w_tc_bf16, float* dLow, int32_t N, int32_t H, int32_t W,
                      int32_t cl, int32_t cu, dg_stream_t stream) {
    if (dCat == nullptr || ct_w_tc_bf16 == nullptr || dLow == nullptr) { set_error("convT dgrad: null pointer"); return 2; }
    bool handled = false;
    int rc = convt_dgrad_tc_launch(dCat, stride, ct_w_tc_bf16, dLow, N, H, W, cl, cu, reinterpret_cast<cudaStream_t>(stream), &handled);
    if (rc == 0 && !handled) { set_error("convT dgrad: no tensor-core kernel for %d -> %d channels / this shape", cl, cu); return 3; }
    return rc;
}

int dg_conv3x3_dgrad_wide(const float* dR, const void* weight_flip_tc_bf16, float* dX, void* scratch_bf16, int32_t N, int32_t H,
                          int32_t W, int32_t cin, int32_t cout, dg_stream_t stream) {
    if (dR == nullptr || weight_flip_tc_bf16 == nullptr || dX == nullptr || scratch_bf16 == nullptr) { set_error("wide dgrad: null pointer"); return 2; }
    if (N < 1 || H < 1 || W < 1) { set_error("wide dgrad: bad shape"); return 3; }
    bool handled = false;
    int rc = conv3x3_dgrad_t5_launch(dR, nullptr, scratch_bf16, weight_flip_tc_bf16, dX, N, H, W, cout, cin,
                                     reinterpret_cast<cudaStream_t>(stream), &handled);
    if (rc == 0 && !handled) { set_error("wide dgrad: no tcgen05 plan for %d -> %d channels at %dx%d (or unaligned pointers)", cin, cout, H, W); return 3; }
    return rc;
}

int dg_image_metrics(const float* output, const float* target, int32_t N, int32_t H, int32_t W, int32_t clip01, double data_range,
                     double* acc, dg_stream_t stream) {
    if (output == nullptr || target == nullptr || acc == nullptr) { set_error("metrics: null pointer"); return 2; }
    return image_metrics_launch(output, target, N, H, W, clip01, data_range, acc, reinterpret_cast<cudaStream_t>(stream));
}

int dg_head1x1(const dg_head_args* a, dg_stream_t stream) {
    if (a == nullptr) { set_error("head: null args"); return 2; }
    int rc = validate_src(a->src, "head");
    if (rc) return rc;
    if (a->src.xform != DG_X_SAME) { set_error("head: source must be same-resolution"); return 3; }
    if (a->weight == nullptr || a->bias == nullptr || a->out == nullptr) { set_error("head: null pointer"); return 2; }
    return head_launch(*a, reinterpret_cast<cudaStream_t>(stream));
}

int dg_tc_conv3x3_bytes(int32_t cin, int32_t cout, size_t* bytes) {
    if (bytes == nullptr) { set_error("null bytes"); return 2; }
    return tc_conv3x3_bytes(cin, cout, bytes);
}
int dg_pack_conv3x3_tc(const float* w, void* out, int32_t cin, int32_t cout, int32_t dtype, dg_stream_t stream) {
    if (w == nullptr || out == nullptr) { set_error("pack: null pointer"); return 2; }
    return pack_conv3x3_tc(w, out, cin, cout, dtype, reinterpret_cast<cudaStream_t>(stream));
}
int dg_tc_convt2x2_bytes(int32_t cin, int32_t cout, size_t* bytes) {
    if (bytes == nullptr) { set_error("null bytes"); return 2; }
    return tc_convt_bytes(cin, cout, bytes);
}
int dg_pack_convt2x2_tc(const float* w, void* out, int32_t cin, int32_t cout, int32_t dtype, dg_stream_t stream) {
    if (w == nullptr || out == nullptr) { set_error("pack: null pointer"); return 2; }
    return pack_convt_tc(w, out, cin, cout, dtype, reinterpret_cast<cudaStream_t>(stream));
}

int dg_dec_composite_bytes(int32_t cl, int32_t cu, size_t* bytes) {
    if (bytes == nullptr) { set_error("null bytes"); return 2; }
    return dec_composite_bytes(cl, cu, bytes);
}
int dg_pack_dec_composite(const float* ct_w, const float* ct_b, const float* conv_w, void* out, int32_t cl, int32_t cu,
                          int32_t dtype, dg_stream_t stream) {
    if (!ct_w || !ct_b || !conv_w || !out) { set_error("pack: null pointer"); return 2; }
    return pack_dec_composite(ct_w, ct_b, conv_w, out, cl, cu, dtype, reinterpret_cast<cudaStream_t>(stream));
}

int dg_lw_workspace_bytes(const dg_lw_params* p, int32_t N, int32_t H, int32_t W, size_t* bytes) {
    LwPlan pl;
    int rc = make_plan(p, N, H, W, &pl);
    if (rc) return rc;
    if (bytes) *bytes = pl.total_bytes;
    return 0;
}

int dg_lw_layout(const dg_lw_params* p, int32_t N, int32_t H, int32_t W, int32_t idx, size_t* raw_offset,
                 size_t* stats_offset, int32_t* channels, int32_t* h, int32_t* w) {
    LwPlan pl;
    int rc = make_plan(p, N, H, W, &pl);
    if (rc) return rc;
    if (idx < 0 || idx >= 18) { set_error("layout: conv index %d", idx); return 2; }
    if (raw_offset) *raw_offset = pl.raw_off[idx];
    if (stats_offset) *stats_offset = pl.stats_off[idx];
    if (channels) *channels = pl.conv_c[idx];
    if (h) *h = pl.conv_h[idx];
    if (w) *w = pl.conv_w[idx];
    return 0;
}

int dg_lw_forward(const dg_lw_params* p, const float* x, float* y, int32_t N, int32_t H, int32_t W, void* workspace,
                  size_t workspace_bytes, const float* target, double* l1_sum, dg_stream_t stream) {
    return lw_forward(p, x, y, N, H, W, workspace, workspace_bytes, target, l1_sum,
                      reinterpret_cast<cudaStream_t>(stream));
}

int dg_convt2x2_fused(const dg_src* src, int32_t dtype, int32_t N, int32_t H, int32_t W, void* out, float eps, int32_t path,
                      dg_stream_t stream) {
    if (src == nullptr || out == nullptr || N < 1 || H < 2 || W < 2) { set_error("convt2x2: bad arguments"); return 2; }
    int rc = check_path(path, "convt2x2");
    if (rc) return rc;
    rc = validate_src(*src, "convt2x2");
    if (rc) return rc;
    bool handled = false;
    rc = convt_tc_launch(*src, dtype, N, H, W, out, eps, path, reinterpret_cast<cudaStream_t>(stream), &handled);
    if (rc) return rc;
    if (!handled) { set_error("convt2x2: configuration not covered by the tensor-core kernel (use the fused DG_X_CONVT2 source)"); return 3; }
    return 0;
}

int dg_band_stats(const double* kernel_stats, const void* rows, int32_t dtype, int32_t W, int32_t C, int32_t halo_top0, int32_t own0,
                  int32_t own1, int32_t halo_bottom1, double* out, dg_stream_t stream) {
    if (!kernel_stats || !rows || !out || W < 1 || halo_top0 < 0 || halo_top0 > own0 || own0 > own1 || own1 > halo_bottom1) {
        set_error("band_stats: bad arguments");
        return 2;
    }
    return band_stats_launch(kernel_stats, rows, dtype, W, C, halo_top0, own0, own1, halo_bottom1, out, reinterpret_cast<cudaStream_t>(stream));
}

int dg_gn_affine(const double* parts, int32_t nparts, size_t part_stride, const float* gamma, const float* beta, int32_t C, int32_t groups,
                 double plane, float eps, float* coef, dg_stream_t stream) {
    if (!parts || nparts < 1 || !gamma || !beta || !coef || C < 1 || groups < 1 || C % groups || plane <= 0 ||
        (nparts > 1 && part_stride < (size_t)2 * C)) {
        set_error("gn_affine: bad arguments");
        return 2;
    }
    return gn_affine_launch(parts, nparts, part_stride, gamma, beta, C, groups, plane, eps, coef, reinterpret_cast<cudaStream_t>(stream));
}

int dg_channel_attention(const double* act_sum, double plane, const float* w1, const float* w2, int32_t N, int32_t C,
                         int32_t hidden, float* scale, dg_stream_t stream) {
    if (!act_sum || !w1 || !w2 || !scale || N < 1 || C < 1 || hidden < 1 || plane <= 0) {
        set_error("channel_attention: bad arguments");
        return 2;
    }
    return se_scale_launch(act_sum, plane, w1, w2, N, C, hidden, scale, reinterpret_cast<cudaStream_t>(stream));
}

// ---- per-op backward entry points (OptimizedUNet training is orchestrated above the C-ABI from these) ----------------------
static int check_gn(const char* who, const void* raw, const double* stats, const float* gamma, const float* beta, int N, int H, int W,
                    int C, int groups) {
    if (raw == nullptr || stats == nullptr || gamma == nullptr || beta == nullptr) { set_error("%s: null pointer", who); return 2; }
    if (N < 1 || N > 65535 || H < 1 || W < 1 || C < 1) { set_error("%s: bad shape (N must be 1..65535: images are grid.y)", who); return 3; }
    if (groups < 1 || C % groups != 0) { set_error("%s: %d channels not divisible into %d groups", who, C, groups); return 2; }
    return 0;
}

int dg_head1x1_bwd(const dg_head_args* a, const float* grad_y, float* G, double* P, float* dW, float* dB, dg_stream_t stream) {
    if (a == nullptr || grad_y == nullptr || G == nullptr || P == nullptr) {   // dW / dB NULL: that gradient is not computed
        set_error("head backward: null pointer");
        return 2;
    }
    int rc = validate_src(a->src, "head backward");
    if (rc) return rc;
    if (a->src.xform != DG_X_SAME || a->src.stats == nullptr || !a->src.silu || a->src.scale != nullptr || a->src.coef != nullptr) {
        set_error("head backward: the source must be a same-resolution GroupNorm + SiLU tensor described by its statistics");
        return 3;
    }
    if (a->weight == nullptr) { set_error("head backward: null weight"); return 2; }
    return head_bwd_launch(a->dtype, a->src.raw, a->src.stats, a->src.gamma, a->src.beta, grad_y, a->weight, G, P, dW, dB, a->N, a->H,
                           a->W, a->src.channels, a->cout, a->src.groups, a->eps, reinterpret_cast<cudaStream_t>(stream));
}

int dg_act_bwd(int32_t dtype, const void* raw, const double* stats, const float* gamma, const float* beta, int32_t groups,
               const float* dA_a, int32_t stride_a, int32_t off_a, const float* dA_b, int32_t stride_b, int32_t off_b, float* G,
               double* P, int32_t N, int32_t H, int32_t W, int32_t C, float eps, dg_stream_t stream) {
    int rc = check_gn("act backward", raw, stats, gamma, beta, N, H, W, C, groups);
    if (rc) return rc;
    if (G == nullptr || P == nullptr || (dA_a == nullptr && dA_b == nullptr)) { set_error("act backward: null pointer"); return 2; }
    if (dA_b != nullptr && ((H | W) & 1)) { set_error("act backward: pooled gradient needs even H, W"); return 3; }
    if ((dA_a != nullptr && (off_a < 0 || off_a + C > stride_a)) || (dA_b != nullptr && (off_b < 0 || off_b + C > stride_b))) {
        set_error("act backward: channel window outside the gradient tensor");
        return 3;
    }
    return act_bwd_launch(dtype, raw, stats, gamma, beta, dA_a, stride_a, off_a, dA_b, stride_b, off_b, G, P, N, H, W, C, groups, eps,
                          reinterpret_cast<cudaStream_t>(stream));
}

int dg_gn_bwd_apply(int32_t dtype, const void* raw, const double* stats, const float* gamma, int32_t groups, const double* P, float* G,
                    float* dgamma, float* dbeta, int32_t N, int32_t H, int32_t W, int32_t C, float eps, dg_stream_t stream) {
    int rc = check_gn("GroupNorm backward", raw, stats, gamma, gamma, N, H, W, C, groups);
    if (rc) return rc;
    if (P == nullptr || G == nullptr || (dgamma == nullptr) != (dbeta == nullptr)) { set_error("GroupNorm backward: null pointer"); return 2; }
    return gn_bwd_apply_launch(dtype, raw, stats, gamma, P, G, dgamma, dbeta, N, H, W, C, groups, eps,
                               reinterpret_cast<cudaStream_t>(stream));
}

int dg_grad_gather(const float* a, int32_t stride_a, int32_t off_a, const float* a_scale, const float* b, int32_t stride_b,
                   int32_t off_b, const float* u, int32_t stride_u, int32_t off_u, const float* add, float* out, int32_t N, int32_t H,
                   int32_t W, int32_t C, dg_stream_t stream) {
    if (out == nullptr || (a == nullptr && b == nullptr && u == nullptr)) { set_error("grad gather: null pointer"); return 2; }
    if (N < 1 || H < 1 || W < 1 || C < 1) { set_error("grad gather: bad shape"); return 3; }
    if (b != nullptr && ((H | W) & 1)) { set_error("grad gather: pooled gradient needs even H, W"); return 3; }
    if ((a != nullptr && (off_a < 0 || off_a + C > stride_a)) || (b != nullptr && (off_b < 0 || off_b + C > stride_b)) ||
        (u != nullptr && (off_u < 0 || off_u + C > stride_u)) || (a == nullptr && a_scale != nullptr)) {
        set_error("grad gather: channel window outside a gradient tensor");
        return 3;
    }
    return grad_gather_launch(a, stride_a, off_a, a_scale, b, stride_b, off_b, u, stride_u, off_u, add, out, N, H, W, C,
                              reinterpret_cast<cudaStream_t>(stream));
}

int dg_scale_bwd_sum(int32_t dtype, const void* raw, const double* stats, const float* gamma, const float* beta, int32_t groups,
                     const float* d, int32_t stride_d, int32_t off_d, double* dscale, int32_t N, int32_t H, int32_t W, int32_t C,
                     float eps, dg_stream_t stream) {
    int rc = check_gn("scale backward", raw, stats, gamma, beta, N, H, W, C, groups);
    if (rc) return rc;
    if (d == nullptr || dscale == nullptr) { set_error("scale backward: null pointer"); return 2; }
    if (off_d < 0 || off_d + C > stride_d) { set_error("scale backward: channel window outside the gradient tensor"); return 3; }
    if (C > 2048) { set_error("scale backward: %d channels > 2048", C); return 3; }
    return scale_bwd_sum_launch(dtype, raw, stats, gamma, beta, d, stride_d, off_d, dscale, N, H, W, C, groups, eps,
                                reinterpret_cast<cudaStream_t>(stream));
}

int dg_channel_attention_bwd(const double* act_sum, double plane, const float* w1, const float* w2, const double* dscale, int32_t N,
                             int32_t C, int32_t hidden, float* add, float* dw1, float* dw2, dg_stream_t stream) {
    if (act_sum == nullptr || w1 == nullptr || w2 == nullptr || dscale == nullptr) {
        set_error("attention backward: null pointer");
        return 2;
    }
    if ((dw1 == nullptr) != (dw2 == nullptr) || (dw1 == nullptr && add == nullptr)) {
        set_error("attention backward: request dw1 and dw2 together, and at least one of them or add");
        return 2;
    }
    if (N < 1 || C < 1 || hidden < 1 || plane <= 0.0 || (size_t)(2 * C + 3 * hidden) * sizeof(float) > 48 * 1024) {
        set_error("attention backward: bad shape");
        return 3;
    }
    return se_bwd_launch(act_sum, plane, w1, w2, dscale, N, C, hidden, add, dw1, dw2, reinterpret_cast<cudaStream_t>(stream));
}

int dg_lw_num_params(const dg_lw_params* p, size_t* count) {
    LwPlan pl;
    int rc = make_plan(p, 1, 16, 16, &pl);
    if (rc) return rc;
    GradLayout gl;
    make_grad_layout(p, pl, &gl);
    if (count) *count = gl.off[kLwTensors];
    return 0;
}

int dg_lw_backward_workspace_bytes(const dg_lw_params* p, int32_t N, int32_t H, int32_t W, size_t* bytes) {
    LwPlan pl;
    int rc = make_plan(p, N, H, W, &pl);
    if (rc) return rc;
    BwdPlan bp;
    make_bwd_plan(p, pl, N, &bp);
    if (bytes) *bytes = bp.total;
    return 0;
}

int dg_lw_backward(const dg_lw_params* p, const float* x, const float* grad_y, int32_t N, int32_t H, int32_t W,
                   void* fwd_workspace, size_t fwd_bytes, void* bwd_workspace, size_t bwd_bytes, float* grads,
                   dg_stream_t stream) {
    return lw_backward(p, x, grad_y, N, H, W, fwd_workspace, fwd_bytes, bwd_workspace, bwd_bytes, grads, ~0ull, nullptr,
                       reinterpret_cast<cudaStream_t>(stream));
}

int dg_lw_backward_l1(const dg_lw_params* p, const float* x, const float* y, const float* target, const float* loss_grad,
                      int32_t N, int32_t H, int32_t W, void* fwd_workspace, size_t fwd_bytes, void* bwd_workspace, size_t bwd_bytes,
                      float* grads, dg_stream_t stream) {
    if (y == nullptr || target == nullptr) { set_error("backward_l1: null output / target"); return 2; }
    if (p == nullptr) { set_error("null params"); return 2; }
    L1Seed l1{y, target, loss_grad, 1.0f / ((float)N * (float)p->out_channels * (float)H * (float)W)};
    return lw_backward(p, x, nullptr, N, H, W, fwd_workspace, fwd_bytes, bwd_workspace, bwd_bytes, grads, ~0ull, nullptr,
                       reinterpret_cast<cudaStream_t>(stream), &l1);
}

int dg_lw_backward_select(const dg_lw_params* p, const float* x, const dg_lw_bwd_request* r, int32_t N, int32_t H, int32_t W,
                          void* fwd_workspace, size_t fwd_bytes, void* bwd_workspace, size_t bwd_bytes, dg_stream_t stream) {
    if (r == nullptr) { set_error("backward_select: null request"); return 2; }
    const bool l1_seed = r->y != nullptr || r->target != nullptr;
    if ((r->grad_y != nullptr) == l1_seed) {
        set_error("backward_select: give exactly one gradient seed, grad_y or the fused-L1 (y, target)");
        return 2;
    }
    if (l1_seed && (r->y == nullptr || r->target == nullptr)) { set_error("backward_select: the fused-L1 seed needs both y and target"); return 2; }
    if (r->param_mask != 0 && r->grads == nullptr) { set_error("backward_select: param_mask 0x%llx without a grads buffer", (unsigned long long)r->param_mask); return 2; }
    if (r->param_mask == 0 && r->grad_x == nullptr) { set_error("backward_select: nothing requested (param_mask 0, grad_x NULL)"); return 2; }
    if (p == nullptr) { set_error("null params"); return 2; }
    if (int rc = check_path(p->path, "lw")) return rc;
    if (r->grad_x != nullptr && p->conv_w[0][0] == nullptr) { set_error("backward_select: grad_x needs conv_w[0][0]"); return 2; }
    L1Seed l1{r->y, r->target, r->loss_grad, 1.0f / ((float)N * (float)p->out_channels * (float)H * (float)W)};
    return lw_backward(p, x, r->grad_y, N, H, W, fwd_workspace, fwd_bytes, bwd_workspace, bwd_bytes, r->grads, r->param_mask, r->grad_x,
                       reinterpret_cast<cudaStream_t>(stream), l1_seed ? &l1 : nullptr);
}

int dg_conv_first_dgrad(const float* dR, const float* w, float* dx, int32_t N, int32_t H, int32_t W, int32_t cin, int32_t cout,
                        dg_stream_t stream) {
    if (dR == nullptr || w == nullptr || dx == nullptr) { set_error("first dgrad: null pointer"); return 2; }
    return first_dgrad_launch(dR, w, dx, N, H, W, cin, cout, reinterpret_cast<cudaStream_t>(stream));
}

int dg_l1_loss_sum(const float* y, const float* target, size_t count, double* sum, dg_stream_t stream) {
    if (!y || !target || !sum || count == 0) { set_error("l1_loss_sum: bad arguments"); return 2; }
    return l1_sum_launch(y, target, count, sum, reinterpret_cast<cudaStream_t>(stream));
}

int dg_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t count, double* scratch,
                  float max_norm, float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                  float grad_scale, dg_stream_t stream) {
    if (!params || !grads || !exp_avg || !exp_avg_sq || !scratch || count == 0 || step < 1) {
        set_error("adamw: bad arguments");
        return 2;
    }
    return adamw_launch(params, grads, exp_avg, exp_avg_sq, count, scratch, max_norm, lr, beta1, beta2, eps, weight_decay,
                        step, grad_scale, reinterpret_cast<cudaStream_t>(stream));
}

int dg_adamw_step_graph(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t count, double* scratch,
                        float max_norm, const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                        int32_t* step_dev, float grad_scale, dg_stream_t stream) {
    if (!params || !grads || !exp_avg || !exp_avg_sq || !scratch || !lr_dev || !step_dev || count == 0) {
        set_error("adamw (device step): bad arguments");
        return 2;
    }
    return adamw_dev_launch(params, grads, exp_avg, exp_avg_sq, count, scratch, max_norm, lr_dev, beta1, beta2, eps, weight_decay,
                            step_dev, grad_scale, reinterpret_cast<cudaStream_t>(stream));
}

int dg_lw_profile(const dg_lw_params* p, const float* x, float* y, int32_t N, int32_t H, int32_t W, void* workspace,
                  size_t workspace_bytes, dg_stream_t stream, float* ms19) {
    if (ms19 == nullptr) { set_error("profile: null output"); return 2; }
    cudaEvent_t evs[20];
    for (int i = 0; i < 20; ++i) cudaEventCreate(&evs[i]);
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    int rc = lw_forward(p, x, y, N, H, W, workspace, workspace_bytes, nullptr, nullptr, st, evs);
    cudaError_t e = cudaStreamSynchronize(st);
    if (rc == 0 && e != cudaSuccess) { set_error("profile: %s", cudaGetErrorString(e)); rc = 10; }
    if (rc == 0)
        for (int i = 0; i < 19; ++i) cudaEventElapsedTime(&ms19[i], evs[i], evs[i + 1]);
    for (int i = 0; i < 20; ++i) cudaEventDestroy(evs[i]);
    return rc;
}

int dg_lw_host_scratch_bytes(const dg_lw_params* p, int32_t chunk, int32_t H, int32_t W, size_t* bytes) {
    LwPlan pl;
    int rc = make_plan(p, chunk, H, W, &pl);
    if (rc) return rc;
    const size_t in_b = align_up((size_t)chunk * p->in_channels * H * W * sizeof(float), 256);
    const size_t out_b = align_up((size_t)chunk * p->out_channels * H * W * sizeof(float), 256);
    if (bytes) *bytes = dg::HostPipe::NS * (in_b + out_b + align_up(pl.total_bytes, 256));
    return 0;
}

// Chunk i: H2D on s_in -> forward on s_cmp[i % NS] with workspace i % NS -> D2H on s_out.  Several compute streams let the
// under-filled deep layers of one chunk (16 images x 8 tiles < 148 SMs) overlap the next chunk's wide layers.
// ticket == nullptr: blocking call (returns when host_y is complete).  ticket != nullptr: everything is enqueued, *ticket names
// the call for dg_lw_infer_host_wait, and the pipeline keeps running across calls.
static int infer_host_impl(const dg_lw_params* p, const void* host_x, void* host_y, int N, int H, int W, int chunk,
                           void* dev_ws, size_t dev_ws_bytes, int io, cudaStream_t caller, int64_t* ticket = nullptr) {
    if (chunk < 1) { set_error("infer_host: chunk %d", chunk); return 2; }
    if (chunk > N) chunk = N;
    LwPlan pl;
    int rc = make_plan(p, chunk, H, W, &pl);
    if (rc) return rc;
    size_t need = 0;
    dg_lw_host_scratch_bytes(p, chunk, H, W, &need);
    if (dev_ws == nullptr || dev_ws_bytes < need) { set_error("infer_host: scratch %zu < %zu", dev_ws_bytes, need); return 4; }
    if (host_x == nullptr || host_y == nullptr) { set_error("infer_host: null host buffer"); return 2; }
    std::lock_guard<std::mutex> lock(dg::g_pipe_mutex);
    dg::HostPipe* pipe = nullptr;
    if ((rc = dg::pipe_init(&pipe))) return rc;
    const size_t esz_in = (io & 1) ? 1 : sizeof(float), esz_out = (io & 2) ? 1 : sizeof(float);
    const size_t in_img = (size_t)p->in_channels * H * W, out_img = (size_t)p->out_channels * H * W;
    const size_t in_b = align_up(chunk * in_img * sizeof(float), 256);
    const size_t out_b = align_up(chunk * out_img * sizeof(float), 256);
    const size_t ws_b = align_up(pl.total_bytes, 256);
    char* base = static_cast<char*>(dev_ws);
    constexpr int NS = dg::HostPipe::NS;
    char *dx[NS], *dy[NS], *ws[NS];
    for (int k = 0; k < NS; ++k) {
        dx[k] = base + k * in_b;
        dy[k] = base + NS * in_b + k * out_b;
        ws[k] = base + NS * (in_b + out_b) + k * ws_b;
    }
    dg::HostPipe& P = *pipe;
    if (P.ws_in_flight != dev_ws || P.chunk_in_flight != chunk || P.h_in_flight != H || P.w_in_flight != W) {
        // other scratch or geometry than the calls still in flight: their slots are not ours -- drain first
        cudaStreamSynchronize(P.s_out);
        for (int k = 0; k < NS; ++k) cudaStreamSynchronize(P.s_cmp[k]);
        P.seq = 0;
        P.ws_in_flight = dev_ws; P.chunk_in_flight = chunk; P.h_in_flight = H; P.w_in_flight = W;
    }
    // everything the caller enqueued on ITS stream (weight packing after a parameter update, the previous consumer of dev_ws) is
    // ordered before the first kernel of the pipeline
    cudaError_t ce = cudaEventRecord(P.start, caller);
    for (int k = 0; k < NS && ce == cudaSuccess; ++k) ce = cudaStreamWaitEvent(P.s_cmp[k], P.start, 0);
    if (ce != cudaSuccess) { set_error("infer_host: %s", cudaGetErrorString(ce)); return 10; }
    const char* hx = static_cast<const char*>(host_x);
    char* hy = static_cast<char*>(host_y);
    // chunk schedule: a half-size first and last chunk shorten the pipeline fill (first H2D) and drain (last D2H)
    const int head = (ticket == nullptr && N >= 3 * chunk && chunk >= 2) ? chunk / 2 : 0;
    const int body = N - 2 * head;
    const int nchunks = (body + chunk - 1) / chunk + (head ? 2 : 0);
    int n0 = 0;
    for (int i = 0; i < nchunks; ++i, ++P.seq) {
        const int b = (int)(P.seq % NS);
        const bool reuse = P.seq >= (unsigned long long)NS;   // slot b was used by chunk seq - NS (possibly of an earlier call)
        int nn;
        if (head && (i == 0 || i == nchunks - 1)) nn = head;
        else { const int left = N - head - n0; nn = left < chunk ? left : chunk; }  // body: what the tail chunk leaves
        if (reuse) cudaStreamWaitEvent(P.s_in, P.cmp_done[b], 0);  // dx[b] consumed by chunk seq-NS
        ce = cudaMemcpyAsync(dx[b], hx + (size_t)n0 * in_img * esz_in, nn * in_img * esz_in, cudaMemcpyHostToDevice, P.s_in);
        if (ce != cudaSuccess) { cudaDeviceSynchronize(); set_error("infer_host: H2D copy: %s", cudaGetErrorString(ce)); return 10; }
        cudaEventRecord(P.in_done[b], P.s_in);
        cudaStreamWaitEvent(P.s_cmp[b], P.in_done[b], 0);
        if (reuse) cudaStreamWaitEvent(P.s_cmp[b], P.out_done[b], 0);  // dy[b] drained by chunk seq-NS
        rc = dg::lw_forward(p, dx[b], dy[b], nn, H, W, ws[b], pl.total_bytes, nullptr, nullptr, P.s_cmp[b], nullptr, io, 1 + b);
        if (rc) { cudaDeviceSynchronize(); return rc; }
        cudaEventRecord(P.cmp_done[b], P.s_cmp[b]);
        cudaStreamWaitEvent(P.s_out, P.cmp_done[b], 0);
        ce = cudaMemcpyAsync(hy + (size_t)n0 * out_img * esz_out, dy[b], nn * out_img * esz_out, cudaMemcpyDeviceToHost, P.s_out);
        if (ce != cudaSuccess) { cudaDeviceSynchronize(); set_error("infer_host: D2H copy: %s", cudaGetErrorString(ce)); return 10; }
        cudaEventRecord(P.out_done[b], P.s_out);
        n0 += nn;
    }
    if (ticket != nullptr) {   // s_out is one stream: its last copy done = every chunk of this call computed and copied out
        const unsigned long long t = P.tickets++;
        ce = cudaEventRecord(P.ticket_done[t % dg::HostPipe::NT], P.s_out);
        if (ce != cudaSuccess) { cudaDeviceSynchronize(); set_error("infer_host: %s", cudaGetErrorString(ce)); return 10; }
        *ticket = (int64_t)t;
        return 0;
    }
    cudaError_t e = cudaStreamSynchronize(P.s_out);
    for (int k = 0; k < NS && e == cudaSuccess; ++k) e = cudaStreamSynchronize(P.s_cmp[k]);
    if (e != cudaSuccess) { set_error("infer_host: %s", cudaGetErrorString(e)); return 10; }
    return 0;
}

int dg_lw_infer_host(const dg_lw_params* p, const float* host_x, float* host_y, int32_t N, int32_t H, int32_t W,
                     int32_t chunk, void* dev_ws, size_t dev_ws_bytes, dg_stream_t stream) {
    return infer_host_impl(p, host_x, host_y, N, H, W, chunk, dev_ws, dev_ws_bytes, 0, reinterpret_cast<cudaStream_t>(stream));
}

int dg_lw_infer_host_u8(const dg_lw_params* p, const uint8_t* host_x, uint8_t* host_y, int32_t N, int32_t H, int32_t W,
                        int32_t chunk, void* dev_ws, size_t dev_ws_bytes, dg_stream_t stream) {
    return infer_host_impl(p, host_x, host_y, N, H, W, chunk, dev_ws, dev_ws_bytes, 3, reinterpret_cast<cudaStream_t>(stream));
}

int dg_lw_infer_host_submit(const dg_lw_params* p, const void* host_x, void* host_y, int32_t N, int32_t H, int32_t W, int32_t chunk,
                            void* dev_ws, size_t dev_ws_bytes, int32_t u8, dg_stream_t stream, int64_t* ticket) {
    if (ticket == nullptr) { set_error("infer_host_submit: null ticket"); return 2; }
    {   // at most NT calls outstanding: the event about to be re-recorded must have completed
        int dev = 0;
        cudaGetDevice(&dev);
        if (dev >= 0 && dev < 16 && dg::g_pipes[dev].ready && dg::g_pipes[dev].tickets >= (unsigned long long)dg::HostPipe::NT)
            cudaEventSynchronize(dg::g_pipes[dev].ticket_done[dg::g_pipes[dev].tickets % dg::HostPipe::NT]);
    }
    return infer_host_impl(p, host_x, host_y, N, H, W, chunk, dev_ws, dev_ws_bytes, u8 ? 3 : 0, reinterpret_cast<cudaStream_t>(stream), ticket);
}

int dg_lw_infer_host_wait(int64_t ticket) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev < 0 || dev >= 16 || !dg::g_pipes[dev].ready) { set_error("infer_host_wait: no pipeline on this device"); return 2; }
    dg::HostPipe& P = dg::g_pipes[dev];
    if (ticket < 0 || (unsigned long long)ticket >= P.tickets) { set_error("infer_host_wait: unknown ticket %lld", (long long)ticket); return 2; }
    if (P.tickets - (unsigned long long)ticket > (unsigned long long)dg::HostPipe::NT) return 0;   // long retired (submit waited on it)
    cudaError_t e = cudaEventSynchronize(P.ticket_done[(unsigned long long)ticket % dg::HostPipe::NT]);
    if (e != cudaSuccess) { set_error("infer_host_wait: %s", cudaGetErrorString(e)); return 10; }
    return 0;
}

int dg_lw_forward_u8(const dg_lw_params* p, const uint8_t* x, uint8_t* y, int32_t N, int32_t H, int32_t W, void* workspace,
                     size_t workspace_bytes, dg_stream_t stream) {
    return dg::lw_forward(p, x, y, N, H, W, workspace, workspace_bytes, nullptr, nullptr,
                          reinterpret_cast<cudaStream_t>(stream), nullptr, 3);
}

}  // extern "C"
