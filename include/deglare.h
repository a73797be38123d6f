/*
 * deglare.h -- C-ABI of the B200-native UNet de-glaring kernels (libdeglare.so).
 *
 * The reference (JTZ18/image-enhancement-deglaring) is 100% Python and has no FFI of
 * its own: its hot path is the nn.Module protocol of src/model.py:LightweightUNet and
 * src/optimized_model.py:OptimizedUNet, executed by torch ATen operators.  This header
 * is the drop-in boundary SURVEY.md section 8(b) specifies: plain pointers and sizes,
 * no torch types, every entry point citing the reference code it replaces.
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless the name says `host`.  The caller (PyTorch's
 *    caching allocator in the shipped binding) owns every buffer; the library keeps no
 *    state between calls except the last error string.
 *  - The caller passes the CUDA stream; nothing in here synchronises the device except
 *    the *_host entry points, which own their private streams and return when the result
 *    is in host memory.
 *  - Return 0 on success, non-zero on error (dg_last_error_string() explains).  Errors are
 *    never thrown across the boundary and there is NO CPU fallback: an unsupported shape
 *    is an error.
 *  - Activations between kernels are "raw" conv outputs (pre-GroupNorm) in NHWC with
 *    storage type `dtype`; GroupNorm statistics travel beside them as per-(n, channel)
 *    double (sum, sum of squares) pairs and are applied, with SiLU, on the CONSUMER's
 *    load.  Pooled / up-sampled / concatenated / normalised tensors never exist in HBM.
 */
#ifndef DEGLARE_H_
#define DEGLARE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* dg_stream_t; /* cudaStream_t */

/* storage type of intermediate activations (accumulation is always fp32) */
enum { DG_F32 = 0, DG_F16 = 1, DG_BF16 = 2 };

/* how a source tensor is mapped onto the consumer conv's input grid */
enum {
    DG_X_SAME = 0,   /* same resolution                                                  */
    DG_X_POOL2 = 1,  /* nn.AvgPool2d(2,2) of the activated source   src/model.py:35-41   */
    DG_X_UP2 = 2,    /* nn.Upsample(x2, nearest)          src/optimized_model.py:112     */
    DG_X_CONVT2 = 3, /* nn.ConvTranspose2d(k=2,s=2)+bias  src/model.py:47-53             */
    DG_X_IMAGE = 4,  /* network input: fp32 NCHW, no norm, no activation                 */
    DG_X_IMAGE_U8 = 5 /* network input: uint8 NCHW, value / 255.0f on load (the /infer normalisation, api/app.py:153) */
};

/* One input of a fused 3x3 conv.  The consumer applies, while staging its halo tile:
 *   y = raw * a_c + b_c          a_c = rstd*gamma_c, b_c = beta_c - mean*a_c   (GroupNorm, src/model.py:94,97)
 *   y = y * sigmoid(y)           if silu                                      (SiLU, src/model.py:95,98)
 *   y = y * scale[n][c]          if scale != NULL   (ChannelAttention, src/optimized_model.py:199-202)
 * then the spatial transform `xform`.  For DG_X_CONVT2 the tensor described by
 * raw/stats/gamma/beta has `channels` = Cin of the transposed conv at half resolution and
 * contributes `ct_cout` channels to the concat. */
typedef struct {
    const void* raw;      /* NHWC [N,Hs,Ws,channels] in `dtype` (fp32 NCHW for DG_X_IMAGE) */
    const double* stats;  /* [N,channels,2] (sum, sumsq) of `raw`; NULL = no GroupNorm     */
    const float* gamma;   /* [channels] GroupNorm weight                                   */
    const float* beta;    /* [channels] GroupNorm bias                                     */
    const float* scale;   /* [N,channels] post-activation multiplier or NULL               */
    const float* ct_w;    /* DG_X_CONVT2: weights packed [2][2][channels][ct_cout] fp32    */
    const float* ct_b;    /* DG_X_CONVT2: bias [ct_cout]                                   */
    const void* ct_w_tc;  /* DG_X_CONVT2: optional tensor-core packing (dg_pack_convt2x2_tc) */
    const float* coef;    /* optional [N,channels,2] finished GroupNorm affine (a, b), e.g. from dg_gn_affine;
                             consumers prefer it over `stats`                                */
    int32_t channels;
    int32_t groups;       /* GroupNorm groups over `channels`                              */
    int32_t xform;        /* DG_X_*                                                        */
    int32_t silu;         /* apply SiLU after the affine                                   */
    int32_t ct_cout;      /* DG_X_CONVT2 only                                              */
    int32_t reserved;
} dg_src;

/* Fused 3x3 conv, stride 1, zero pad 1, no bias, over the channel concat (src[0], src[1]).
 * Replaces, per call, one nn.Conv2d(3x3) of LightweightUNet._block (src/model.py:93,96) /
 * OptimizedUNet._block/_upblock (src/optimized_model.py:91-98,111-116) TOGETHER WITH the
 * GroupNorm+SiLU (+AvgPool2d / ConvTranspose2d / Upsample / torch.cat / ChannelAttention scale)
 * that precede it, and accumulates the GroupNorm statistics of its own output. */
typedef struct {
    dg_src src[2];
    int32_t nsrc;
    int32_t dtype;        /* DG_F32 / DG_F16 / DG_BF16: storage of src raws and of `out`   */
    int32_t N, H, W;      /* output (= conv input grid) size                               */
    int32_t cout;
    const float* weight;  /* packed [3][3][Cin_total][cout] fp32                           */
    const void* weight_tc;/* optional tensor-core packing of the same weights (dg_pack_conv3x3_tc),
                             in `dtype`; NULL = generic CUDA-core path only                 */
    void* out;            /* NHWC [N,H,W,cout] raw conv output                             */
    double* out_stats;    /* [N,cout,2], must be zero on entry; accumulated atomically     */
    double* act_sum;      /* optional [N,src[0].channels]: sum over pixels of the ACTIVATED
                             src[0] (for ChannelAttention's global average); zero on entry  */
    float eps;            /* GroupNorm eps of the sources (1e-5)                           */
    int32_t path;         /* bits 0-1: 0 = auto, 1 = force generic CUDA-core path, 2 = force tensor-core path;
                             bit 7: do not use the tcgen05 kernel (conv3x3_t5.cu); bit 8: insist on it (tests);
                             bit 9 / bit 10: do not use the persistent TMA-fed 8 -> 8 kernel (conv3x3_ring.cu) / the composite
                             decoder kernel (conv3x3_dec.cu).
                             Bits 2-6 and 11 are unused: a call that sets one fails with 2.                                 */
    const void* weight_comp;  /* optional, decoder conv over (DG_X_CONVT2 low, DG_X_SAME skip) only: dg_pack_dec_composite blob --
                                 the ConvTranspose folded into the conv's taps (conv3x3_dec.cu); NULL = stage `up` in the CTA  */
} dg_conv3x3_args;

int dg_conv3x3_fused(const dg_conv3x3_args* args, dg_stream_t stream);

/* Weight gradient of the same fused conv (autograd of src/model.py:93,96 as driven by optimized_train.py:210/226):
 *   dW[tap*s_tap + ci*s_ci + co*s_co] += sum_{n,y,x} A[n, y+ky-1, x+kx-1, ci] * dR[n, y, x, co],   tap = 3*ky + kx,
 * A = the ACTIVATED input rebuilt from args->src exactly as the forward does, dR = fp32 NHWC [N,H,W,cout] gradient at the raw
 * conv output.  dW must be zero (or hold a running sum) on entry; args->weight / out / out_stats are ignored.
 * path bits 0-1 as in dg_conv3x3_fused: the tensor-core kernel (16-bit storage, bf16 operands, fp32 accumulate) covers the
 * LightweightUNet(features_start=8) layers with a ConvTranspose source given MATERIALISED (src[0] = identity `up`). */
int dg_conv3x3_wgrad(const dg_conv3x3_args* args, const float* dR, float* dW, int32_t s_tap, int32_t s_ci, int32_t s_co,
                     dg_stream_t stream);

/* Data gradients on the tensor cores (16-bit tiers of dg_lw_backward; exposed for per-op tests), bf16 operands, fp32 accumulate:
 *   dg_conv3x3_dgrad:  dX[n,y,x,ci] = sum_{ky,kx,co} dR[n, y+1-ky, x+1-kx, co] * W[co][ci][ky][kx]  (autograd of src/model.py:93,96
 *     w.r.t. the conv INPUT); dR fp32 NHWC [N,H,W,cout], dX fp32 NHWC [N,H,W,cin]; weight_tc_bf16 = the FORWARD weights in
 *     dg_pack_conv3x3_tc(..., DG_BF16) packing (read transposed, no second layout).  Covers the (cin, cout) pairs of
 *     LightweightUNet(features_start=8) except the first layer; returns 3 otherwise.
 *   dg_convt2x2_dgrad: dLow[n,i,j,ci] = sum_{a,b,co} dCat[n, 2i+a, 2j+b, co] * Wt[ci][co][a][b] (autograd of src/model.py:47-53) from
 *     the first cu channels of dCat fp32 [N,H,W,stride]; dLow fp32 [N,H/2,W/2,cl]; ct_w_tc_bf16 = dg_pack_convt2x2_tc(..., DG_BF16). */
int dg_conv3x3_dgrad(const float* dR, const void* weight_tc_bf16, float* dX, int32_t N, int32_t H, int32_t W, int32_t cin,
                     int32_t cout, dg_stream_t stream);
int dg_convt2x2_dgrad(const float* dCat, int32_t stride, const void* ct_w_tc_bf16, float* dLow, int32_t N, int32_t H, int32_t W,
                      int32_t cl, int32_t cu, dg_stream_t stream);
/* dg_conv3x3_dgrad_wide: the same data gradient as dg_conv3x3_dgrad for the wide layers (cin >= 32, cin % 32 == 0, cout % 16 == 0;
 * LightweightUNet(features_start=64), BASELINE.json configs[4]) as a tcgen05 implicit GEMM: dR is rounded to bf16 into
 * `scratch_bf16` (N*H*W*cout bf16, caller-owned) and convolved with weight_flip_tc_bf16 = dg_pack_conv3x3_tc of the fp32
 * [3][3][cout][cin] taps-flipped weights (w.flip(2,3).permute(2,3,0,1)) in DG_BF16; dX fp32.  Returns 3 where it has no plan. */
int dg_conv3x3_dgrad_wide(const float* dR, const void* weight_flip_tc_bf16, float* dX, void* scratch_bf16, int32_t N, int32_t H,
                          int32_t W, int32_t cin, int32_t cout, dg_stream_t stream);

/* Output head: GroupNorm+SiLU of the last block, then nn.Conv2d(C, out_channels, 1) + bias
 * (src/model.py:57,131; src/optimized_model.py:74,158).  fp32 (or quantised uint8) NCHW output.  If `target` is
 * given, also accumulates sum|out-target| into *l1_sum (nn.L1Loss forward, optimized_train.py:439). */
typedef struct {
    dg_src src;
    int32_t dtype;
    int32_t N, H, W;
    int32_t cout;
    const float* weight;  /* [cout][channels] */
    const float* bias;    /* [cout]           */
    void* out;            /* [N,cout,H,W] fp32 (out_kind 0) or uint8 (out_kind 1) */
    const float* target;  /* optional [N,cout,H,W] */
    double* l1_sum;       /* optional, zero on entry */
    float eps;
    int32_t out_kind;     /* 0: fp32.  1: uint8 = (uint8)(clip(y, 0, 1) * 255), the /infer post-processing (api/app.py:190-193) */
} dg_head_args;

int dg_head1x1(const dg_head_args* args, dg_stream_t stream);

/* On-device validation metrics (SURVEY 8f4) for fp32 [N,1,H,W] tensors: what optimized_train.py:92-122 / evaluate.py:254-272
 * get per image on the host from skimage's peak_signal_noise_ratio(target, output, data_range) and
 * structural_similarity(target, output, data_range) with default arguments (7x7 uniform window, K1 .01, K2 .03, sample
 * covariance, border cropped).  acc [N][2] doubles, zero on entry: acc[n][0] += sum of squared errors,
 * acc[n][1] += sum of S over the (H-6)(W-6) full windows.  PSNR = 10 log10(R^2 H W / acc[n][0]), SSIM = acc[n][1] / ((H-6)(W-6)).
 * clip01 != 0 clips the OUTPUT to [0, 1] first (evaluate.py:262). */
int dg_image_metrics(const float* output, const float* target, int32_t N, int32_t H, int32_t W, int32_t clip01, double data_range,
                     double* acc, dg_stream_t stream);

/* Stand-alone nn.ConvTranspose2d(k=2, s=2) + bias (src/model.py:47-53) of the ACTIVATED low-resolution tensor described by
 * `src` (xform DG_X_CONVT2 with ct_w_tc / ct_b / ct_cout; GroupNorm + SiLU applied on load), on the tensor cores, 16-bit
 * storage only.  out: NHWC [N,H,W,ct_cout] (H, W = the up-sampled size).  The result is consumed by dg_conv3x3_fused as an
 * identity source (stats = NULL, silu = 0) next to the skip source.  Returns 3 for configurations it does not cover --
 * the fused DG_X_CONVT2 source of dg_conv3x3_fused covers everything. */
int dg_convt2x2_fused(const dg_src* src, int32_t dtype, int32_t N, int32_t H, int32_t W, void* out, float eps, int32_t path,
                      dg_stream_t stream);

/* ChannelAttention of OptimizedUNet (src/optimized_model.py:161-202): scale[n][c] = sigmoid(W2 . silu(W1 . mean)),
 * mean[n][c] = act_sum[n][c] / plane, with act_sum the `act_sum` output of the conv that pools the same tensor.
 * w1 [hidden][C], w2 [C][hidden] (the nn.Linear weights as they are).  The result feeds dg_src.scale. */
int dg_channel_attention(const double* act_sum, double plane, const float* w1, const float* w2, int32_t N, int32_t C,
                         int32_t hidden, float* scale, dg_stream_t stream);

/* ---- per-op backward (autograd of the pieces above; OptimizedUNet training, src/optimized_model.py:118-158 under
 * optimized_train.py:210/226, is orchestrated above the C-ABI from these; LightweightUNet uses dg_lw_backward_select) -
 * Notation per conv i: R = its raw output, y = GroupNorm(R), A = SiLU(y).  Gradient tensors are fp32 NHWC.
 *
 * dg_head1x1_bwd: backward of dg_head1x1 (src/optimized_model.py:74,158) for grad_y = dL/d(out) fp32 [N,cout,H,W] (cout <= 4):
 *   G [N,H,W,C] = dL/dy of the head's source conv, P [N,C,2] += per-(n, c) (sum G, sum G*xhat) (zero on entry),
 *   dW [cout][C] and dB [cout] += the 1x1 conv's parameter gradients (zero on entry, or a running sum); either may be NULL, and
 *   that gradient is then not computed (G and P are the same).  `a` is the forward call's argument block (out / target / l1_sum
 *   ignored).
 * dg_act_bwd: G = (dA_a + 0.25 * replicate2x2(dA_b)) * SiLU'(y) and P += (sum G, sum G*xhat).  dA_a = same-resolution gradient
 *   [N,H,W,stride_a], channels off_a .. off_a+C (one half of a concat gradient is a window of it); dA_b = optional gradient
 *   of the 2x2 average pool of A, [N,H/2,W/2,stride_b] (nn.AvgPool2d backward).  Either may be NULL, not both.
 * dg_gn_bwd_apply: in place G -> dR = rstd * (gamma*G - mean_g(gamma*G) - xhat * mean_g(gamma*G*xhat)) (nn.GroupNorm backward
 *   from the sums P), and dgamma[c] += sum_n P[n][c][1], dbeta[c] += sum_n P[n][c][0] (both NULL = skip). */
int dg_head1x1_bwd(const dg_head_args* a, const float* grad_y, float* G, double* P, float* dW, float* dB, dg_stream_t stream);
int dg_act_bwd(int32_t dtype, const void* raw, const double* stats, const float* gamma, const float* beta, int32_t groups,
               const float* dA_a, int32_t stride_a, int32_t off_a, const float* dA_b, int32_t stride_b, int32_t off_b, float* G,
               double* P, int32_t N, int32_t H, int32_t W, int32_t C, float eps, dg_stream_t stream);
int dg_gn_bwd_apply(int32_t dtype, const void* raw, const double* stats, const float* gamma, int32_t groups, const double* P, float* G,
                    float* dgamma, float* dbeta, int32_t N, int32_t H, int32_t W, int32_t C, float eps, dg_stream_t stream);

/* dg_grad_gather: the gradient at an ACTIVATED tensor A [N,H,W,C] collected from its consumers' input gradients into one dense
 * fp32 tensor:  out = a[.., off_a + c] * a_scale[n][c]  (the skip half of torch.cat((dec, enc * att)), src/optimized_model.py:141-156)
 *                   + 0.25 * b[n, y/2, x/2, off_b + c]   (nn.AvgPool2d(2, 2) backward, :131-135)
 *                   + sum_{dy,dx} u[n, 2y+dy, 2x+dx, off_u + c]   (nn.Upsample(x2, nearest) backward, :112)
 *                   + add[n][c]                          (gradient of ChannelAttention's global mean, dg_channel_attention_bwd)
 * every term optional (a_scale needs a); a [N,H,W,stride_a], b [N,H/2,W/2,stride_b], u [N,2H,2W,stride_u], a_scale / add [N,C]. */
int dg_grad_gather(const float* a, int32_t stride_a, int32_t off_a, const float* a_scale, const float* b, int32_t stride_b,
                   int32_t off_b, const float* u, int32_t stride_u, int32_t off_u, const float* add, float* out, int32_t N, int32_t H,
                   int32_t W, int32_t C, dg_stream_t stream);

/* ChannelAttention backward (src/optimized_model.py:185-202: `x * weights`, weights = fc(avg_pool(x))).
 * dg_scale_bwd_sum: dscale[n][c] += sum_pixels d[n, y, x, off_d + c] * A[n, y, x, c] with A rebuilt from (raw, stats, gamma, beta)
 *   as the forward does; d = the consumer's input gradient [N,H,W,stride_d]; dscale [N,C] double, zero on entry.
 * dg_channel_attention_bwd: from the forward's act_sum / plane / w1 / w2 (dg_channel_attention) and dscale:
 *   dw1 [hidden][C], dw2 [C][hidden] += the two nn.Linear weight gradients summed over the batch (zero on entry or a running
 *   sum); add[n][c] = dL/dmean[n][c] / plane, the constant every pixel of A receives through the global average.
 *   dw1 = dw2 = NULL (both or neither) skips the weight gradients, add = NULL skips the mean's gradient; at least one of the
 *   two must be requested (else 2). */
int dg_scale_bwd_sum(int32_t dtype, const void* raw, const double* stats, const float* gamma, const float* beta, int32_t groups,
                     const float* d, int32_t stride_d, int32_t off_d, double* dscale, int32_t N, int32_t H, int32_t W, int32_t C,
                     float eps, dg_stream_t stream);
int dg_channel_attention_bwd(const double* act_sum, double plane, const float* w1, const float* w2, const double* dscale, int32_t N,
                             int32_t C, int32_t hidden, float* add, float* dw1, float* dw2, dg_stream_t stream);

/* ---- whole-network entry points (native orchestrator) ------------------------------- */

#define DG_MAX_BLOCKS 10  /* enc1-4, bottleneck, dec4-1 */

/* Parameters of a LightweightUNet (src/model.py:14-57).  Device pointers to fp32 tensors:
 * conv weights packed [3][3][Cin][Cout]; ConvTranspose weights packed [2][2][Cin][Cout]. */
typedef struct {
    int32_t in_channels, out_channels, features_start, dtype;
    int32_t groups[DG_MAX_BLOCKS];          /* GroupNorm groups of block b (both norms)    */
    const float* conv_w[DG_MAX_BLOCKS][2];  /* block b: `.0.weight`, `.3.weight`           */
    const float* gn_w[DG_MAX_BLOCKS][2];    /* `.1.weight`, `.4.weight`                    */
    const float* gn_b[DG_MAX_BLOCKS][2];    /* `.1.bias`, `.4.bias`                        */
    const float* up_w[4];                   /* upconv4..upconv1                            */
    const float* up_b[4];
    const void* conv_w_tc[DG_MAX_BLOCKS][2];/* optional tensor-core packings (16-bit dtypes) */
    const void* up_w_tc[4];
    const float* conv_w_flip[DG_MAX_BLOCKS][2]; /* backward only: [3][3][Cout][Cin] with taps flipped
                                               (w.flip(2,3).permute(2,3,0,1)): dgrad is a forward conv */
    const float* up_w_t[4];                 /* backward only: ConvTranspose weights as [2][2][Cout][Cin]   */
    const void* up_w_tc_bf16[4];            /* backward only, optional: dg_pack_convt2x2_tc(..., DG_BF16) for the tensor-core
                                               ConvTranspose data gradient                                    */
    const void* conv_w_tc_bf16[DG_MAX_BLOCKS][2]; /* backward only, optional: dg_pack_conv3x3_tc(..., DG_BF16) of the forward
                                               weights; the tensor-core dgrad reads it transposed (NULL = CUDA-core dgrad) */
    const float* head_w;                    /* output_conv.weight [out][f0]                */
    const float* head_b;
    int32_t path;                           /* dg_conv3x3_args.path: 0 auto, 1 generic, 2 tensor-core, ... */
    int32_t reserved;
    const void* dec_comp[4];                /* optional: dg_pack_dec_composite blobs of (upconv4..1, dec4..1 `.0`) for the
                                               levels with (cl, cu) = (16, 8), the only pair it covers: of the shipped model
                                               only the upconv1 slot [3] is used; NULL elsewhere                       */
    const void* conv_w_flip_tc_bf16[DG_MAX_BLOCKS][2]; /* backward only, optional: dg_pack_conv3x3_tc(conv_w_flip, DG_BF16) -- the
                                               taps-flipped weights in the tensor-core packing: the data gradient of the layers the
                                               mma.sync dgrad does not cover (wider variants, configs[4]) runs as a tcgen05 conv  */
    const void* up_w_dgrad_tc_bf16[4];      /* backward only, optional: the ConvTranspose weights as the [4 Cout][Cin] matrix
                                               W2[(2a+b) Cout + co][ci] = w[ci][co][a][b] in the [K/16][k-half][N][8] tensor-core packing
                                               (dg_pack_convt2x2_tc of its [2][2][4 Cout][Cin/4] view, DG_BF16): the ConvTranspose data
                                               gradient of the wider variants runs as a one-tap tcgen05 GEMM                     */
} dg_lw_params;

/* Bytes of workspace dg_lw_forward needs for an [N,in,H,W] batch (raw activations of all 18
 * convs + statistics; everything backward needs stays live in it). */
int dg_lw_workspace_bytes(const dg_lw_params* p, int32_t N, int32_t H, int32_t W, size_t* bytes);

/* LightweightUNet.forward (src/model.py:101-133): x fp32 [N,in,H,W] -> y fp32 [N,out,H,W].
 * H, W multiples of 16.  Optional target/l1_sum as in dg_head1x1. */
int dg_lw_forward(const dg_lw_params* p, const float* x, float* y, int32_t N, int32_t H, int32_t W,
                  void* workspace, size_t workspace_bytes, const float* target, double* l1_sum,
                  dg_stream_t stream);

/* Byte offset of the raw output of conv `idx` (0..17, forward order) inside the workspace, and of
 * its statistics; for tests and for backward. */
int dg_lw_layout(const dg_lw_params* p, int32_t N, int32_t H, int32_t W, int32_t idx,
                 size_t* raw_offset, size_t* stats_offset, int32_t* channels, int32_t* h, int32_t* w);

/* ---- training (autograd of src/model.py:101-133 as driven by optimized_train.py:206-233) -------
 * dg_lw_backward consumes the workspace a dg_lw_forward of the same batch left behind (raw activations and
 * GroupNorm statistics) and writes EVERY parameter gradient into `grads`, a flat fp32 buffer in the module's
 * parameters() order and the parameters' own layouts (dg_lw_num_params elements, 486,409 for the shipped model):
 *   enc1.0.weight, enc1.1.weight, enc1.1.bias, enc1.3.weight, enc1.4.weight, enc1.4.bias, enc2..., bottleneck...,
 *   upconv4.weight, upconv4.bias, dec4..., upconv3..., dec3..., upconv2..., dec2..., upconv1..., dec1...,
 *   output_conv.weight, output_conv.bias.
 * grad_y is dL/d(output) fp32 [N,out,H,W] (nn.L1Loss backward = sign(o-t)/numel comes from the caller's autograd).
 * dg_lw_backward_l1 below takes the L1 loss's seed instead of grad_y; dg_lw_backward_select computes only a requested subset of
 * the gradients, the input image's included. */
int dg_lw_num_params(const dg_lw_params* p, size_t* count);
int dg_lw_backward_workspace_bytes(const dg_lw_params* p, int32_t N, int32_t H, int32_t W, size_t* bytes);
int dg_lw_backward(const dg_lw_params* p, const float* x, const float* grad_y, int32_t N, int32_t H, int32_t W,
                   void* fwd_workspace, size_t fwd_bytes, void* bwd_workspace, size_t bwd_bytes, float* grads,
                   dg_stream_t stream);

/* nn.L1Loss (optimized_train.py:439) fused into the training path (SURVEY 8a row a10).
 * dg_l1_loss_sum: *sum += sum_i |y_i - target_i| (double, zero on entry); the mean is sum / count.
 * dg_lw_backward_l1: dg_lw_backward for loss = mean |y - target| without a gradient tensor at the output: the head backward
 * generates sign(y - target) * (*loss_grad) / numel itself from the forward output `y` (fp32 [N,out,H,W]) and `target`;
 * `loss_grad` = device pointer to dL/dloss (the GradScaler scale; NULL = 1).  sign(0) = 0 as in torch. */
int dg_l1_loss_sum(const float* y, const float* target, size_t count, double* sum, dg_stream_t stream);
int dg_lw_backward_l1(const dg_lw_params* p, const float* x, const float* y, const float* target, const float* loss_grad,
                      int32_t N, int32_t H, int32_t W, void* fwd_workspace, size_t fwd_bytes, void* bwd_workspace, size_t bwd_bytes,
                      float* grads, dg_stream_t stream);

/* dg_lw_backward_select: the backward of dg_lw_backward / dg_lw_backward_l1 restricted to the gradients a caller asks for -- the
 * input-image gradient and any subset of the 64 parameter tensors (frozen layers, decoder-only fine-tuning).  The kernels of
 * parameter tensors that are not requested do not run, and the backward stops below the lowest requested tensor in forward
 * order (conv i and the GroupNorm after it at position i, an upconv just before the decoder conv that consumes it, the head
 * last, x first).  With every bit of param_mask set and grad_x == NULL it launches exactly what dg_lw_backward launches.
 * Returns 2 when both or neither gradient seed is given, when param_mask != 0 and grads == NULL, and when nothing is requested. */
typedef struct {
    const float* grad_y;      /* dL/dy fp32 [N,out,H,W]; or NULL and the fused-L1 seed below                               */
    const float* y;           /* fused L1 seed (as dg_lw_backward_l1): forward output, target, device dL/dloss or NULL (= 1) */
    const float* target;
    const float* loss_grad;
    float* grads;             /* flat buffer in parameters() order (dg_lw_num_params elements) or NULL                      */
    uint64_t param_mask;      /* bit k = the k-th of the 64 parameter tensors in the order listed above dg_lw_num_params;
                                 only those are written (zeroed, then set), the others are left untouched; 0 = none         */
    float* grad_x;            /* dL/dx fp32 NCHW [N,in,H,W], overwritten; NULL = not wanted                                 */
} dg_lw_bwd_request;

int dg_lw_backward_select(const dg_lw_params* p, const float* x, const dg_lw_bwd_request* r, int32_t N, int32_t H, int32_t W,
                          void* fwd_workspace, size_t fwd_bytes, void* bwd_workspace, size_t bwd_bytes, dg_stream_t stream);

/* dg_conv_first_dgrad: data gradient of the first conv (enc1.0) w.r.t. the input image, the last step of dg_lw_backward_select
 * when grad_x is requested:  dX[n,ci,y,x] = sum_{ky,kx,co} dR[n, y+1-ky, x+1-kx, co] * W[co][ci][ky][kx]  (zero padding).
 * dR fp32 NHWC [N,H,W,cout]; w = the packed fp32 [3][3][cin][cout] weights (dg_lw_params.conv_w[0][0]); dX fp32 NCHW
 * [N,cin,H,W], overwritten.  CUDA cores, fp32; exposed for per-op tests. */
int dg_conv_first_dgrad(const float* dR, const float* w, float* dx, int32_t N, int32_t H, int32_t W, int32_t cin, int32_t cout,
                        dg_stream_t stream);

/* Fused optimizer tail over flat buffers: torch.nn.utils.clip_grad_norm_(max_norm) (skipped if max_norm <= 0) followed by
 * torch.optim.AdamW (optimized_train.py:215-218,230-233,440-446).  grads are first multiplied by grad_scale (1/world after a
 * sum all-reduce).  `scratch` = one device double.  `step` counts from 1. */
int dg_adamw_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t count, double* scratch,
                  float max_norm, float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                  float grad_scale, dg_stream_t stream);

/* The same optimizer tail with nothing baked into the launch: the step count (incremented by the call) and the learning rate are
 * read from DEVICE memory, so a whole training step -- forward, loss, backward, gradient all-reduce, clip, AdamW -- can be captured
 * in a CUDA graph once and replayed (train.GraphedTrainStep): at the reference's own configuration of 4 images per GPU on 8 GPUs
 * (optimized_train.py:383-446 with global batch 32) the step is ~75 launches of 10-50 us kernels and is host-launch bound otherwise. */
int dg_adamw_step_graph(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, size_t count, double* scratch,
                        float max_norm, const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                        int32_t* step_dev, float grad_scale, dg_stream_t stream);

/* One forward with a CUDA-event pair around each of its 19 kernels (18 fused convs + head), recorded on
 * `stream`; synchronises the stream and writes the per-kernel milliseconds to ms19[19].  For bench.py's
 * roofline line -- the events add launch gaps, so use dg_lw_forward for throughput. */
int dg_lw_profile(const dg_lw_params* p, const float* x, float* y, int32_t N, int32_t H, int32_t W,
                  void* workspace, size_t workspace_bytes, dg_stream_t stream, float* ms19);

/* End-to-end inference from HOST buffers (what api/app.py:171 `ort_session.run` and
 * evaluate.py:245 do from the caller's point of view): pipelines H2D copy, forward and D2H
 * copy over `chunk`-image slices on private streams (up to four chunks in flight on their own compute streams,
 * with a workspace each); returns when host_y is complete.
 * host_x/host_y should be pinned for full PCIe rate.  `dev_ws` is caller-owned device scratch of
 * dg_lw_host_scratch_bytes() bytes.  `stream` is the CALLER's stream: the pipeline's private streams wait for everything
 * enqueued on it so far (e.g. the packing kernels of freshly updated weights) before their first kernel.  One pipeline per
 * device; concurrent calls are serialised. */
int dg_lw_host_scratch_bytes(const dg_lw_params* p, int32_t chunk, int32_t H, int32_t W, size_t* bytes);
int dg_lw_infer_host(const dg_lw_params* p, const float* host_x, float* host_y, int32_t N, int32_t H,
                     int32_t W, int32_t chunk, void* dev_ws, size_t dev_ws_bytes, dg_stream_t stream);

/* uint8 in / uint8 out (SURVEY 8f1): what api/app.py:153-193 does around `ort_session.run` -- `img.astype(float32) / 255.0`
 * before, `(np.clip(y, 0, 1) * 255).astype(np.uint8)` after -- folded into the first and the last kernel, so a quarter of
 * the bytes cross PCIe and HBM at both ends.  Bit-identical to running the fp32 entry points on u/255.0f and quantising
 * their output on the host.  Same workspace / scratch sizes as the fp32 entry points. */
int dg_lw_forward_u8(const dg_lw_params* p, const uint8_t* x, uint8_t* y, int32_t N, int32_t H, int32_t W,
                     void* workspace, size_t workspace_bytes, dg_stream_t stream);
int dg_lw_infer_host_u8(const dg_lw_params* p, const uint8_t* host_x, uint8_t* host_y, int32_t N, int32_t H,
                        int32_t W, int32_t chunk, void* dev_ws, size_t dev_ws_bytes, dg_stream_t stream);

/* Row-sharded whole-image inference (SURVEY 8e definition B; whole_image.py): nn.GroupNorm (src/model.py:94,97) normalises over the
 * WHOLE image, so a rank that holds a band of rows contributes the partial sums of the rows it owns, the partial sums of all ranks are
 * exchanged (one all-gather per conv, which carries the halo rows as well), and the consumers take the finished affine through
 * dg_src.coef.
 *  dg_band_stats: `rows` = NHWC [R, W, C] band tensor (N = 1) of which the producing conv computed rows [halo_top0, halo_bottom1) and
 *    the band owns [own0, own1); out[C][2] = kernel_stats[C][2] (the conv's out_stats over every computed row) minus the (sum, sum of
 *    squares) of the computed halo rows.  C <= 1024.
 *  dg_gn_affine: `nparts` blocks of [C][2] partial sums, one every `part_stride` doubles (the gathered packets of all ranks), are added in
 *    block order; `plane` = H_total * W of the whole image at this level -> coef[C][2] = (a, b), y = x * a + b, by the same
 *    double-precision chain the conv kernels run on their own statistics.  C <= 2048. */
int dg_band_stats(const double* kernel_stats, const void* rows, int32_t dtype, int32_t W, int32_t C, int32_t halo_top0, int32_t own0,
                  int32_t own1, int32_t halo_bottom1, double* out, dg_stream_t stream);
int dg_gn_affine(const double* parts, int32_t nparts, size_t part_stride, const float* gamma, const float* beta, int32_t C, int32_t groups,
                 double plane, float eps, float* coef, dg_stream_t stream);

/* Asynchronous twin of dg_lw_infer_host / dg_lw_infer_host_u8 (`u8` != 0) for a service with several requests in flight
 * (uvicorn workers in front of api/app.py:171, evaluate.py:245's loop over batches): _submit enqueues the whole call -- H2D
 * copies, forwards, D2H copies -- and returns a ticket at once; _wait blocks until that call's host_y is complete.  The chunk
 * pipeline runs ACROSS calls (call k+1's first chunks are copied in and computed while call k's last chunks are still being
 * computed / copied out), so with two calls in flight the fill and drain of the pipeline are hidden and larger chunks (which
 * run the kernels at better efficiency) cost no latency.  Calls in flight must share `dev_ws`, `chunk`, H and W (a different
 * combination drains the pipeline first); host_x / host_y must stay valid and untouched until _wait returns; at most 8 calls
 * outstanding (_submit blocks on the oldest).  Tickets are per device. */
int dg_lw_infer_host_submit(const dg_lw_params* p, const void* host_x, void* host_y, int32_t N, int32_t H, int32_t W,
                            int32_t chunk, void* dev_ws, size_t dev_ws_bytes, int32_t u8, dg_stream_t stream, int64_t* ticket);
int dg_lw_infer_host_wait(int64_t ticket);

/* ---- tensor-core weight packing (16-bit storage types) ---------------------------------
 * The HMMA implicit-GEMM kernels read B operands as ldmatrix-ready tiles
 *   [chunk][k-half(2)][cout][8]  of `dtype`,  one chunk = 16 values of K = (tap, cin):
 *   cin >= 16: chunk = tap*(cin/16) + cin/16-block;   cin == 8: chunk j = taps (2j, 2j+1), tap 9 = zeros.
 * `w` is the fp32 [3][3][cin][cout] (resp. [2][2][cin][cout]) packing; returns bytes via *bytes. */
int dg_tc_conv3x3_bytes(int32_t cin, int32_t cout, size_t* bytes);
int dg_pack_conv3x3_tc(const float* w, void* out, int32_t cin, int32_t cout, int32_t dtype, dg_stream_t stream);
int dg_tc_convt2x2_bytes(int32_t cin, int32_t cout, size_t* bytes);
int dg_pack_convt2x2_tc(const float* w, void* out, int32_t cin, int32_t cout, int32_t dtype, dg_stream_t stream);

/* Composite decoder taps (conv3x3_dec.cu): ConvTranspose2d(k=2, s=2)+bias folded into the 3x3 conv that consumes cat((up, skip)).
 * ct_w fp32 [2][2][cl][cu], ct_b [cu], conv_w fp32 [3][3][2 cu][cu] (the packings dg_conv3x3_fused takes); out = blob of
 * *bytes bytes in `dtype` (16-bit only).  Covers only (cl, cu) = (16, 8) -- upconv1 + dec1.0 of LightweightUNet(features_start=8),
 * src/model.py:53,54; any other pair fails with 3. */
int dg_dec_composite_bytes(int32_t cl, int32_t cu, size_t* bytes);
int dg_pack_dec_composite(const float* ct_w, const float* ct_b, const float* conv_w, void* out, int32_t cl, int32_t cu,
                          int32_t dtype, dg_stream_t stream);

/* ---- image pre/post-processing on the device (SURVEY 8 rows f1, f2) ------------------- */
/* Replaces the host calls of api/app.py:143-150 -- `Image.fromarray(img).convert('L')` and `.resize((512, 512), Image.LANCZOS)` -- and
 * of api/app.py:199-203 (resize of the uint8 result back to the upload's size), bit-exactly: Pillow's rgb2l (16-bit fixed point) and
 * its two-pass resampler with 22-bit fixed-point taps and uint8 rounding after each pass (libImaging/Convert.c, Resample.c).
 * src: uint8 [N][in_h][in_w][channels], channels 1 (L), 3 (RGB) or 4 (RGBA, alpha ignored);  dst: uint8 [N][out_h][out_w].
 * bounds_* int32 [out][2] = (first source index, tap count), kk_* int32 [out][ksize_*]: Pillow's precompute_coeffs +
 * normalize_coeffs_8bpc tables (device memory; the host binding computes them, imageops.pil_lanczos_tables).  A pass whose size does
 * not change is skipped as in Pillow (its tables may be NULL).  [row0, row0 + rows) = the source rows the vertical pass reads
 * (Pillow's ybox); tmp holds the horizontal result, N * rows * out_w bytes. */
int dg_pil_resize_u8(const uint8_t* src, int32_t channels, int32_t N, int32_t in_h, int32_t in_w, uint8_t* dst, int32_t out_h,
                     int32_t out_w, const int32_t* bounds_h, const int32_t* kk_h, int32_t ksize_h, const int32_t* bounds_v,
                     const int32_t* kk_v, int32_t ksize_v, int32_t row0, int32_t rows, uint8_t* tmp, size_t tmp_bytes,
                     dg_stream_t stream);

/* Replaces src/optimized_dataset.py:104-123 (and :56-82): the triptych split is the column panel [x_off, x_off + in_w) of an image of
 * width in_w_full (`img[:, :third]`, `img[:, third:2*third]`), then cv2.cvtColor(COLOR_RGB2GRAY) (15-bit fixed point) when
 * channels == 3 and cv2.resize(..., (out_w, out_h)) (INTER_LINEAR on uint8: 11-bit taps; exact 2x down-scaling takes the library's
 * INTER_AREA fast path), bit-exactly.  xofs / yofs int32 [out], xab / yab int32 [out][2]: source index and the two taps per
 * destination index (imageops.cv2_linear_tables).  src uint8 [N][in_h][in_w_full][channels], dst uint8 [N][out_h][out_w]. */
int dg_cv2_resize_u8(const uint8_t* src, int32_t channels, int32_t N, int32_t in_h, int32_t in_w_full, int32_t x_off, int32_t in_w,
                     uint8_t* dst, int32_t out_h, int32_t out_w, const int32_t* xofs, const int32_t* xab, const int32_t* yofs,
                     const int32_t* yab, dg_stream_t stream);

/* Replaces the per-sample albumentations pipeline of src/optimized_dataset.py:126-127,159-172 given the SAMPLED parameters:
 * image / mask uint8 [N][H][W] -> float32 [N][1][H][W] = x / 255; HorizontalFlip of both; on the image only
 * RandomBrightnessContrast = clip(alpha x + beta, 0, 1) and GaussNoise = clip(x + N(0, sigma), 0, 1).
 * params float32 [N][4] = (flip != 0, alpha, beta, sigma); alpha = 1, beta = 0, sigma = 0 switch a transform off.  The noise field
 * comes from a counter-based generator keyed on (seed, sample, pixel) -- not albumentations' stream.  mask / mask_out may be NULL. */
int dg_augment(const uint8_t* image, const uint8_t* mask, float* image_out, float* mask_out, int32_t N, int32_t H, int32_t W,
               const float* params, uint64_t seed, dg_stream_t stream);

/* ---- misc --------------------------------------------------------------------------- */
const char* dg_last_error_string(void);
int dg_version(void);
/* dg_lw_forward / dg_lw_forward_u8 run the two halves of a batch of at least `min_batch` images (default 16) concurrently
 * on two library-private streams forked from and joined to the caller's stream; 0 disables.  Returns the previous value.
 * Results do not depend on it (images are independent). */
int dg_set_batch_split(int min_batch);

/* Programmatic dependent launch for the library's kernel chain (default on); returns the previous setting. */
int dg_set_pdl(int enabled);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t dg_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* DEGLARE_H_ */
