"""Thin per-op wrappers over the C-ABI (used by tests and by the training autograd path).

Tensors are torch CUDA tensors; this module only marshals pointers -- the arithmetic is in csrc/.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import (DG_BF16, DG_F16, DG_F32, DG_X_CONVT2, DG_X_IMAGE, DG_X_POOL2, DG_X_SAME, DG_X_UP2,  # noqa: F401
                   DgConv3x3Args, DgHeadArgs, DgSrc)

TORCH_DTYPE = {DG_F32: torch.float32, DG_F16: torch.float16, DG_BF16: torch.bfloat16}
DTYPE_OF_TORCH = {v: k for k, v in TORCH_DTYPE.items()}


def _ptr(t):
    return None if t is None else t.data_ptr()


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("image_enhancement_deglaring_b200 runs on CUDA tensors only (no CPU fallback)")


def pack_conv3x3(w):
    """nn.Conv2d weight [Co,Ci,3,3] -> [3,3,Ci,Co] fp32 contiguous."""
    return w.detach().float().permute(2, 3, 1, 0).contiguous()


def pack_convt2x2(w):
    """nn.ConvTranspose2d weight [Ci,Co,2,2] -> [2,2,Ci,Co] fp32 contiguous."""
    return w.detach().float().permute(2, 3, 0, 1).contiguous()


def pack_conv3x3_tc(w_packed, dtype, stream=None):
    """fp32 [3,3,Ci,Co] -> the HMMA kernels' B-tile packing in `dtype` (dg_pack_conv3x3_tc); None if unsupported."""
    lib = _lib.load()
    ci, co = int(w_packed.shape[2]), int(w_packed.shape[3])
    n = C.c_size_t(0)
    if dtype == DG_F32 or lib.dg_tc_conv3x3_bytes(ci, co, C.byref(n)) != 0:
        return None
    out = torch.empty(n.value // 2, dtype=TORCH_DTYPE[dtype], device=w_packed.device)
    _lib.check(lib.dg_pack_conv3x3_tc(w_packed.data_ptr(), out.data_ptr(), ci, co, dtype, _stream(stream)))
    return out


def pack_convt2x2_tc(w_packed, dtype, stream=None):
    """fp32 [2,2,Ci,Co] -> tensor-core packing (dg_pack_convt2x2_tc); None if unsupported."""
    lib = _lib.load()
    ci, co = int(w_packed.shape[2]), int(w_packed.shape[3])
    n = C.c_size_t(0)
    if dtype == DG_F32 or lib.dg_tc_convt2x2_bytes(ci, co, C.byref(n)) != 0:
        return None
    out = torch.empty(n.value // 2, dtype=TORCH_DTYPE[dtype], device=w_packed.device)
    _lib.check(lib.dg_pack_convt2x2_tc(w_packed.data_ptr(), out.data_ptr(), ci, co, dtype, _stream(stream)))
    return out


def pack_dec_composite(ct_w_packed, ct_b, conv_w_packed, dtype, stream=None):
    """ConvTranspose2d(2,2)+bias folded into the taps of the 3x3 conv that consumes cat((up, skip)) (dg_pack_dec_composite);
    ct_w_packed fp32 [2,2,Cl,Cu], ct_b [Cu], conv_w_packed fp32 [3,3,2Cu,Cu].  None where the composite kernel has no coverage."""
    lib = _lib.load()
    cl, cu = int(ct_w_packed.shape[2]), int(ct_w_packed.shape[3])
    n = C.c_size_t(0)
    if dtype == DG_F32 or lib.dg_dec_composite_bytes(cl, cu, C.byref(n)) != 0:
        return None
    out = torch.empty(n.value, dtype=torch.uint8, device=ct_w_packed.device)
    _lib.check(lib.dg_pack_dec_composite(ct_w_packed.data_ptr(), ct_b.data_ptr(), conv_w_packed.data_ptr(), out.data_ptr(), cl, cu,
                                         dtype, _stream(stream)))
    return out


def make_src(raw, channels, xform=DG_X_SAME, stats=None, gamma=None, beta=None, groups=1, silu=True,
             scale=None, ct_w=None, ct_b=None, ct_cout=0, ct_w_tc=None):
    _require_cuda(raw, stats, gamma, beta, scale, ct_w, ct_b, ct_w_tc)
    s = DgSrc()
    s.ct_w_tc = _ptr(ct_w_tc)
    s._keep_tc = ct_w_tc
    # the struct only carries raw pointers: pin the tensors to it so temporaries passed inline by the caller
    # stay alive until the launch (after which the caching allocator's stream ordering protects them)
    s._keep = (raw, stats, gamma, beta, scale, ct_w, ct_b)
    s.raw = _ptr(raw)
    s.stats = _ptr(stats)
    s.gamma = _ptr(gamma)
    s.beta = _ptr(beta)
    s.scale = _ptr(scale)
    s.ct_w = _ptr(ct_w)
    s.ct_b = _ptr(ct_b)
    s.channels = channels
    s.groups = groups
    s.xform = xform
    s.silu = 1 if silu else 0
    s.ct_cout = ct_cout
    return s


def _stream(stream):
    return (torch.cuda.current_stream() if stream is None else stream).cuda_stream


def conv3x3_fused(srcs, weight, cout, N, H, W, dtype, out=None, out_stats=None, act_sum=None, path=0, stream=None,
                  eps=1e-5, weight_tc=None, weight_comp=None, want_stats=True):
    """Fused 3x3 conv over the concat of `srcs` (list of DgSrc).  Returns (raw NHWC out, stats [N,cout,2] f64);
    want_stats=False (generic path only, e.g. a data gradient) skips the statistics epilogue and returns None for them."""
    lib = _lib.load()
    dev = weight.device
    if out is None:
        out = torch.empty((N, H, W, cout), dtype=TORCH_DTYPE[dtype], device=dev)
    if out_stats is None and want_stats:
        out_stats = torch.zeros((N, cout, 2), dtype=torch.float64, device=dev)
    a = DgConv3x3Args()
    for i, s in enumerate(srcs):
        a.src[i] = s  # copies the struct; `srcs` (and the tensors pinned to it) outlive the call below
    a.nsrc = len(srcs)
    a.dtype = dtype
    a.N, a.H, a.W, a.cout = N, H, W, cout
    a.weight = _ptr(weight)
    a.weight_tc = _ptr(weight_tc)
    a.weight_comp = _ptr(weight_comp)
    a.out = _ptr(out)
    a.out_stats = _ptr(out_stats)
    a.act_sum = _ptr(act_sum)
    a.eps = eps
    a.path = path
    _lib.check(lib.dg_conv3x3_fused(C.byref(a), _stream(stream)))
    return out, out_stats


def conv3x3_wgrad(srcs, dR, cin_total, cout, N, H, W, dtype, path=0, stream=None, eps=1e-5, out=None):
    """Weight gradient of conv3x3_fused's conv: dW [cout, cin_total, 3, 3] fp32 (the nn.Conv2d.weight layout) from the same
    source descriptions and dR = fp32 NHWC [N,H,W,cout] gradient at the raw conv output.  `out` (contiguous, that many
    elements) is ACCUMULATED into -- e.g. a zeroed window of a flat gradient bucket."""
    lib = _lib.load()
    dW = torch.zeros((cout, cin_total, 3, 3), dtype=torch.float32, device=dR.device) if out is None else out
    if dW.numel() != cout * cin_total * 9 or dW.dtype != torch.float32 or not dW.is_contiguous():
        raise RuntimeError("conv3x3_wgrad: `out` must be a contiguous fp32 tensor of cout*cin*9 elements")
    a = DgConv3x3Args()
    for i, s in enumerate(srcs):
        a.src[i] = s
    a.nsrc = len(srcs)
    a.dtype = dtype
    a.N, a.H, a.W, a.cout = N, H, W, cout
    a.eps = eps
    a.path = path
    _lib.check(lib.dg_conv3x3_wgrad(C.byref(a), _ptr(dR), _ptr(dW), 1, 9, 9 * cin_total, _stream(stream)))
    return dW


def conv3x3_dgrad(dR, weight_tc_bf16, cin, cout, stream=None):
    """Data gradient of the 3x3 conv on the tensor cores (dg_conv3x3_dgrad): dR fp32 NHWC [N,H,W,cout] -> dX fp32 NHWC [N,H,W,cin];
    weight_tc_bf16 = pack_conv3x3_tc(pack_conv3x3(weight), DG_BF16) of the FORWARD weights."""
    _require_cuda(dR, weight_tc_bf16)
    N, H, W, _ = dR.shape
    dX = torch.empty((N, H, W, cin), dtype=torch.float32, device=dR.device)
    _lib.check(_lib.load().dg_conv3x3_dgrad(_ptr(dR), _ptr(weight_tc_bf16), _ptr(dX), N, H, W, cin, cout, _stream(stream)))
    return dX


def conv3x3_dgrad_wide(dR, weight_flip_tc_bf16, cin, cout, stream=None):
    """Data gradient of the 3x3 conv as a tcgen05 implicit GEMM (dg_conv3x3_dgrad_wide; cin >= 32): dR fp32 NHWC [N,H,W,cout] -> dX fp32
    NHWC [N,H,W,cin]; weight_flip_tc_bf16 = pack_conv3x3_tc(flip_conv3x3(weight), DG_BF16)."""
    _require_cuda(dR, weight_flip_tc_bf16)
    N, H, W, _ = dR.shape
    dX = torch.empty((N, H, W, cin), dtype=torch.float32, device=dR.device)
    scratch = torch.empty(dR.numel(), dtype=torch.bfloat16, device=dR.device)
    _lib.check(_lib.load().dg_conv3x3_dgrad_wide(_ptr(dR), _ptr(weight_flip_tc_bf16), _ptr(dX), _ptr(scratch), N, H, W, cin, cout,
                                                 _stream(stream)))
    return dX


def convt2x2_dgrad(dCat, ct_w_tc_bf16, cl, cu, stream=None):
    """Data gradient of ConvTranspose2d(2,2) on the tensor cores (dg_convt2x2_dgrad): the first cu channels of dCat fp32 NHWC
    [N,H,W,stride] -> dLow fp32 NHWC [N,H/2,W/2,cl]; ct_w_tc_bf16 = pack_convt2x2_tc(pack_convt2x2(weight), DG_BF16)."""
    _require_cuda(dCat, ct_w_tc_bf16)
    N, H, W, stride = dCat.shape
    dLow = torch.empty((N, H // 2, W // 2, cl), dtype=torch.float32, device=dCat.device)
    _lib.check(_lib.load().dg_convt2x2_dgrad(_ptr(dCat), stride, _ptr(ct_w_tc_bf16), _ptr(dLow), N, H, W, cl, cu, _stream(stream)))
    return dLow


def head1x1(src, weight, bias, N, H, W, dtype, out=None, target=None, l1_sum=None, stream=None, eps=1e-5):
    lib = _lib.load()
    cout = weight.shape[0]
    if out is None:
        out = torch.empty((N, cout, H, W), dtype=torch.float32, device=weight.device)
    a = DgHeadArgs()
    a.src = src
    a.dtype = dtype
    a.N, a.H, a.W, a.cout = N, H, W, cout
    a.weight = _ptr(weight)
    a.bias = _ptr(bias)
    a.out = _ptr(out)
    a.target = _ptr(target)
    a.l1_sum = _ptr(l1_sum)
    a.eps = eps
    _lib.check(lib.dg_head1x1(C.byref(a), _stream(stream)))
    return out


def channel_attention(act_sum, plane, w1, w2, stream=None):
    """ChannelAttention weights (dg_channel_attention): act_sum [N,C] f64 = pixel sums of the activated tensor (the `act_sum`
    epilogue of the conv that pools it), plane = H*W, w1 [hidden,C], w2 [C,hidden] -> scale [N,C] fp32 (feeds dg_src.scale)."""
    _require_cuda(act_sum, w1, w2)
    N, channels = act_sum.shape
    scale = torch.empty((N, channels), dtype=torch.float32, device=act_sum.device)
    _lib.check(_lib.load().dg_channel_attention(_ptr(act_sum), float(plane), _ptr(w1), _ptr(w2), N, channels, int(w1.shape[0]),
                                                _ptr(scale), _stream(stream)))
    return scale


def convt2x2_fused(src, N, H, W, dtype, out=None, path=0, stream=None, eps=1e-5):
    """Stand-alone tensor-core ConvTranspose2d(2,2)+bias of the activated low-res source -> NHWC [N,H,W,ct_cout]."""
    lib = _lib.load()
    if out is None:
        out = torch.empty((N, H, W, src.ct_cout), dtype=TORCH_DTYPE[dtype], device=src._keep[0].device)
    _lib.check(lib.dg_convt2x2_fused(C.byref(src), dtype, N, H, W, _ptr(out), eps, path, _stream(stream)))
    return out


# ---- per-op backward (OptimizedUNet training; include/deglare.h "per-op backward") ------------------------------------------
def conv3x3_dgrad_generic(dR, weight_flip, cin, N, H, W, out=None, stream=None):
    """Data gradient of a 3x3 conv as the forward generic kernel on an identity fp32 source: dR fp32 NHWC [N,H,W,cout] ->
    dX fp32 NHWC [N,H,W,cin]; weight_flip = flip_conv3x3(weight) ([3,3,cout,cin], taps flipped)."""
    src = make_src(dR, int(dR.shape[-1]), xform=DG_X_SAME, silu=False)
    dX, _ = conv3x3_fused([src], weight_flip, cin, N, H, W, DG_F32, out=out, path=1, stream=stream, want_stats=False)
    return dX


def flip_conv3x3(w):
    """nn.Conv2d weight [Co,Ci,3,3] -> [3,3,Co,Ci] fp32 with the taps flipped: the data gradient is a forward conv with it."""
    return w.detach().float().flip(2, 3).permute(2, 3, 0, 1).contiguous()


def head1x1_bwd(src, weight, grad_y, N, H, W, dtype, G, P, dW, dB, stream=None, eps=1e-5):
    """G / P of the head's source conv; dW / dB accumulated (None: that gradient is not computed)."""
    a = DgHeadArgs()
    a.src = src
    a.dtype = dtype
    a.N, a.H, a.W, a.cout = N, H, W, int(weight.shape[0])
    a.weight = _ptr(weight)
    a.eps = eps
    _require_cuda(grad_y, G, P, dW, dB)
    _lib.check(_lib.load().dg_head1x1_bwd(C.byref(a), _ptr(grad_y), _ptr(G), _ptr(P), _ptr(dW), _ptr(dB), _stream(stream)))


def act_bwd(raw, stats, gamma, beta, groups, dtype, N, H, W, channels, G, P, dA_a=None, off_a=0, dA_b=None, off_b=0, stream=None,
            eps=1e-5):
    """G = (dA_a[..., off_a:off_a+C] + 0.25 * replicate2x2(dA_b[..., off_b:off_b+C])) * SiLU'(GN(raw)); P += (sum G, sum G*xhat)."""
    _require_cuda(raw, stats, gamma, beta, dA_a, dA_b, G, P)
    sa = int(dA_a.shape[-1]) if dA_a is not None else 0
    sb = int(dA_b.shape[-1]) if dA_b is not None else 0
    _lib.check(_lib.load().dg_act_bwd(dtype, _ptr(raw), _ptr(stats), _ptr(gamma), _ptr(beta), groups, _ptr(dA_a), sa, off_a,
                                      _ptr(dA_b), sb, off_b, _ptr(G), _ptr(P), N, H, W, channels, eps, _stream(stream)))


def gn_bwd_apply(raw, stats, gamma, groups, dtype, N, H, W, channels, P, G, dgamma, dbeta, stream=None, eps=1e-5):
    """In place G -> dR (nn.GroupNorm backward), dgamma / dbeta accumulated."""
    _require_cuda(raw, stats, gamma, P, G, dgamma, dbeta)
    _lib.check(_lib.load().dg_gn_bwd_apply(dtype, _ptr(raw), _ptr(stats), _ptr(gamma), groups, _ptr(P), _ptr(G), _ptr(dgamma),
                                           _ptr(dbeta), N, H, W, channels, eps, _stream(stream)))


def grad_gather(N, H, W, channels, a=None, off_a=0, a_scale=None, b=None, off_b=0, u=None, off_u=0, add=None, out=None, stream=None):
    """Dense fp32 [N,H,W,C] gradient at an activated tensor from its consumers' input gradients (dg_grad_gather)."""
    _require_cuda(a, a_scale, b, u, add, out)
    ref = a if a is not None else (b if b is not None else u)
    if out is None:
        out = torch.empty((N, H, W, channels), dtype=torch.float32, device=ref.device)
    st = lambda t: int(t.shape[-1]) if t is not None else 0
    _lib.check(_lib.load().dg_grad_gather(_ptr(a), st(a), off_a, _ptr(a_scale), _ptr(b), st(b), off_b, _ptr(u), st(u), off_u,
                                          _ptr(add), _ptr(out), N, H, W, channels, _stream(stream)))
    return out


def scale_bwd_sum(raw, stats, gamma, beta, groups, dtype, N, H, W, channels, d, off_d, stream=None, eps=1e-5):
    """dscale [N,C] f64 = sum over pixels of d[..., off_d:off_d+C] * SiLU(GN(raw)) (dg_scale_bwd_sum)."""
    _require_cuda(raw, stats, gamma, beta, d)
    out = torch.zeros((N, channels), dtype=torch.float64, device=d.device)
    _lib.check(_lib.load().dg_scale_bwd_sum(dtype, _ptr(raw), _ptr(stats), _ptr(gamma), _ptr(beta), groups, _ptr(d),
                                            int(d.shape[-1]), off_d, _ptr(out), N, H, W, channels, eps, _stream(stream)))
    return out


def channel_attention_bwd(act_sum, plane, w1, w2, dscale, dw1, dw2, want_add=True, stream=None):
    """ChannelAttention backward (dg_channel_attention_bwd): accumulates dw1 / dw2 (both None: skipped), returns add [N,C] fp32
    (None with want_add=False)."""
    _require_cuda(act_sum, w1, w2, dscale, dw1, dw2)
    N, channels = act_sum.shape
    add = torch.empty((N, channels), dtype=torch.float32, device=act_sum.device) if want_add else None
    _lib.check(_lib.load().dg_channel_attention_bwd(_ptr(act_sum), float(plane), _ptr(w1), _ptr(w2), _ptr(dscale), N, channels,
                                                    int(w1.shape[0]), _ptr(add), _ptr(dw1), _ptr(dw2), _stream(stream)))
    return add
