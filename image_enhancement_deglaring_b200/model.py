"""Drop-in `nn.Module` surface of the reference's UNet de-glaring models on B200 kernels.

`LightweightUNet` keeps the constructor, parameter names/shapes/dtypes, `str(model)`, and
`forward(x[N,in,H,W]) -> [N,out,H,W]` contract of /root/reference/src/model.py:9-133, so
`optimized_train.py`, `evaluate.py`, `main.py` and `sweep.py` can construct and call it
unchanged and `best_model.pth` loads with strict=True.  The sub-modules (`enc1.0`, `enc1.1`,
...) exist only as parameter containers with the reference's names and default initialisation;
`forward` never calls them -- it hands raw pointers to libdeglare.so (csrc/), where
Conv3x3 + GroupNorm statistics, GroupNorm-apply + SiLU (+AvgPool / ConvTranspose+concat) on load
and the 1x1 head run as hand-written sm_100a kernels.  No CPU / eager fallback exists.
"""
import ctypes as C

import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import DTYPE_CODES, DgLwParams
from .train import _gather_index, train_forward

_BLOCKS = ("enc1", "enc2", "enc3", "enc4", "bottleneck", "dec4", "dec3", "dec2", "dec1")


class LightweightUNet(nn.Module):
    """Lightweight U-Net with GroupNorm for grayscale image de-glaring (src/model.py:9).

    Extra keyword-only knobs (all optional, defaults keep reference behaviour):
      storage: "fp32" (default; matches the reference to ~1e-5), "fp16" or "bf16" -- HBM storage type of
               the intermediate raw conv outputs (accumulation is always fp32).
      path:    0 auto, 1 force generic CUDA-core kernels, 2 force tensor-core kernels.
    """

    def __init__(self, in_channels=1, out_channels=1, num_groups=8, features_start=8, *, storage="fp32", path=0):
        super().__init__()
        if storage not in DTYPE_CODES:
            raise ValueError(f"storage must be one of {sorted(DTYPE_CODES)}")
        self.num_groups = num_groups
        self.in_channels = in_channels
        self.out_channels = out_channels
        self.features_start = features_start
        self.storage = storage
        self.path = path
        f = [features_start * (1 << i) for i in range(5)]
        self._block_groups = []

        self.enc1 = self._block(in_channels, f[0])
        self.pool1 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.enc2 = self._block(f[0], f[1])
        self.pool2 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.enc3 = self._block(f[1], f[2])
        self.pool3 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.enc4 = self._block(f[2], f[3])
        self.pool4 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.bottleneck = self._block(f[3], f[4])
        self.upconv4 = nn.ConvTranspose2d(f[4], f[3], kernel_size=2, stride=2)
        self.dec4 = self._block(f[3] * 2, f[3])
        self.upconv3 = nn.ConvTranspose2d(f[3], f[2], kernel_size=2, stride=2)
        self.dec3 = self._block(f[2] * 2, f[2])
        self.upconv2 = nn.ConvTranspose2d(f[2], f[1], kernel_size=2, stride=2)
        self.dec2 = self._block(f[1] * 2, f[1])
        self.upconv1 = nn.ConvTranspose2d(f[1], f[0], kernel_size=2, stride=2)
        self.dec1 = self._block(f[0] * 2, f[0])
        self.output_conv = nn.Conv2d(f[0], out_channels, kernel_size=1)

        self._cache = {}   # train flag -> (key, tensors kept alive, dg_lw_params); both variants stay valid side by side
        self._ws = {}

    def _block(self, in_channels, features):
        # group-count rule of src/model.py:69-86: largest divisor of `features` that is <= num_groups
        groups = self.num_groups
        if features < self.num_groups or features % self.num_groups != 0:
            for i in range(min(self.num_groups, features), 0, -1):
                if features % i == 0:
                    groups = i
                    break
        self._block_groups.append(groups)
        return nn.Sequential(
            nn.Conv2d(in_channels, features, kernel_size=3, padding=1, bias=False),
            nn.GroupNorm(num_groups=groups, num_channels=features),
            nn.SiLU(inplace=True),
            nn.Conv2d(features, features, kernel_size=3, padding=1, bias=False),
            nn.GroupNorm(num_groups=groups, num_channels=features),
            nn.SiLU(inplace=True),
        )

    # ---- packed-parameter cache (derived from the fp32 nn.Parameters; refreshed when they change) -----
    def _key(self, train):
        return tuple((p.data_ptr(), p._version) for p in self.parameters()) + (self.storage, self.path, train,
                                                                               _lib.generation())

    def _refresh(self, train=False):
        key = self._key(train)
        hit = self._cache.get(train)
        if hit is not None and hit[0] == key:
            return hit[2]
        dev = self.output_conv.weight.device
        if dev.type != "cuda":
            raise RuntimeError("LightweightUNet (B200) needs its parameters on a CUDA device: call .to('cuda'); "
                               "there is no CPU fallback")
        keep = []
        pc = DgLwParams()
        pc.in_channels, pc.out_channels = self.in_channels, self.out_channels
        pc.features_start = self.features_start
        pc.dtype = DTYPE_CODES[self.storage]
        pc.path = self.path
        for b, name in enumerate(_BLOCKS):
            blk = getattr(self, name)
            pc.groups[b] = self._block_groups[b]
            for j, (ci, gi) in enumerate(((0, 1), (3, 4))):
                w = ops.pack_conv3x3(blk[ci].weight)
                g = blk[gi].weight.detach().float().contiguous()
                bt = blk[gi].bias.detach().float().contiguous()
                wtc = ops.pack_conv3x3_tc(w, pc.dtype) if self.path != 1 else None
                # backward only.  Tensor-core tier (16-bit storage): the mma.sync data gradient reads the bf16 packing of the
                # FORWARD weights transposed (bf16 because dR underflows fp16); it has an instance for every layer of the shipped
                # widths (features_start = 8).  Wider variants (configs[4]) also get the taps-flipped weights in the tensor-core
                # packing for the tcgen05 data gradient (conv3x3_t5.cu, T5_IDENT), and the fp32 flipped weights as the CUDA-core
                # fallback of whatever neither covers.  CUDA-core tier: dgrad = the forward generic conv on the flipped weights.
                tc_tier = train and self.path != 1 and pc.dtype != ops.DG_F32
                tc_only = tc_tier and self.features_start == 8
                wfl = blk[ci].weight.detach().float().flip(2, 3).permute(2, 3, 0, 1).contiguous() if (train and not tc_only) else None
                pc.conv_w_flip[b][j] = None if wfl is None else wfl.data_ptr()
                wbf = wflt = None
                if tc_tier and (b, j) != (0, 0):
                    wbf = wtc if (pc.dtype == ops.DG_BF16 and wtc is not None) else ops.pack_conv3x3_tc(w, ops.DG_BF16)
                    if not tc_only:
                        wflt = ops.pack_conv3x3_tc(wfl, ops.DG_BF16)
                pc.conv_w_tc_bf16[b][j] = None if wbf is None else wbf.data_ptr()
                pc.conv_w_flip_tc_bf16[b][j] = None if wflt is None else wflt.data_ptr()
                keep += [w, g, bt, wtc, wfl, wbf, wflt]
                pc.conv_w_tc[b][j] = None if wtc is None else wtc.data_ptr()
                pc.conv_w[b][j] = w.data_ptr()
                pc.gn_w[b][j] = g.data_ptr()
                pc.gn_b[b][j] = bt.data_ptr()
        for u, name in enumerate(("upconv4", "upconv3", "upconv2", "upconv1")):
            m = getattr(self, name)
            w = ops.pack_convt2x2(m.weight)
            bt = m.bias.detach().float().contiguous()
            wtc = ops.pack_convt2x2_tc(w, pc.dtype) if self.path != 1 else None
            tc_tier = train and self.path != 1 and pc.dtype != ops.DG_F32
            tc_only = tc_tier and self.features_start == 8
            wtt = m.weight.detach().float().permute(2, 3, 1, 0).contiguous() if (train and not tc_only) else None   # [2,2,Co,Ci]
            pc.up_w_t[u] = None if wtt is None else wtt.data_ptr()
            wbf = None
            if tc_tier:
                wbf = wtc if (pc.dtype == ops.DG_BF16 and wtc is not None) else ops.pack_convt2x2_tc(w, ops.DG_BF16)
            pc.up_w_tc_bf16[u] = None if wbf is None else wbf.data_ptr()
            # wider variants: the data gradient as a one-tap tcgen05 GEMM with K = (position, co), N = ci (conv3x3_t5.cu)
            w2t = None
            if tc_tier and not tc_only and m.weight.shape[0] % 32 == 0:
                ci_, co_ = int(m.weight.shape[0]), int(m.weight.shape[1])
                w2 = m.weight.detach().float().permute(2, 3, 1, 0).reshape(4 * co_, ci_)              # [(2a+b) Co + co][ci]
                w2 = w2.reshape(4 * co_, 4, ci_ // 4).permute(1, 0, 2).contiguous().reshape(2, 2, 4 * co_, ci_ // 4)
                w2t = ops.pack_convt2x2_tc(w2, ops.DG_BF16)
            pc.up_w_dgrad_tc_bf16[u] = None if w2t is None else w2t.data_ptr()
            keep.append(w2t)
            # composite decoder taps (ConvTranspose folded into the consuming conv, conv3x3_dec.cu) where that kernel has coverage:
            # level 1 (16 -> 8), forward of both modes
            comp = None
            cu_ = int(w.shape[3])
            if self.path != 1 and pc.dtype != ops.DG_F32 and cu_ == 8:
                dblk = getattr(self, _BLOCKS[5 + u])
                comp = ops.pack_dec_composite(w, bt, ops.pack_conv3x3(dblk[0].weight), pc.dtype)
            pc.dec_comp[u] = None if comp is None else comp.data_ptr()
            keep += [w, bt, wtc, wtt, wbf, comp]
            pc.up_w_tc[u] = None if wtc is None else wtc.data_ptr()
            pc.up_w[u] = w.data_ptr()
            pc.up_b[u] = bt.data_ptr()
        hw = self.output_conv.weight.detach().float().reshape(self.out_channels, -1).contiguous()
        hb = self.output_conv.bias.detach().float().contiguous()
        keep += [hw, hb]
        pc.head_w, pc.head_b = hw.data_ptr(), hb.data_ptr()
        self._cache[train] = (key, keep, pc)
        return pc

    def c_params(self):
        """The dg_lw_params struct (ctypes) for the current parameter values."""
        return self._refresh()

    def workspace_bytes(self, N, H, W):
        n = C.c_size_t(0)
        _lib.check(_lib.load().dg_lw_workspace_bytes(C.byref(self._refresh()), N, H, W, C.byref(n)))
        return n.value

    def _workspace(self, N, H, W, dev):
        k = (N, H, W, self.storage, dev)
        ws = self._ws.get(k)
        if ws is None:
            self._ws.clear()
            ws = torch.empty(self.workspace_bytes(N, H, W), dtype=torch.uint8, device=dev)
            self._ws[k] = ws
        return ws

    def forward(self, x):
        """x: float32 [N, in_channels, H, W] on CUDA, H and W multiples of 16 -> float32 [N, out_channels, H, W]."""
        lib = _lib.load()
        if not x.is_cuda:
            raise RuntimeError("LightweightUNet (B200) runs on CUDA tensors only; there is no CPU fallback")
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise RuntimeError(f"expected input [N,{self.in_channels},H,W], got {tuple(x.shape)}")
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return train_forward(self, x)
        x = x.detach().float().contiguous()
        N, _, H, W = x.shape
        with torch.cuda.device(x.device):   # the library launches on the CURRENT device's stream: make it the tensors' device
            pc = self._refresh()
            ws = self._workspace(N, H, W, x.device)
            y = torch.empty((N, self.out_channels, H, W), dtype=torch.float32, device=x.device)
            _lib.check(lib.dg_lw_forward(C.byref(pc), x.data_ptr(), y.data_ptr(), N, H, W, ws.data_ptr(), ws.numel(),
                                         None, None, torch.cuda.current_stream().cuda_stream))
        return y

    # ---- training: the model half of train._TrainFn ------------------------------------------------------------------------
    _fused_l1 = True   # the backward generates train.L1Loss's gradient seed inside the head backward

    def _train_forward(self, x):
        """y, and what the backward re-reads: a workspace of its own (raw activations, statistics) and x as fp32."""
        x = x.detach().float().contiguous()
        N, _, H, W = x.shape
        pc = self._refresh(train=True)
        ws = torch.empty(self.workspace_bytes(N, H, W), dtype=torch.uint8, device=x.device)
        y = torch.empty((N, self.out_channels, H, W), dtype=torch.float32, device=x.device)
        _lib.check(_lib.load().dg_lw_forward(C.byref(pc), x.data_ptr(), y.data_ptr(), N, H, W, ws.data_ptr(), ws.numel(),
                                             None, None, torch.cuda.current_stream().cuda_stream))
        return y, (ws, x)

    def _train_backward(self, saved, grad_y, tctx, want_p, grad_x, sink):
        """One dg_lw_backward_select for every request: any subset of the parameters, dL/dx or not, grad_y or the fused-L1 seed.
        The native layout is the full one; a sink over a subset of the parameters is filled by one gather from a scratch buffer."""
        lib = _lib.load()
        ws, x = saved
        N, _, H, W = x.shape
        params = list(self.parameters())
        total = sum(p.numel() for p in params)
        if len(want_p) != 64:
            raise RuntimeError(f"gradient layout mismatch: {len(want_p)} parameter tensors, the library's backward has 64")
        mask = sum(1 << k for k, w in enumerate(want_p) if w)
        pc = self._refresh(train=True)
        nb = C.c_size_t(0)
        _lib.check(lib.dg_lw_backward_workspace_bytes(C.byref(pc), N, H, W, C.byref(nb)))
        bws = torch.empty(nb.value, dtype=torch.uint8, device=x.device)
        cnt = C.c_size_t(0)
        _lib.check(lib.dg_lw_num_params(C.byref(pc), C.byref(cnt)))
        if cnt.value != total:
            raise RuntimeError(f"gradient layout mismatch: library {cnt.value} vs module {total}")
        # the backward zeroes the requested ranges itself; a frozen range is never written
        if sink is not None and sink.numel() == total:
            flat = sink
        else:
            flat = torch.empty(total, dtype=torch.float32, device=x.device) if mask else None
        req = _lib.DgLwBwdRequest()
        if (tctx.l1_target is not None and tctx.l1_marker is not None and grad_y.data_ptr() == tctx.l1_marker.data_ptr()
                and all(s == 0 for s in grad_y.stride())):
            # loss = train.L1Loss: the seed sign(y - t) * dloss / numel is generated inside the head backward
            req.y, req.target, req.loss_grad = tctx.y.data_ptr(), tctx.l1_target.data_ptr(), tctx.l1_scale.data_ptr()
        else:
            grad_y = grad_y.detach().float().contiguous()
            req.grad_y = grad_y.data_ptr()
        req.grads = flat.data_ptr() if flat is not None else None
        req.param_mask = mask
        req.grad_x = grad_x.data_ptr() if grad_x is not None else None
        _lib.check(lib.dg_lw_backward_select(C.byref(pc), x.data_ptr(), C.byref(req), N, H, W, ws.data_ptr(), ws.numel(),
                                             bws.data_ptr(), bws.numel(), torch.cuda.current_stream().cuda_stream))
        if sink is not None and sink is not flat:
            torch.index_select(flat, 0, _gather_index(self, params, want_p, flat.device), out=sink)
            return sink
        return flat

    def forward_u8(self, x):
        """uint8 in, uint8 out: the /infer pre/post-processing of api/app.py:153,190-193 folded into the first and last
        kernel -- `x.float() / 255.0` on load, `(clip(y, 0, 1) * 255).to(uint8)` on store.  x: uint8 [N,in,H,W] on CUDA.
        Bit-identical to quantising `forward(x.float() / 255.0)`; inference only."""
        lib = _lib.load()
        if not x.is_cuda or x.dtype != torch.uint8:
            raise RuntimeError("forward_u8 expects a uint8 CUDA tensor")
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise RuntimeError(f"expected input [N,{self.in_channels},H,W], got {tuple(x.shape)}")
        x = x.contiguous()
        N, _, H, W = x.shape
        with torch.cuda.device(x.device):
            pc = self._refresh()
            ws = self._workspace(N, H, W, x.device)
            y = torch.empty((N, self.out_channels, H, W), dtype=torch.uint8, device=x.device)
            _lib.check(lib.dg_lw_forward_u8(C.byref(pc), x.data_ptr(), y.data_ptr(), N, H, W, ws.data_ptr(), ws.numel(),
                                            torch.cuda.current_stream().cuda_stream))
        return y

    # ---- debugging / test hooks ----------------------------------------------------------------------
    def raw_activation(self, idx, N, H, W):
        """View of the raw output of conv `idx` (0..17) from the last forward at this shape, as NCHW fp32."""
        lib = _lib.load()
        ro, so = C.c_size_t(0), C.c_size_t(0)
        c, h, w = C.c_int32(0), C.c_int32(0), C.c_int32(0)
        _lib.check(lib.dg_lw_layout(C.byref(self._refresh()), N, H, W, idx, C.byref(ro), C.byref(so), C.byref(c),
                                    C.byref(h), C.byref(w)))
        ws = next(iter(self._ws.values()))
        tdt = ops.TORCH_DTYPE[DTYPE_CODES[self.storage]]
        nbytes = N * h.value * w.value * c.value * torch.empty((), dtype=tdt).element_size()
        raw = ws[ro.value:ro.value + nbytes].view(tdt).view(N, h.value, w.value, c.value)
        stats = ws[so.value:so.value + N * c.value * 16].view(torch.float64).view(N, c.value, 2)
        return raw.permute(0, 3, 1, 2).float(), stats


def count_parameters(model):
    """src/model.py:364 -- number of trainable parameters."""
    return sum(p.numel() for p in model.parameters() if p.requires_grad)


def get_model_size_mb(model):
    """src/model.py:377 -- state_dict size in MiB."""
    return sum(v.element_size() * v.nelement() for v in model.state_dict().values()) / (1024 * 1024)
