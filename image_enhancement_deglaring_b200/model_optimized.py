"""Drop-in `OptimizedUNet` (src/optimized_model.py:6-158) on the B200 fused ops.

Same constructor (`in_channels=1, out_channels=1`), the same 76 state_dict keys / shapes (parameter containers only), and
`forward(x[N,in,H,W]) -> [N,out,H,W]`.  No checkpoint ships for this architecture; parity is taken on deterministic
weights against the reference module (tests/golden/opt_rand.npz forward, opt_train.npz one training step).  Training: under
autograd the forward keeps the raw activations and `_backward` mirrors it op by op (per-op backward entry points of
include/deglare.h; DESIGN.md 3.4).

Mapping onto the fused 3x3 conv (include/deglare.h):
  _block conv .0 / .3          -> DG_X_SAME / DG_X_POOL2 sources (GroupNorm+SiLU[+AvgPool] on load)       :91-98, :33-42
  _upblock (nearest x2 + conv) -> DG_X_UP2 source; its own GroupNorm(4)+SiLU is applied by the consumer   :111-116
  ChannelAttention             -> global mean from the `act_sum` epilogue of the conv that pools the same tensor,
                                  two tiny mat-vecs (dg_channel_attention), scale applied on load (dg_src.scale) :185-202
  torch.cat((up, skip*att))    -> two-source conv, never materialised                                    :140-156
"""
import torch
import torch.nn as nn

from . import _lib, ops
from ._lib import DTYPE_CODES
from .train import _on_device_of, train_forward


def _producers():
    """Which units' outputs each unit reads in `_run`: a unit is a 3x3 conv with its GroupNorm, a ChannelAttention, or the head."""
    enc = ["enc1", "enc2", "enc3", "enc4", "bottleneck"]
    t = {"enc1.0": (), "enc1.3": ("enc1.0",), "head": ("dec1.3",)}
    for lvl in range(1, 5):
        t[enc[lvl] + ".0"] = (enc[lvl - 1] + ".3",)
        t[enc[lvl] + ".3"] = (enc[lvl] + ".0",)
        t[f"attention{lvl}"] = (f"enc{lvl}.3",)
    for k in (4, 3, 2, 1):
        t[f"upconv{k}.1"] = (f"dec{k + 1}.3" if k < 4 else "bottleneck.3",)
        t[f"dec{k}.0"] = (f"upconv{k}.1", f"enc{k}.3", f"attention{k}")
        t[f"dec{k}.3"] = (f"dec{k}.0",)
    return t


def _unit_params(unit):
    if unit == "head":
        return ("output.weight", "output.bias")
    if unit.startswith("attention"):
        return (unit + ".fc.0.weight", unit + ".fc.2.weight")
    blk, idx = unit.rsplit(".", 1)
    return (unit + ".weight", f"{blk}.{int(idx) + 1}.weight", f"{blk}.{int(idx) + 1}.bias")


_PRODUCERS = _producers()
_UNIT_PARAMS = {u: _unit_params(u) for u in _PRODUCERS}


def _upstream():
    """unit -> every unit whose output reaches its inputs (transitively)."""
    up = {}

    def walk(u):
        if u not in up:
            up[u] = set()
            for p in _PRODUCERS[u]:
                up[u] |= {p} | walk(p)
        return up[u]
    for u in _PRODUCERS:
        walk(u)
    return up


_UPSTREAM = _upstream()


class ChannelAttention(nn.Module):
    """Parameter container with the reference's layout (src/optimized_model.py:161-183); evaluated by dg_channel_attention."""

    def __init__(self, channels, reduction=16):
        super().__init__()
        reduced = max(channels // reduction, 8)
        self.avg_pool = nn.AdaptiveAvgPool2d(1)
        self.fc = nn.Sequential(nn.Linear(channels, reduced, bias=False), nn.SiLU(inplace=True),
                                nn.Linear(reduced, channels, bias=False), nn.Sigmoid())


class OptimizedUNet(nn.Module):
    def __init__(self, in_channels=1, out_channels=1, *, storage="fp32", path=0):
        super().__init__()
        if storage not in DTYPE_CODES:
            raise ValueError(f"storage must be one of {sorted(DTYPE_CODES)}")
        self.in_channels, self.out_channels = in_channels, out_channels
        self.storage, self.path = storage, path
        f = self.init_features = 16
        self.enc1 = self._block(in_channels, f, groups=1)
        self.pool1 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.enc2 = self._block(f, f * 2)
        self.pool2 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.enc3 = self._block(f * 2, f * 4)
        self.pool3 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.enc4 = self._block(f * 4, f * 8)
        self.pool4 = nn.AvgPool2d(kernel_size=2, stride=2)
        self.bottleneck = nn.Sequential(
            nn.Conv2d(f * 8, f * 16, kernel_size=3, padding=1, bias=False), nn.GroupNorm(8, f * 16), nn.SiLU(inplace=True),
            nn.Conv2d(f * 16, f * 16, kernel_size=3, padding=1, bias=False), nn.GroupNorm(8, f * 16), nn.SiLU(inplace=True))
        self.attention4 = ChannelAttention(f * 8)
        self.attention3 = ChannelAttention(f * 4)
        self.attention2 = ChannelAttention(f * 2)
        self.attention1 = ChannelAttention(f)
        self.upconv4 = self._upblock(f * 16, f * 8)
        self.dec4 = self._block(f * 16, f * 8)
        self.upconv3 = self._upblock(f * 8, f * 4)
        self.dec3 = self._block(f * 8, f * 4)
        self.upconv2 = self._upblock(f * 4, f * 2)
        self.dec2 = self._block(f * 4, f * 2)
        self.upconv1 = self._upblock(f * 2, f)
        self.dec1 = self._block(f * 2, f)
        self.output = nn.Conv2d(f, out_channels, kernel_size=1)
        self._pack_key = None
        self._pk = None

    @staticmethod
    def _block(in_channels, features, groups=4):
        groups = max(1, min(groups, features))
        return nn.Sequential(
            nn.Conv2d(in_channels, features, kernel_size=3, padding=1, bias=False), nn.GroupNorm(groups, features),
            nn.SiLU(inplace=True),
            nn.Conv2d(features, features, kernel_size=3, padding=1, bias=False), nn.GroupNorm(groups, features),
            nn.SiLU(inplace=True))

    @staticmethod
    def _upblock(in_channels, out_channels):
        return nn.Sequential(nn.Upsample(scale_factor=2, mode="nearest"),
                             nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1, bias=False),
                             nn.GroupNorm(4, out_channels), nn.SiLU(inplace=True))

    # ---- packed parameters -------------------------------------------------------------------------------------------------
    def _packs(self):
        key = tuple((p.data_ptr(), p._version) for p in self.parameters()) + (self.storage, self.path, _lib.generation())
        if key == self._pack_key:
            return self._pk
        dt = DTYPE_CODES[self.storage]
        pk = {}

        pk["_convs"] = []

        def conv(name, m):
            w = ops.pack_conv3x3(m.weight)
            pk[name] = (w, ops.pack_conv3x3_tc(w, dt) if self.path != 1 else None)
            pk["_convs"].append(name)

        def gn(name, m):
            pk[name] = (m.weight.detach().float().contiguous(), m.bias.detach().float().contiguous(), m.num_groups)

        for b in ("enc1", "enc2", "enc3", "enc4", "bottleneck", "dec4", "dec3", "dec2", "dec1"):
            blk = getattr(self, b)
            conv(b + ".0", blk[0]); gn(b + ".1", blk[1]); conv(b + ".3", blk[3]); gn(b + ".4", blk[4])
        for u in ("upconv4", "upconv3", "upconv2", "upconv1"):
            blk = getattr(self, u)
            conv(u + ".1", blk[1]); gn(u + ".2", blk[2])
        for a in ("attention4", "attention3", "attention2", "attention1"):
            fc = getattr(self, a).fc
            pk[a] = (fc[0].weight.detach().float().contiguous(), fc[2].weight.detach().float().contiguous())
        pk["head"] = (self.output.weight.detach().float().reshape(self.out_channels, -1).contiguous(),
                      self.output.bias.detach().float().contiguous())
        self._pk, self._pack_key = pk, key
        return pk

    def _packs_bwd(self):
        """Backward-only weight copies: taps-flipped [3,3,Co,Ci] fp32 for the CUDA-core data gradient and, in the 16-bit tiers,
        the bf16 tensor-core packing of the forward weights the tensor-core data gradient reads transposed."""
        pk = self._packs()
        if pk.get("_bwd") is None:
            bk = {}
            for name in pk["_convs"]:          # every 3x3 conv: "enc1.0" ... "dec1.3", "upconv4.1" ... "upconv1.1"
                v = pk[name]
                blk, idx = name.rsplit(".", 1)
                w = getattr(self, blk)[int(idx)].weight
                tc = tcf = None
                wflip = ops.flip_conv3x3(w)
                if self.storage != "fp32" and (self.path & 3) != 1:
                    tc = ops.pack_conv3x3_tc(v[0], ops.DG_BF16)
                    tcf = ops.pack_conv3x3_tc(wflip, ops.DG_BF16)   # for the tcgen05 data gradient of the pairs mma.sync lacks
                bk[name] = (wflip, tc, tcf)
            pk["_bwd"] = bk
        return pk["_bwd"]

    def forward(self, x):
        _lib.load()
        if not x.is_cuda:
            raise RuntimeError("OptimizedUNet (B200) runs on CUDA tensors only; there is no CPU fallback")
        if self.output.weight.device.type != "cuda":
            raise RuntimeError("OptimizedUNet (B200) needs its parameters on a CUDA device; there is no CPU fallback")
        if x.dim() != 4 or x.shape[1] != self.in_channels:
            raise RuntimeError(f"expected input [N,{self.in_channels},H,W], got {tuple(x.shape)}")
        N, _, H, W = x.shape
        if H % 16 or W % 16 or H < 16 or W < 16:
            raise RuntimeError(f"input {N}x{H}x{W}: H and W must be positive multiples of 16")
        if torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()):
            if x.requires_grad:
                raise NotImplementedError("gradient w.r.t. the input image is not implemented (the reference never needs it)")
            return train_forward(self, x)
        with _on_device_of(x):
            return self._run(x)

    def _run(self, x, keep=None):
        """The forward of src/optimized_model.py:118-158 on the fused ops.  `keep` (training): filled with everything backward
        re-reads -- per conv its raw output, statistics and source descriptions, per attention its squeeze sums and scales."""
        N, _, H, W = x.shape
        x = x.detach().float().contiguous()
        pk = self._packs()
        dt = DTYPE_CODES[self.storage]
        dev = x.device

        def src(t, gnname, xform=ops.DG_X_SAME, scale=None):
            raw, stats, c = t
            g, b, groups = pk[gnname]
            return ops.make_src(raw, c, xform=xform, stats=stats, gamma=g, beta=b, groups=groups, scale=scale)

        def conv(name, srcs, cout, h, w, act_sum=None):
            wp, wtc = pk[name]
            raw, stats = ops.conv3x3_fused(srcs, wp, cout, N, h, w, dt, act_sum=act_sum, path=self.path, weight_tc=wtc)
            if keep is not None:
                keep[name] = dict(raw=raw, stats=stats, c=cout, h=h, w=w, srcs=srcs, cin=int(wp.shape[2]))
            return raw, stats, cout

        def attention(name, t, act_sum, h, w):
            w1, w2 = pk[name]
            scale = ops.channel_attention(act_sum, float(h * w), w1, w2)
            if keep is not None:
                keep[name] = dict(act_sum=act_sum, scale=scale, plane=float(h * w))
            return scale

        f = self.init_features
        chans = [f, f * 2, f * 4, f * 8, f * 16]
        hw = [(H >> i, W >> i) for i in range(5)]
        names = ["enc1", "enc2", "enc3", "enc4", "bottleneck"]
        # encoder: the pooling conv of the next block also reduces the activated skip's global mean (SE squeeze)
        t = conv("enc1.0", [ops.make_src(x, self.in_channels, xform=ops.DG_X_IMAGE, silu=False)], chans[0], *hw[0])
        t = conv("enc1.3", [src(t, "enc1.1")], chans[0], *hw[0])
        skips, scales = [t], []
        for lvl in range(1, 5):
            prev = names[lvl - 1]
            asum = torch.zeros((N, chans[lvl - 1]), dtype=torch.float64, device=dev)
            t = conv(names[lvl] + ".0", [src(skips[-1], prev + ".4", xform=ops.DG_X_POOL2)], chans[lvl], *hw[lvl], act_sum=asum)
            scales.append(attention(f"attention{lvl}", skips[-1], asum, *hw[lvl - 1]))
            t = conv(names[lvl] + ".3", [src(t, names[lvl] + ".1")], chans[lvl], *hw[lvl])
            if lvl < 4:
                skips.append(t)
        # decoder
        d, dname = t, "bottleneck.4"
        for lvl in (3, 2, 1, 0):
            k = lvl + 1
            up = conv(f"upconv{k}.1", [src(d, dname, xform=ops.DG_X_UP2)], chans[lvl], *hw[lvl])
            cat = [src(up, f"upconv{k}.2"), src(skips[lvl], names[lvl] + ".4", scale=scales[lvl])]
            d = conv(f"dec{k}.0", cat, chans[lvl], *hw[lvl])
            d = conv(f"dec{k}.3", [src(d, f"dec{k}.1")], chans[lvl], *hw[lvl])
            dname = f"dec{k}.4"
        hw_, hb = pk["head"]
        hsrc = src(d, dname)
        if keep is not None:
            keep["head"] = hsrc
        return ops.head1x1(hsrc, hw_, hb, N, H, W, dt)

    # ---- training: autograd of the forward above (optimized_train.py:210/226 drives it through loss.backward()) ----------------
    _tc_dgrad_ok = {}   # (cin, cout) -> does the mma.sync data gradient cover the pair (probed once per process)
    _t5_dgrad_ok = {}   # (cin, cout, h, w) -> does the tcgen05 data gradient have a plan

    def _train_forward(self, x):
        """The model half of train._TrainFn: y, and the raw activations the backward re-reads."""
        keep = {}
        return self._run(x, keep), keep

    def _train_backward(self, keep, grad_y, tctx, want_p, grad_x, sink):
        """The gradients of the parameters flagged in `want_p` into `sink`, or into a zeroed buffer in the compact layout over
        them.  No input gradient (the forward refuses an input that requires one) and no fused L1 seed (`tctx` is None)."""
        named = list(self.named_parameters())
        want = [k for (k, _), w in zip(named, want_p) if w]
        grad_y = grad_y.detach().float().contiguous()
        flat = sink if sink is not None else torch.zeros(sum(p.numel() for (_, p), w in zip(named, want_p) if w),
                                                          dtype=torch.float32, device=grad_y.device)
        self._backward(keep, grad_y, flat, want)
        return flat

    def _backward(self, keep, grad_y, flat, want=None):
        """The parameter gradients named in `want` (None: all 76) into `flat`, zero on entry, in parameters() order and the
        parameters' own layouts; `flat` holds either every parameter (unrequested ranges are never written) or only the requested
        ones.  Nothing no request reads is computed: a conv's weight gradient runs only if its weight is requested, its data
        gradient only if a requested tensor lies upstream of its inputs, so the walk stops below the lowest request."""
        pk, bk = self._packs(), self._packs_bwd()
        dt = DTYPE_CODES[self.storage]
        N, _, H, W = grad_y.shape
        dev = grad_y.device
        sizes = {name: p.numel() for name, p in self.named_parameters()}
        want = set(sizes) if want is None else set(want)
        if want - set(sizes):
            raise ValueError(f"OptimizedUNet has no parameters {sorted(want - set(sizes))}")
        req = {u for u, ps in _UNIT_PARAMS.items() if want.intersection(ps)}
        reach = {u for u, up in _UPSTREAM.items() if up & req}     # a gradient at the unit's inputs is needed
        need = reach | req                                            # a gradient at the unit's output is needed
        layout = list(sizes) if flat.numel() == sum(sizes.values()) else [k for k in sizes if k in want]
        views, off = {}, 0
        for name in layout:
            views[name] = flat[off:off + sizes[name]]
            off += sizes[name]
        if off != flat.numel():
            raise ValueError(f"flat gradient of {flat.numel()} elements: expected {sum(sizes.values())} or {off}")
        if not want:
            return
        T = {}   # conv name -> gradient at the conv's input grid, fp32 NHWC [N,h,w,cin_total]

        def outs(*names):
            """Views of the requested tensors of a pair a kernel computes together: None for an unrequested pair, a scratch
            buffer for the unrequested half of a requested one."""
            if not want.intersection(names):
                return (None,) * len(names)
            return tuple(views[k] if k in want else torch.zeros(sizes[k], dtype=torch.float32, device=dev) for k in names)

        def gn_of(name):
            blk, idx = name.rsplit(".", 1)
            return f"{blk}.{int(idx) + 1}"

        def dgrad(name, dR):
            L = keep[name]
            wflip, wtc, wtcf = bk[name]
            key = (L["cin"], L["c"])
            if wtc is not None and OptimizedUNet._tc_dgrad_ok.get(key, True):
                try:
                    return ops.conv3x3_dgrad(dR, wtc, L["cin"], L["c"])
                except RuntimeError as e:   # rc 3 is raised before any launch: the pair is outside the tensor-core kernel's table
                    if "no tensor-core kernel" not in str(e):
                        raise
                    OptimizedUNet._tc_dgrad_ok[key] = False
            wkey = key + (L["h"], L["w"])
            if wtcf is not None and OptimizedUNet._t5_dgrad_ok.get(wkey, True):
                try:
                    return ops.conv3x3_dgrad_wide(dR, wtcf, L["cin"], L["c"])
                except RuntimeError as e:   # likewise: no plan for this shape, nothing was launched
                    if "no tcgen05 plan" not in str(e):
                        raise
                    OptimizedUNet._t5_dgrad_ok[wkey] = False
            return ops.conv3x3_dgrad_generic(dR, wflip, L["cin"], N, L["h"], L["w"])

        def finish(name, G, P):
            """G = dL/dy of conv `name` -> dR in place; GroupNorm / conv parameter gradients; the conv's input gradient."""
            L = keep[name]
            gn = gn_of(name)
            g, _, groups = pk[gn]
            ops.gn_bwd_apply(L["raw"], L["stats"], g, groups, dt, N, L["h"], L["w"], L["c"], P, G,
                             *outs(gn + ".weight", gn + ".bias"))
            if name + ".weight" in want:
                ops.conv3x3_wgrad(L["srcs"], G, L["cin"], L["c"], N, L["h"], L["w"], dt, path=self.path & 3,
                                  out=views[name + ".weight"])
            if name in reach:
                T[name] = dgrad(name, G)

        def act(name, dA, off_a=0):
            L = keep[name]
            g, b, groups = pk[gn_of(name)]
            G = torch.empty((N, L["h"], L["w"], L["c"]), dtype=torch.float32, device=dev)
            P = torch.zeros((N, L["c"], 2), dtype=torch.float64, device=dev)
            ops.act_bwd(L["raw"], L["stats"], g, b, groups, dt, N, L["h"], L["w"], L["c"], G, P, dA_a=dA, off_a=off_a)
            finish(name, G, P)

        # head (src/optimized_model.py:158) and the last conv's activation
        L = keep["dec1.3"]
        G = torch.empty((N, H, W, L["c"]), dtype=torch.float32, device=dev)
        P = torch.zeros((N, L["c"], 2), dtype=torch.float64, device=dev)
        dW, dB = (views[k] if k in want else None for k in ("output.weight", "output.bias"))
        ops.head1x1_bwd(keep["head"], pk["head"][0], grad_y, N, H, W, dt, G, P, dW, dB)
        if "dec1.3" in need:
            finish("dec1.3", G, P)
        # decoder, top level first (:138-156 backwards)
        for k in (1, 2, 3, 4):
            if f"dec{k}.0" in need:
                act(f"dec{k}.0", T.pop(f"dec{k}.3"))
            if f"upconv{k}.1" in need:
                act(f"upconv{k}.1", T[f"dec{k}.0"], 0)                    # first half of torch.cat((dec, enc * att))
            prod = f"dec{k + 1}.3" if k < 4 else "bottleneck.3"           # nn.Upsample(x2, nearest) backward: 2x2 sums
            if prod in need:
                Lp = keep[prod]
                act(prod, ops.grad_gather(N, Lp["h"], Lp["w"], Lp["c"], u=T.pop(f"upconv{k}.1")))
        if "bottleneck.0" in need:
            act("bottleneck.0", T.pop("bottleneck.3"))
        # encoder: each skip tensor feeds the decoder concat (x att), the next level's pool and the attention squeeze
        for lvl in (4, 3, 2, 1):
            name = f"enc{lvl}.3"
            if f"attention{lvl}" not in need:
                T.pop(f"dec{lvl}.0", None)     # the concat gradient, the level's largest tensor: nothing below reads it
                continue
            nxt = "bottleneck.0" if lvl == 4 else f"enc{lvl + 1}.0"
            L = keep[name]
            g, b, groups = pk[gn_of(name)]
            att = keep[f"attention{lvl}"]
            w1, w2 = pk[f"attention{lvl}"]
            tdec = T.pop(f"dec{lvl}.0")
            dscale = ops.scale_bwd_sum(L["raw"], L["stats"], g, b, groups, dt, N, L["h"], L["w"], L["c"], tdec, L["c"])
            dw1, dw2 = outs(f"attention{lvl}.fc.0.weight", f"attention{lvl}.fc.2.weight")
            if name not in need:   # only the attention's own weights are requested
                ops.channel_attention_bwd(att["act_sum"], att["plane"], w1, w2, dscale, dw1, dw2, want_add=False)
                continue
            add = ops.channel_attention_bwd(att["act_sum"], att["plane"], w1, w2, dscale, dw1, dw2)
            dA = ops.grad_gather(N, L["h"], L["w"], L["c"], a=tdec, off_a=L["c"], a_scale=att["scale"], b=T.pop(nxt), add=add)
            del tdec
            act(name, dA)
            del dA
            if f"enc{lvl}.0" in need:
                act(f"enc{lvl}.0", T.pop(name))
