#!/usr/bin/env python
"""One fused conv at a LightweightUNet layer geometry, batch 64, with the t5 kernel's role timeline (DG_T5_TRACE=1) --
debug aid for the warp-specialised pipeline.   DG_T5_TRACE=1 python tools/t5_layer_trace.py same 32 32 128 128"""
import sys, os, time
import numpy as np
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from image_enhancement_deglaring_b200 import ops
mode, cin, cout, H, W = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), int(sys.argv[5])
N = int(sys.argv[6]) if len(sys.argv) > 6 else 64
dt = ops.DG_F16
rs = np.random.RandomState(0)
w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) / np.sqrt(9 * cin)).astype(np.float32)).cuda()
wp = ops.pack_conv3x3(w); wtc = ops.pack_conv3x3_tc(wp, dt)
g = torch.ones(cin).cuda(); b = torch.zeros(cin).cuda()
f = 2 if mode == "pool" else 1
if mode == "dec":   # ConvTranspose + cat + conv as one low-resolution conv: cout = C of the output, H, W = OUTPUT size
    c = cout
    ql = torch.randn(N, H // 2, W // 2, 2 * c, device="cuda").half(); sk = torch.randn(N, H, W, c, device="cuda").half()
    stl = torch.stack((ql.double().sum((1, 2)), (ql.double() ** 2).sum((1, 2))), 2).contiguous()
    sts = torch.stack((sk.double().sum((1, 2)), (sk.double() ** 2).sum((1, 2))), 2).contiguous()
    ctw = torch.randn(2 * c, c, 2, 2, device="cuda") / np.sqrt(2 * c); ctb = torch.randn(c, device="cuda")
    w = torch.randn(c, 2 * c, 3, 3, device="cuda") / np.sqrt(18 * c)
    wp = ops.pack_conv3x3(w); wtc = ops.pack_conv3x3_tc(wp, dt); ctp = ops.pack_convt2x2(ctw)
    g2 = torch.ones(2 * c).cuda(); b2 = torch.zeros(2 * c).cuda()
    srcs = [ops.make_src(ql, 2 * c, xform=ops.DG_X_CONVT2, stats=stl, gamma=g2, beta=b2, groups=8, ct_w=ctp, ct_b=ctb, ct_cout=c,
                         ct_w_tc=ops.pack_convt2x2_tc(ctp, dt)),
            ops.make_src(sk, c, stats=sts, gamma=g2[:c], beta=b2[:c], groups=8)]
    comp = ops.pack_dec_composite(ctp, ctb, wp, dt)
    out = torch.empty(N, H, W, c, device="cuda", dtype=torch.float16)
    stt = torch.zeros(N, c, 2, device="cuda", dtype=torch.float64)
    for it in range(3):
        torch.cuda.synchronize(); t = time.perf_counter()
        ops.conv3x3_fused(srcs, wp, c, N, H, W, dt, out=out, out_stats=stt, path=2 | 256, weight_tc=wtc, weight_comp=comp)
        torch.cuda.synchronize(); print("ms", (time.perf_counter() - t) * 1e3)
    sys.exit(0)
if mode == "cat2":
    up = torch.randn(N, H, W, cout, device="cuda").half(); sk = torch.randn(N, H, W, cout, device="cuda").half()
    st = torch.stack((sk.double().sum((1, 2)), (sk.double() ** 2).sum((1, 2))), 2).contiguous()
    srcs = [ops.make_src(up, cout, silu=False), ops.make_src(sk, cout, stats=st, gamma=g[:cout], beta=b[:cout], groups=8)]
else:
    raw = torch.randn(N, f * H, f * W, cin, device="cuda").half()
    st = torch.stack((raw.double().sum((1, 2)), (raw.double() ** 2).sum((1, 2))), 2).contiguous()
    srcs = [ops.make_src(raw, cin, xform=ops.DG_X_POOL2 if mode == "pool" else ops.DG_X_SAME, stats=st, gamma=g, beta=b, groups=8)]
out = torch.empty(N, H, W, cout, device="cuda", dtype=torch.float16)
stt = torch.zeros(N, cout, 2, device="cuda", dtype=torch.float64)
for it in range(3):
    torch.cuda.synchronize(); t = time.perf_counter()
    ops.conv3x3_fused(srcs, wp, cout, N, H, W, dt, out=out, out_stats=stt, path=2 | 256, weight_tc=wtc)
    torch.cuda.synchronize(); print("ms", (time.perf_counter() - t) * 1e3)
