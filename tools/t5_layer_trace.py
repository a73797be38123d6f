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
