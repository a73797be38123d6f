#!/usr/bin/env python
"""Accuracy / determinism diagnostics on the GPU box (writes a human-readable report to stdout).

  * fp32 / fp16 / bf16 storage, generic vs tensor-core path: max-abs error and PSNR vs the CPU oracle on the two
    golden PNG inputs and on seeded random batches;
  * per-layer raw-activation error (which layer drifts);
  * run-to-run determinism and batch-size independence of the tensor-core path.
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import image_enhancement_deglaring_b200 as dg  # noqa: E402
from oracle import torch_unet as tpo  # noqa: E402

ORDER = ["enc1.0", "enc1.3", "enc2.0", "enc2.3", "enc3.0", "enc3.3", "enc4.0", "enc4.3", "bottleneck.0",
         "bottleneck.3", "dec4.0", "dec4.3", "dec3.0", "dec3.3", "dec2.0", "dec2.3", "dec1.0", "dec1.3"]


def psnr(a, b):
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    return 99.0 if mse == 0 else 10 * np.log10(1.0 / mse)


def net_for(sd, storage, path):
    net = dg.LightweightUNet(storage=storage, path=path)
    net.load_state_dict(sd, strict=True)
    return net.cuda().eval()


def main():
    sd = torch.load(os.path.join(ROOT, "weights", "best_model.pth"))
    g = np.load(os.path.join(ROOT, "tests", "golden", "lw_png.npz"))
    xs = torch.stack([torch.from_numpy(g[f"x{i}_u8"].astype(np.float32) / 255.0)[None] for i in (1, 2)])
    refs = np.stack([g["y1"], g["y2"]])[:, None]
    xr = torch.rand(4, 1, 512, 512, generator=torch.Generator().manual_seed(7))
    with torch.no_grad():
        taps = {}
        ref_r = tpo.lightweight_forward(xr, sd, taps=taps).numpy()
    print("== whole-net error vs oracle (max-abs / PSNR dB) ==")
    for storage in ("fp32", "fp16", "bf16"):
        for path in ((1,) if storage == "fp32" else (1, 0)):
            net = net_for(sd, storage, path)
            with torch.no_grad():
                yp = net(xs.cuda()).cpu().numpy()
                yr = net(xr.cuda()).cpu().numpy()
            print(f"{storage:5s} path={'generic' if path == 1 else 'tensor':7s}: png {np.abs(yp - refs).max():.3e} / "
                  f"{psnr(yp, refs):.1f} dB   random4 {np.abs(yr - ref_r).max():.3e} / {psnr(yr, ref_r):.1f} dB")
            if storage != "fp32":
                errs = []
                for i, name in enumerate(ORDER):
                    raw, _ = net.raw_activation(i, 4, 512, 512)
                    t = taps[name].numpy()
                    errs.append(f"{name}:{float(np.abs(raw.cpu().numpy() - t).max() / max(1.0, np.abs(t).max())):.1e}")
                print("      per-layer rel err:", " ".join(errs))
    print("== determinism (tensor path, fp16) ==")
    net = net_for(sd, "fp16", 0)
    x64 = torch.rand(16, 1, 512, 512, generator=torch.Generator().manual_seed(3)).cuda()
    with torch.no_grad():
        a = net(x64).clone()
        b = net(x64).clone()
        c = net(x64[:4].contiguous()).clone()
    print("run-to-run max diff:", float((a - b).abs().max()), " batch16-vs-batch4 max diff:", float((a[:4] - c).abs().max()))


if __name__ == "__main__":
    main()
