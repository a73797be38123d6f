#!/usr/bin/env python
"""Accuracy of storage tiers / kernel paths on the golden PNGs and a seeded random batch (GPU box).
    python tools/accuracy_paths.py [--paths 0,128]
The reference values come from tests/golden (generated from the reference) -- no oracle import here."""
import argparse
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import image_enhancement_deglaring_b200 as dg  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--paths", default="0,128")
ap.add_argument("--storage", default="fp16")
a = ap.parse_args()
g = np.load(os.path.join(ROOT, "tests", "golden", "lw_png.npz"))
sd = torch.load(os.path.join(ROOT, "weights", "best_model.pth"))
for path in [int(p) for p in a.paths.split(",")]:
    net = dg.LightweightUNet(storage=a.storage, path=path)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().eval()
    out = []
    for i in (1, 2):
        x = torch.from_numpy(g[f"x{i}_u8"].astype(np.float32) / 255.0)[None, None].cuda()
        with torch.no_grad():
            y = net(x)[0, 0].cpu().numpy()
        err = np.abs(y - g[f"y{i}"]).max()
        mse = float(((y - g[f"y{i}"]) ** 2).mean())
        out.append(f"png{i} max-abs {err:.3e} psnr {10 * np.log10(1.0 / mse):.1f} dB")
    print(f"storage {a.storage} path {path}: " + "; ".join(out))
