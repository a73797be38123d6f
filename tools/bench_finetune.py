"""Time one fine-tuning step of a partially frozen network, eager and replayed from a CUDA graph (train.GraphedTrainStep).

    python tools/bench_finetune.py [--batches 4 32] [--size 512] [--warmup 10] [--iters 100] [--models lw opt]

LightweightUNet with the shipped weights and OptimizedUNet with seeded default-initialised weights, fp16 storage, seeded inputs.
Three regimes: full (every parameter trainable), decoder (encoder, bottleneck and attention frozen) and head (only the 1x1 output
conv trainable).  A step is the reference loop's (zero_grad, forward, L1, backward, clip 1.0 folded into FusedAdamW, AdamW); each
of the `iters` steps is timed alone with CUDA events after `warmup` untimed ones, and the median is reported together with the
kernel launches per step (_lib.launch_count; for the graph, averaged over the three warm-up steps and the captured one).  The
card's name, power limit and maximum SM clock are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import image_enhancement_deglaring_b200 as dg  # noqa: E402
from image_enhancement_deglaring_b200 import _lib  # noqa: E402
from image_enhancement_deglaring_b200.train import FusedAdamW, GraphedTrainStep, L1Loss  # noqa: E402

TRAINABLE = {
    "full": lambda k: True,
    "decoder": lambda k: not k.startswith(("enc", "bottleneck", "attention")),
    "head": lambda k: k.startswith(("output_conv", "output.")),
}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError:
        q = "unknown"
    return name, q


def make(model, regime):
    if model == "lw":
        net = dg.LightweightUNet(storage="fp16")
        net.load_state_dict(torch.load(os.path.join(ROOT, "weights", "best_model.pth")))
    else:
        torch.manual_seed(1234)
        net = dg.OptimizedUNet(storage="fp16")
    net = net.cuda().train()
    for k, p in net.named_parameters():
        p.requires_grad_(TRAINABLE[regime](k))
    return net


def time_steps(step, batches, warmup, iters):
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for it in range(warmup + iters):
        x, t = batches[it % len(batches)]
        if it >= warmup:
            ev[it - warmup][0].record()
        step(x, t)
        if it >= warmup:
            ev[it - warmup][1].record()
    torch.cuda.synchronize()
    ms = sorted(a.elapsed_time(b) for a, b in ev)
    return ms[len(ms) // 2]


def bench(model, regime, graphed, batch, size, warmup, iters):
    net = make(model, regime)
    opt = FusedAdamW(net.parameters(), lr=1e-5, weight_decay=1e-2, max_grad_norm=1.0, capturable=graphed)
    crit = L1Loss()
    gen = torch.Generator().manual_seed(0)
    batches = [(torch.rand(batch, 1, size, size, generator=gen).cuda(), torch.rand(batch, 1, size, size, generator=gen).cuda())
               for _ in range(2)]
    if graphed:
        n0 = _lib.launch_count()
        step = GraphedTrainStep(net, opt, crit, batches[0][0].shape, warmup=3)
        launches = (_lib.launch_count() - n0) // 4          # three warm-up steps and the captured one
    else:
        def step(x, t):
            opt.zero_grad(set_to_none=True)
            crit(net(x), t).backward()
            opt.step()
        step(*batches[0])
        n0 = _lib.launch_count()
        step(*batches[0])
        launches = _lib.launch_count() - n0
    ms = time_steps(step, batches, warmup, iters)
    del net, opt, step
    torch.cuda.empty_cache()
    return ms, launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[4, 32])
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--models", nargs="+", default=["lw", "opt"], choices=["lw", "opt"])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_finetune: needs a CUDA device")
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}")
    rows = []
    for model in a.models:
        for batch in a.batches:
            for regime in TRAINABLE:
                for graphed in (False, True):
                    ms, launches = bench(model, regime, graphed, batch, a.size, a.warmup, a.iters)
                    row = dict(model=model, batch=batch, regime=regime, mode="graph" if graphed else "eager", median_ms=round(ms, 3),
                               launches=launches)
                    print(json.dumps(row), flush=True)
                    rows.append(row)
    print(json.dumps({"size": a.size, "storage": "fp16", "warmup": a.warmup, "iters": a.iters, "card": name, "power": power,
                      "rows": rows}))


if __name__ == "__main__":
    main()
