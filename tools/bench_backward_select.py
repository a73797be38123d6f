"""Time LightweightUNet backwards that compute only what autograd asks for (dg_lw_backward_select), against the full backward.

    python tools/bench_backward_select.py [--batch 32] [--size 512] [--warmup 10] [--iters 100] [--profile]

Shipped weights, fp16 storage, seeded inputs.  Three backwards, each timed with CUDA events around `y.backward(gy)` alone (the
forward runs untimed before every iteration, as it must: backward consumes its workspace):
  full          every parameter, not the input (what training does today)
  frozen_dx     net.requires_grad_(False), x.requires_grad: the input-image gradient only
  decoder_only  encoder and bottleneck frozen: upconv / decoder / head gradients
--profile runs the frozen backward under torch.profiler (a separate run: tracing slows the host) and reports the first conv's
input-gradient kernel against its memory bound: it reads dR0 (N*H*W*C*4 B) and writes dX (N*H*W*in*4 B) once.
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import image_enhancement_deglaring_b200 as dg  # noqa: E402

HBM_TBPS = 6.54   # BASELINE.md: measured copy bandwidth of the B200


def card():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except OSError:
        q = "unknown"
    return name, q


def make(setup, storage):
    net = dg.LightweightUNet(storage=storage)
    net.load_state_dict(torch.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "weights",
                                                "best_model.pth")))
    net = net.cuda().train()
    want_x = setup == "frozen_dx"
    if setup == "frozen_dx":
        net.requires_grad_(False)
    elif setup == "decoder_only":
        for k, p in net.named_parameters():
            p.requires_grad_(not k.startswith(("enc", "bottleneck")))
    return net, want_x


def time_backward(setup, x, gy, warmup, iters, storage):
    net, want_x = make(setup, storage)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for it in range(warmup + iters):
        for p in net.parameters():
            p.grad = None
        xi = x.detach().requires_grad_(want_x)
        y = net(xi)
        if it >= warmup:
            ev[it - warmup][0].record()
        y.backward(gy)
        if it >= warmup:
            ev[it - warmup][1].record()
    torch.cuda.synchronize()
    ts = sorted(a.elapsed_time(b) for a, b in ev)
    return {"median_ms": ts[len(ts) // 2], "mean_ms": sum(ts) / len(ts), "min_ms": ts[0]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--storage", default="fp16")
    ap.add_argument("--profile", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_backward_select: needs a CUDA device")
    name, power = card()
    print(f"card: {name}; power.limit, clocks.max.sm: {power}")
    g = torch.Generator().manual_seed(0)
    shape = (a.batch, 1, a.size, a.size)
    x = torch.rand(shape, generator=g).cuda()
    gy = (torch.randn(shape, generator=g) / x.numel()).cuda()
    if a.profile:
        net, _ = make("frozen_dx", a.storage)
        for _ in range(3):
            net(x.detach().requires_grad_(True)).backward(gy)
        torch.cuda.synchronize()
        reps = 20
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(reps):
                net(x.detach().requires_grad_(True)).backward(gy)
            torch.cuda.synchronize()
        times = [e.device_time for e in prof.events() if "first_dgrad" in e.name]
        C = net.features_start
        bytes_ = a.batch * a.size * a.size * (C + 1) * 4
        bound_us = bytes_ / (HBM_TBPS * 1e12) * 1e6
        # two-stream split: one launch per sub-batch, each over half the batch
        per_bwd = sum(times) / reps
        print(json.dumps({"kernel": "first_dgrad", "launches": len(times), "us_per_backward": round(per_bwd, 2),
                          "bytes": bytes_, "bound_us": round(bound_us, 2), "share_of_bound": round(bound_us / per_bwd, 3),
                          "card": name, "power": power}))
        return
    res = {s: time_backward(s, x, gy, a.warmup, a.iters, a.storage) for s in ("full", "frozen_dx", "decoder_only")}
    for s, r in res.items():
        print(f"{s:13s} median {r['median_ms']:.3f} ms  mean {r['mean_ms']:.3f}  min {r['min_ms']:.3f}")
    print(json.dumps({"batch": a.batch, "size": a.size, "storage": a.storage, "iters": a.iters, "card": name, "power": power,
                      **{s: round(r["median_ms"], 4) for s, r in res.items()}}))


if __name__ == "__main__":
    main()
