#!/usr/bin/env python
"""Headline benchmark: LightweightUNet de-glaring inference, images/sec (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W

A step = one forward pass of the 486,409-parameter best_model UNet over one batch of 64 synthetic
1x512x512 grayscale images per GPU (BASELINE.json configs[1]); batches shard over GPUs with no
collective (weak scaling).  `value` is device-resident throughput (CUDA events, max over ranks);
`e2e` goes through the session API with pinned HOST buffers, every step's H2D + D2H inside the timed region:
`InferenceSession.submit` / `wait` -> `dg_lw_infer_host_submit` / `_wait` with two batches in flight (the service shape; `e2e.blocking`
is the one-batch-at-a-time `run_pinned` -> `dg_lw_infer_host` call; `e2e_u8`: the uint8-in / uint8-out twins).  `train_step` is one
BASELINE.json configs[3] training step (batch 32 per GPU) in the same storage tier; `latency_n1` is configs[0] (fp32, batch 1) and
`wide` configs[4] (features_start=64 on the tcgen05 kernel), both rank 0 only.  `roofline` is for the dominant kernel,
timed live with CUDA events by `dg_lw_profile` (whole batch on one stream; the timed steps themselves run the batch as two
concurrent halves, see DESIGN.md section 5).  `cpu_baseline` / `--impl reference` time the reference's
PyTorch-CPU path on all host cores: the unmodified reference module when oracle/_ref exists (oracle/build_ref.py puts it there in
the build container; it travels to the GPU box with the snapshot), else the pinned oracle port oracle/torch_unet.py.
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "unet_deglare_512x512_images_per_sec"
UNIT = "images/s"
LAYERS = ["enc1.0", "enc1.3", "enc2.0", "enc2.3", "enc3.0", "enc3.3", "enc4.0", "enc4.3", "bottleneck.0",
          "bottleneck.3", "up4+dec4.0", "dec4.3", "up3+dec3.0", "dec3.3", "up2+dec2.0", "dec2.3", "up1+dec1.0",
          "dec1.3", "head"]


def algorithmic_bytes_per_image(H, W, fs=8, esize=2):
    """SURVEY.md section 8(d) minimal-traffic model, per kernel: every raw conv output written once and read once
    per consumer, input fp32 read once, output fp32 written once; pooled/up-sampled/concat tensors never stored."""
    f = [fs << i for i in range(5)]
    px = [(H >> i) * (W >> i) for i in range(5)]
    out = []
    out.append(px[0] * 4 + px[0] * f[0] * esize)                                   # enc1.0: image in, raw out
    out.append(2 * px[0] * f[0] * esize)                                            # enc1.3
    for l in range(1, 5):
        out.append(px[l - 1] * f[l - 1] * esize + px[l] * f[l] * esize)             # encL.0 reads full-res producer
        out.append(2 * px[l] * f[l] * esize)                                        # encL.3
    for l in (3, 2, 1, 0):
        out.append(px[l + 1] * f[l + 1] * esize + 2 * px[l] * f[l] * esize)         # up + dec.0: low, skip, out
        out.append(2 * px[l] * f[l] * esize)                                        # dec.3
    out.append(px[0] * f[0] * esize + px[0] * 4)                                    # head
    return out


def training_algorithmic_bytes_per_image(H, W, fs=8, esize=2):
    """Minimal-traffic model of one training step (DESIGN.md section 5): the forward bytes, plus in backward, for every raw conv
    output X (18 tensors, E elements each): X re-read twice (by its own GroupNorm/SiLU backward and as the recomputed input of
    its consumer's weight gradient), its gradient written once and read twice (data- and weight-gradient of the producing conv),
    all in the 16-bit storage type -> 5 * esize bytes per element; plus target and output (fp32) read once by the loss."""
    fwd = sum(algorithmic_bytes_per_image(H, W, fs, esize))
    f = [fs << i for i in range(5)]
    px = [(H >> i) * (W >> i) for i in range(5)]
    elems = 2 * sum(px[l] * f[l] for l in range(5)) + 2 * sum(px[l] * f[l] for l in range(4))   # enc + bottleneck, dec
    return fwd + 5 * esize * elems + 2 * px[0] * 4


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe): NVML polled every few milliseconds
    from a thread (the timed region of the default run is tens of milliseconds, nvidia-smi's 100 ms loop gave it 2-3 samples);
    `nvidia-smi -lms 100` is the fallback when the NVML binding is missing."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []     # (time, sm_mhz, reasons bitmask)
        self.smax = None
        self._stop = threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            import torch
            props = torch.cuda.get_device_properties(self.index)
            bus = "%08x:%02x:%02x.0" % (getattr(props, "pci_domain_id", 0), props.pci_bus_id, props.pci_device_id)
            h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        return pynvml, h

    def _poll(self):
        nv, h = self.nvml
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(get_reasons(h))))
            except Exception:
                pass
            self._stop.wait(0.004)

    def sample_now(self):
        """One sample taken by the CALLER (the main thread, right after it has enqueued the timed steps: the GPU is still executing
        them), so the timed region holds a reading under load even when it is shorter than the poll thread's NVML round trips."""
        if self.nvml is None:
            return
        nv, h = self.nvml
        try:
            get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
            self.samples.append((time.perf_counter(), float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(get_reasons(h))))
        except Exception:
            pass

    def start(self):
        try:
            self.nvml = self._nvml_handle()
            nv, h = self.nvml
            self.smax = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if self.nvml is not None:
            self._stop.set()
            self.thread.join(timeout=1)
            rows = [s for s in self.samples if t0 <= s[0] <= t1] or self.samples
            sm = [s[1] for s in rows]
            mask = 0
            for s in rows:
                mask |= s[2]
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.smax,
                    "reasons": sorted(nm for nm, bit in self.REASONS if mask & bit), "samples": len(sm), "source": "nvml, 4 ms poll"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        rows = [l for t, l in self.lines if t0 - 0.05 <= t <= t1 + 0.15] or [l for _, l in self.lines]
        for l in rows:
            parts = [p.strip() for p in l.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                smax.append(float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


DUMP_BYTES = 64 * 10**6


def dump_output(d, y):
    """Write the timed forward's output `y` [N,C,H,W] as <d>/output.npy, float32.  An output larger than DUMP_BYTES keeps its leading
    images that fit (or, when one image does not, the leading rows of the first), so element [n,c,h,w] of the file is element [n,c,h,w]
    of the output and two builds run with the same arguments compare element for element."""
    import numpy as np
    y = y.detach().float()
    cap = (DUMP_BYTES - 4096) // 4     # elements; room for the .npy header
    if y.numel() > cap:
        per_image = y[0].numel()
        y = y[:cap // per_image] if per_image <= cap else y[:1, :, :cap // (y.shape[1] * y.shape[3])]
    y = y.cpu()
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "output.npy"), y.numpy())


ORT_NOTE = "onnxruntime unavailable \u2014 not installed, no network"


def onnxruntime_status():
    """BASELINE.md asks for the reference's ONNX-Runtime-CPU path beside the PyTorch-CPU one; say so when it cannot be timed."""
    try:
        import onnxruntime  # noqa: F401
        return "onnxruntime importable but the reference's best_model.onnx does not travel to the GPU box: not timed"
    except Exception:
        return ORT_NOTE


def cpu_forward_fn():
    """The reference's PyTorch-CPU forward: the UNMODIFIED reference module from oracle/_ref (placed there by oracle/build_ref.py
    in the build container; kind "reference") when present, else the pinned oracle port (kind "port")."""
    import torch
    sd = torch.load(os.path.join(ROOT, "weights", "best_model.pth"))
    try:
        from oracle import build_ref
        mod = build_ref.load("model")
    except Exception:
        mod = None
    if mod is not None:
        net = mod.LightweightUNet()
        net.load_state_dict(sd, strict=True)
        net.eval()
        return (lambda x: net(x)), "reference"
    from oracle import torch_unet as tpo
    return (lambda x: tpo.lightweight_forward(x, sd)), "port"


def cpu_reference_rate(batch, reps, H, W):
    """The reference's PyTorch-CPU path on all host cores; returns (images/s, cores, times, kind)."""
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fwd, kind = cpu_forward_fn()
    x = torch.rand(batch, 1, H, W, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        fwd(x[:1])
        times = []
        t_all = time.perf_counter()
        # bounded sample: at least `reps` forwards and ~10 s of CPU work, at most 30 s
        while len(times) < reps or (time.perf_counter() - t_all < 10.0 and time.perf_counter() - t_all < 30.0):
            t = time.perf_counter()
            fwd(x)
            times.append(time.perf_counter() - t)
            if time.perf_counter() - t_all > 30.0:
                break
    return batch / statistics.median(times), cores, times, kind


def run_reference(args, rank, world):
    if rank != 0:
        return
    batch = args.ref_batch
    if batch <= 0:   # the GPU arm's per-step batch when the whole run stays within a few minutes, else a bounded sample of it
        batch = args.batch if (args.steps + args.warmup) * args.batch <= 4096 else max(1, 4096 // (args.steps + args.warmup))
    t0 = time.perf_counter()
    import torch
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    fwd, kind = cpu_forward_fn()
    x = torch.rand(batch, 1, args.hw, args.hw, generator=torch.Generator().manual_seed(0))
    with torch.no_grad():
        for _ in range(args.warmup):
            fwd(x)
        t = time.perf_counter()
        for _ in range(args.steps):
            y = fwd(x)
        dt = time.perf_counter() - t
    if args.dump_outputs:
        dump_output(args.dump_outputs, y)
    rate = batch * args.steps / dt
    sample = (f"{args.steps} steps x {batch} images of 1x{args.hw}x{args.hw}, fp32, torch CPU {cores} threads"
              + ("" if batch == args.batch else f"; a bounded sample of the GPU arm's batch of {args.batch} (per-image CPU cost is flat in "
                                                "the batch size, measured 8 vs 1)"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": f"best_model.pth LightweightUNet (486,409 params) batched inference, batch {args.batch} x 1x{args.hw}x{args.hw} "
                               "per GPU (BASELINE.json configs[1])",
                   "arm": "reference PyTorch-CPU path, fp32 (" + ("the unmodified reference module, oracle/_ref" if kind == "reference"
                                                                   else "pinned oracle port") + ")",
                   "batch_per_step": batch, "l2": "n/a (CPU)", "onnxruntime_cpu": onnxruntime_status()},
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline forward (the side measurements use their own counts)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--storage", default="fp16", choices=["fp16", "bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--hw", type=int, default=512)
    ap.add_argument("--ref-batch", type=int, default=0, help="images per step of the CPU reference arm (0 = the GPU arm's batch, reduced only if steps x batch would exceed ~4096 images = a few minutes of CPU work)")
    ap.add_argument("--path", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the configs[3] training-step measurement")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[0] latency and configs[4] wide-variant side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the measurements, write what the last timed step computed (rank 0's "
                    "output images, float32) as DIR/output.npy; above 64 MB, the leading images that fit")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist

    import image_enhancement_deglaring_b200 as dg
    from image_enhancement_deglaring_b200 import _lib
    from image_enhancement_deglaring_b200.session import InferenceSession

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa_cpus = None
    if world > 1:   # one process per GPU: keep each rank (and the pinned buffers it allocates) on its GPU's NUMA node
        from image_enhancement_deglaring_b200.parallel import bind_to_gpu_numa_node
        numa_cpus = bind_to_gpu_numa_node(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    H = W = args.hw
    B = args.batch
    sd = torch.load(os.path.join(ROOT, "weights", "best_model.pth"))
    net = dg.LightweightUNet(storage=args.storage, path=args.path)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    x = torch.rand(B, 1, H, W, generator=torch.Generator().manual_seed(rank)).to(dev)

    with torch.no_grad():
        for _ in range(args.warmup):
            y = net(x)
        barrier()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
            if sampler.nvml is None:
                time.sleep(0.25)   # nvidia-smi needs a moment to produce its first line
        barrier()
        l0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(args.steps):
            y = net(x)
        e1.record()
        if rank == 0:
            sampler.sample_now()
        barrier()
        t1 = time.perf_counter()
        launches = _lib.launch_count() - l0
        ms = e0.elapsed_time(e1)
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    value = world * B * args.steps / (ms_max * 1e-3)

    # ---- end to end through the reference-facing session API, host buffers in and out ------------
    # Two flavours, both with every step's H2D copy of its inputs and D2H copy of its result inside the timed region:
    #   blocking  -- InferenceSession.run_pinned per batch (returns when the result is in host memory; chunk 8)
    #   pipelined -- InferenceSession.submit / wait with THREE batches in flight on three pinned buffer pairs, each batch one
    #                chunk: the service shape (several requests outstanding) -- the H2D copy of batch k+2, the forward of batch k+1
    #                and the D2H copy of batch k overlap (tools/e2e_sweep.py: chunk 8..32 or two in flight 27.5-29k img/s, this 31-33k)
    sess = InferenceSession(net, chunk=8)
    e2e_steps = max(6, min(args.steps, 12))
    x2 = torch.flip(x, dims=(0,))
    with torch.no_grad():
        y2 = net(x2)

    def host_pairs(dtype):
        xs = []
        for src in (x, x2, x):
            h = (src * 255).to(torch.uint8).cpu() if dtype == torch.uint8 else src.cpu()
            xs.append((h.pin_memory(), torch.empty((B, 1, H, W), dtype=dtype).pin_memory()))
        return xs

    def rate(step_fn, drain):
        for i in range(3):
            step_fn(i)
        drain()
        barrier()
        te = time.perf_counter()
        for i in range(e2e_steps):
            step_fn(i)
        drain()
        barrier()
        t = torch.tensor([time.perf_counter() - te], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return world * B * e2e_steps / float(t.item())

    def measure(dtype):
        pairs = host_pairs(dtype)
        run = sess.run_pinned_u8 if dtype == torch.uint8 else sess.run_pinned
        blocking = rate(lambda i: run(*pairs[i % 3]), lambda: None)
        pending = []

        def step(i):
            if len(pending) == 3:
                sess.wait(pending.pop(0))
            pending.append(sess.submit(*pairs[i % 3], chunk=B))

        def drain():
            while pending:
                sess.wait(pending.pop(0))

        pipelined = rate(step, drain)
        return blocking, pipelined, pairs

    e2e_blocking, e2e_value, pairs32 = measure(torch.float32)
    e2e_err = max(float((pairs32[0][1].to(dev) - y).abs().max()), float((pairs32[1][1].to(dev) - y2).abs().max()))
    # ---- the same, uint8 images in / uint8 images out (api/app.py:153,190-193 folded into the kernels; SURVEY 8f1)
    e2e_u8_blocking, e2e_u8_value, pairs8 = measure(torch.uint8)
    del pairs32, pairs8

    # ---- BASELINE.json configs[3]: one optimized_train.py step (forward + L1 + backward + clip 1.0 + AdamW), batch 32 per GPU,
    # same storage tier; data parallel = one flat-gradient all-reduce inside FusedAdamW.step.  Reported beside the headline.
    train_step = None
    if not args.no_train:
        from image_enhancement_deglaring_b200.train import FusedAdamW, L1Loss
        tb = 32
        tnet = dg.LightweightUNet(storage=args.storage, path=args.path)
        tnet.load_state_dict(sd, strict=True)
        tnet = tnet.to(dev).train()
        opt = FusedAdamW(tnet.parameters(), lr=0.002362532125818593, weight_decay=6.753784966611083e-05, max_grad_norm=1.0)
        crit = L1Loss()   # drop-in for nn.L1Loss: seed generated inside the head backward, gradients written into the flat bucket
        tx = torch.rand(tb, 1, H, W, generator=torch.Generator().manual_seed(10 + rank)).to(dev)
        tt = torch.rand(tb, 1, H, W, generator=torch.Generator().manual_seed(110 + rank)).to(dev)

        def tstep():
            opt.zero_grad(set_to_none=True)
            loss = crit(tnet(tx), tt)
            loss.backward()
            opt.step()
            return loss

        for _ in range(3):
            tstep()
        barrier()
        tsteps = max(3, min(args.steps, 10))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(tsteps):
            tloss = tstep()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / tsteps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        tbytes = training_algorithmic_bytes_per_image(H, W, 8, 4 if args.storage == "fp32" else 2) * tb
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                tpk = float(json.load(f).get("hbm_gbs", 6650.0))
        except (OSError, ValueError):
            tpk = 6650.0
        train_step = {"value": world * tb / (float(t.item()) * 1e-3), "unit": UNIT, "ms_per_step": float(t.item()), "batch_per_gpu": tb,
                      "roofline": {"bound": "hbm", "scope": "whole step (per GPU)", "algorithmic_bytes_per_step": tbytes,
                                   "achieved": tbytes / (float(t.item()) * 1e-3) / 1e9, "peak": tpk, "unit": "GB/s",
                                   "frac": tbytes / (float(t.item()) * 1e-3) / 1e9 / tpk},
                      "steps": tsteps, "loss": float(tloss.detach()),
                      "what": "forward + L1 + backward + clip_grad_norm 1.0 + AdamW (FusedAdamW), tensor-core forward / dgrad / wgrad "
                              "for 16-bit storage, CUDA events, max over ranks"}
        del tnet, opt, tx, tt
        torch.cuda.empty_cache()
        # the same step captured in ONE CUDA graph (train.GraphedTrainStep: forward, loss, backward, all-reduce, clip, AdamW; step
        # count and learning rate in device memory) at 32 and at 4 images per GPU -- the latter is the reference's own global batch
        # of 32 on 8 GPUs, where the eager step is host-launch bound
        # (single-process runs only: tools/bench_train.py --graph times it under torchrun, where a captured NCCL all-reduce is involved)
        if not args.no_extras and world == 1:
            from image_enhancement_deglaring_b200.train import GraphedTrainStep
            graphed = {}
            for gb in (tb, 4):
                try:
                    gnet = dg.LightweightUNet(storage=args.storage, path=args.path)
                    gnet.load_state_dict(sd, strict=True)
                    gnet = gnet.to(dev).train()
                    gopt = FusedAdamW(gnet.parameters(), lr=0.002362532125818593, weight_decay=6.753784966611083e-05, max_grad_norm=1.0,
                                      capturable=True)
                    gx = torch.rand(gb, 1, H, W, generator=torch.Generator().manual_seed(10 + rank)).to(dev)
                    gt = torch.rand(gb, 1, H, W, generator=torch.Generator().manual_seed(110 + rank)).to(dev)
                    eager_ms = None
                    if gb != tb:      # eager time at this batch for comparison (batch 32 is the line above)
                        def estep():
                            gopt.zero_grad(set_to_none=True)
                            crit(gnet(gx), gt).backward()
                            gopt.step()
                        for _ in range(3):
                            estep()
                        barrier()
                        e0.record()
                        for _ in range(tsteps):
                            estep()
                        e1.record()
                        torch.cuda.synchronize()
                        eager_ms = e0.elapsed_time(e1) / tsteps
                    gstep = GraphedTrainStep(gnet, gopt, crit, gx.shape)
                    for _ in range(3):
                        gstep(gx, gt)
                    barrier()
                    e0.record()
                    for _ in range(tsteps):
                        gloss = gstep(gx, gt)
                    e1.record()
                    torch.cuda.synchronize()
                    tg = torch.tensor([e0.elapsed_time(e1) / tsteps], dtype=torch.float64, device=dev)
                    if world > 1:
                        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
                    graphed[f"batch_{gb}_per_gpu"] = {"ms_per_step": float(tg.item()), "value": world * gb / (float(tg.item()) * 1e-3),
                                                      "unit": UNIT, "eager_ms_per_step": eager_ms, "loss": float(gloss)}
                    del gstep, gnet, gopt, gx, gt
                except Exception as e:   # noqa: BLE001 -- an extra: report instead of losing the line
                    graphed[f"batch_{gb}_per_gpu"] = {"error": repr(e)[:300]}
                torch.cuda.empty_cache()
            train_step["cuda_graph"] = graphed

    # ---- BASELINE.json configs[0]: fp32, batch 1, 1x512x512 -- latency of one image through the module (device-resident input,
    # CUDA events) and through the ORT-shaped session call (host buffers); the CPU batch-1 number is cpu_baseline.batch1_ms
    latency_n1 = None
    if rank == 0 and not args.no_extras:
        latency_n1 = {}
        x1 = torch.rand(1, 1, H, W, generator=torch.Generator().manual_seed(7)).to(dev)
        for storage in ("fp32", args.storage):
            n1 = dg.LightweightUNet(storage=storage, path=args.path)
            n1.load_state_dict(sd, strict=True)
            n1 = n1.to(dev).eval()
            with torch.no_grad():
                for _ in range(5):
                    n1(x1)
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                torch.cuda.synchronize()
                ev[0].record()
                for _ in range(50):
                    n1(x1)
                ev[1].record()
                torch.cuda.synchronize()
                # the same forward captured once and replayed as a CUDA graph (launch overhead off the critical path)
                graph_ms = None
                try:
                    g1, gs = torch.cuda.CUDAGraph(), torch.cuda.Stream()
                    with torch.cuda.stream(gs):
                        with torch.cuda.graph(g1, stream=gs):
                            n1(x1)
                    g1.replay()
                    gev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
                    torch.cuda.synchronize()
                    gev[0].record()
                    for _ in range(50):
                        g1.replay()
                    gev[1].record()
                    torch.cuda.synchronize()
                    graph_ms = gev[0].elapsed_time(gev[1]) / 50
                    del g1
                except RuntimeError as e:   # reported, not hidden
                    graph_ms = f"capture failed: {str(e)[:80]}"
            s1 = InferenceSession(n1, chunk=1)
            xh = x1.cpu().numpy()
            for _ in range(3):
                s1.run(["output"], {"input": xh})
            tl = time.perf_counter()
            for _ in range(20):
                s1.run(["output"], {"input": xh})
            latency_n1[storage] = {"device_ms": ev[0].elapsed_time(ev[1]) / 50, "graph_replay_ms": graph_ms,
                                   "session_run_ms": (time.perf_counter() - tl) / 20 * 1e3}
            del n1, s1
        latency_n1["what"] = ("one 1x1x512x512 image: device_ms = module forward with the input resident in HBM (CUDA events, mean of 50); "
                              "graph_replay_ms = the same forward replayed from a captured CUDA graph; "
                              "session_run_ms = InferenceSession.run from a pageable numpy array and back (api/app.py:171 call shape)")

    # ---- BASELINE.json configs[4]: the wide variant LightweightUNet(features_start=64), 31.0 M parameters, 384.7 GFLOP per
    # 512x512 image: every conv with C_out >= 32 and every ConvTranspose on the tcgen05 kernel (conv3x3_t5.cu)
    wide = None
    if rank == 0 and not args.no_extras:
        torch.manual_seed(42)
        wb = 4
        wnet = dg.LightweightUNet(features_start=64, storage=args.storage, path=args.path).to(dev).eval()
        wx = torch.rand(wb, 1, H, W, generator=torch.Generator().manual_seed(3)).to(dev)
        with torch.no_grad():
            for _ in range(3):
                wnet(wx)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(5):
                wnet(wx)
            ev[1].record()
            torch.cuda.synchronize()
        wms = ev[0].elapsed_time(ev[1]) / 5
        flop = 384.7e9 * (H * W) / (512 * 512)
        peaks_w = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks_w = json.load(f)
        except OSError:
            pass
        tpeak = float(peaks_w.get("bf16_tflops_sustained", 1400.0))
        wide = {"model": "LightweightUNet(features_start=64)", "params": dg.count_parameters(wnet), "batch": wb, "ms_per_step": wms,
                "value": wb / (wms * 1e-3), "unit": UNIT, "tflops": flop * wb / (wms * 1e-3) / 1e12,
                "roofline": {"bound": "tensor", "achieved": flop * wb / (wms * 1e-3) / 1e12, "peak": tpeak, "unit": "TFLOP/s",
                             "frac": flop * wb / (wms * 1e-3) / 1e12 / tpeak,
                             "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks_w else "fallback 1400"},
                "what": "inference forward, random-init weights (no checkpoint exists for this width), CUDA events, mean of 5"}
        # configs[4] asks for "training + inference": one training step of the same width (forward + L1 + backward + clip 1.0 +
        # AdamW), tensor-core backward (wgrad_tc wide instances, tcgen05 data gradient, blocked ConvTranspose weight gradient);
        # 3 x the forward FLOPs per step
        try:
            from image_enhancement_deglaring_b200.train import FusedAdamW, L1Loss
            wnet.train()
            wnet.ddp_sync = False   # a rank-0-only side measurement: no gradient all-reduce (the other ranks are not in this step)
            wopt = FusedAdamW(wnet.parameters(), lr=2.3e-3, weight_decay=6.75e-5, max_grad_norm=1.0)
            wcrit = L1Loss()
            wt = torch.rand(wb, 1, H, W, generator=torch.Generator().manual_seed(6)).to(dev)

            def wstep():
                wopt.zero_grad(set_to_none=True)
                l = wcrit(wnet(wx), wt)
                l.backward()
                wopt.step()
                return l
            for _ in range(3):
                wstep()
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(5):
                wl = wstep()
            ev[1].record()
            torch.cuda.synchronize()
            wtms = ev[0].elapsed_time(ev[1]) / 5
            wide["train_step"] = {"batch": wb, "ms_per_step": wtms, "value": wb / (wtms * 1e-3), "unit": UNIT,
                                  "tflops": 3 * flop * wb / (wtms * 1e-3) / 1e12, "frac": 3 * flop * wb / (wtms * 1e-3) / 1e12 / tpeak,
                                  "loss": float(wl.detach()),
                                  "what": "forward + L1 + backward + clip 1.0 + AdamW (FusedAdamW), tensor-core backward; "
                                          "ConvTranspose data gradient, GroupNorm / activation backward above 128 channels on CUDA cores"}
            del wopt, wt
        except Exception as e:  # a side measurement must never take the headline line down
            wide["train_step"] = {"error": repr(e)[:200]}
        del wnet, wx
        torch.cuda.empty_cache()

    # ---- src/optimized_model.py:OptimizedUNet (north_star's module file; SURVEY 8 a13/a14): inference at batch 16, random-init
    # weights (no checkpoint ships for it), 16.35 GMAC per 512x512 image
    optimized = None
    if rank == 0 and not args.no_extras:
        torch.manual_seed(7)
        ob = 16
        onet = dg.OptimizedUNet(storage=args.storage).to(dev).eval()
        ox = torch.rand(ob, 1, H, W, generator=torch.Generator().manual_seed(4)).to(dev)
        with torch.no_grad():
            for _ in range(3):
                onet(ox)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(5):
                onet(ox)
            ev[1].record()
            torch.cuda.synchronize()
        oms = ev[0].elapsed_time(ev[1]) / 5
        oflop = 2 * 16.35e9 * (H * W) / (512 * 512)
        optimized = {"model": "OptimizedUNet()", "params": dg.count_parameters(onet), "batch": ob, "ms_per_step": oms,
                     "value": ob / (oms * 1e-3), "unit": UNIT, "tflops": oflop * ob / (oms * 1e-3) / 1e12,
                     "what": "inference forward (nearest-up + ChannelAttention variant), random-init weights, CUDA events, mean of 5"}
        # its training step (round 2, SURVEY 8 a13): optimized_train.py:220-233 -- zero_grad, forward, L1, backward, clip 1.0, AdamW --
        # at batch 8; the backward is orchestrated per op above the C-ABI (model_optimized.py), ~190 launches per step
        try:
            from image_enhancement_deglaring_b200.train import FusedAdamW
            tb = 8
            onet.train()
            onet.ddp_sync = False   # rank-0-only side measurement: no gradient all-reduce
            oopt = FusedAdamW(onet.parameters(), lr=2.3e-3, weight_decay=6.75e-5, max_grad_norm=1.0)
            ocrit = torch.nn.L1Loss()
            otx, ott = ox[:tb].contiguous(), torch.rand(tb, 1, H, W, generator=torch.Generator().manual_seed(5)).to(dev)

            def ostep():
                oopt.zero_grad(set_to_none=True)
                l = ocrit(onet(otx), ott)
                l.backward()
                oopt.step()
                return l
            for _ in range(3):
                ostep()
            torch.cuda.synchronize()
            ev[0].record()
            for _ in range(5):
                ol = ostep()
            ev[1].record()
            torch.cuda.synchronize()
            otms = ev[0].elapsed_time(ev[1]) / 5
            optimized["train_step"] = {"batch": tb, "ms_per_step": otms, "value": tb / (otms * 1e-3), "unit": UNIT, "loss": float(ol.detach()),
                                       "what": "forward + L1 + backward (all 76 parameter tensors) + clip 1.0 + AdamW (FusedAdamW); "
                                               "tensor-core wgrad / dgrad where the channel pair is covered, CUDA-core kernels elsewhere"}
            del oopt, otx, ott
        except Exception as e:  # a side measurement must never take the headline line down
            optimized["train_step"] = {"error": repr(e)[:200]}
        del onet, ox
        torch.cuda.empty_cache()

    # ---- per-kernel device times (CUDA events on the launching stream) -> roofline of the dominant kernel
    roofline = None
    if rank == 0:
        ws = torch.empty(net.workspace_bytes(B, H, W), dtype=torch.uint8, device=dev)
        yy = torch.empty_like(y)
        acc = [0.0] * 19
        reps = max(3, min(args.steps, 10))
        buf = (C.c_float * 19)()
        for it in range(reps + 1):
            _lib.check(_lib.load().dg_lw_profile(C.byref(net.c_params()), x.data_ptr(), yy.data_ptr(), B, H, W,
                                                 ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream, buf))
            if it:
                acc = [a + b for a, b in zip(acc, buf)]
        per_kernel_ms = [a / reps for a in acc]
        esize = 4 if args.storage == "fp32" else 2
        abytes = [b * B for b in algorithmic_bytes_per_image(H, W, 8, esize)]
        top = max(range(19), key=lambda i: per_kernel_ms[i])
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                peaks = json.load(f)
        except OSError:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        achieved = abytes[top] / (per_kernel_ms[top] * 1e-3) / 1e9
        # DRAM bytes of the same kernel from one `ncu --set full` capture at this batch size (profiles/ncu_traffic.json)
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
                tr = json.load(f).get(LAYERS[top])
            if tr and B == 64 and H == 512 and args.storage == "fp16":
                traffic = tr["traffic"]
        except (OSError, ValueError):
            pass
        net_bytes = sum(abytes)
        roofline = {
            "bound": "hbm", "kernel": LAYERS[top], "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": traffic,
            "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650 GB/s",
            "kernel_ms": per_kernel_ms[top], "kernel_share_of_step": per_kernel_ms[top] / sum(per_kernel_ms),
            "whole_net": {"algorithmic_bytes_per_step": net_bytes, "achieved": net_bytes / (ms_max / args.steps * 1e-3) / 1e9,
                          "frac": net_bytes / (ms_max / args.steps * 1e-3) / 1e9 / peak},
            "per_kernel": {n: {"ms": round(m, 4), "GBps": round(b / (m * 1e-3) / 1e9, 1)}
                           for n, m, b in zip(LAYERS, per_kernel_ms, abytes)},
        }

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:   # rank 0 at N = 1 only (the other ranks would idle behind it)
        reps = 3
        cb = args.ref_batch if args.ref_batch > 0 else 8   # bounded sample: ~10 s of CPU work at 512x512
        rate, cores, times, kind = cpu_reference_rate(cb, reps, H, W)
        rate1, _, times1, _ = cpu_reference_rate(1, 3, H, W) if H * W <= 512 * 512 else (None, None, [], None)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": kind,
                        "sample": f"median of {len(times)} forwards of {cb} x 1x{H}x{W} fp32 images, torch CPU, "
                                  f"{cores} threads ({sum(times):.1f} s of CPU work)",
                        "batch1_ms": (1e3 / rate1 if rate1 else None),
                        "onnxruntime_cpu": onnxruntime_status()}

    if rank == 0 and args.dump_outputs:
        dump_output(args.dump_outputs, y)
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": args.storage, "data": "synthetic",
            "config": {"workload": f"best_model.pth LightweightUNet (486,409 params) batched inference, batch {B} x 1x{H}x{W} "
                                   f"per GPU, {args.storage} storage / fp32 accumulate (BASELINE.json configs[1])",
                       "batch_per_gpu": B, "global_batch": B * world, "sharding": "images over ranks, no collective",
                       "streams": "dg_lw_forward runs the two halves of the batch concurrently on two library-private streams "
                                  "(default for >= 16 images; DG_BATCH_SPLIT=0 disables); roofline.per_kernel is timed on one stream",
                       "cpu_affinity": (f"rank 0 bound to {len(numa_cpus)} CPUs local to its GPU (NVML)" if numa_cpus else "unbound"),
                       "l2": f"inputs+intermediates per step ({sum(algorithmic_bytes_per_image(H, W)) * B / 2**20:.0f} MiB) exceed the 126 MB L2; no flush"},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * H * W * 4, "d2h_bytes_per_step": B * H * W * 4,
                    "steps": e2e_steps, "api": "InferenceSession.submit / wait -> dg_lw_infer_host_submit / _wait (pinned host buffers, "
                    "three batches in flight, one chunk per batch)", "max_abs_vs_device_path": e2e_err,
                    "blocking": {"value": e2e_blocking, "api": "InferenceSession.run_pinned -> dg_lw_infer_host, one batch at a time"}},
            "e2e_u8": {"value": e2e_u8_value, "unit": UNIT, "h2d_bytes_per_step": B * H * W, "d2h_bytes_per_step": B * H * W,
                       "steps": e2e_steps, "api": "InferenceSession.submit / wait on uint8 buffers -> dg_lw_infer_host_submit (uint8 pixels "
                                                  "in and out, /255 and clip*255 on the GPU as api/app.py:153,190-193 do on the host; "
                                                  "three batches in flight)",
                       "blocking": {"value": e2e_u8_blocking, "api": "InferenceSession.run_pinned_u8 -> dg_lw_infer_host_u8"}},
            "train_step": train_step,
            "latency_n1": latency_n1,
            "wide": wide,
            "optimized": optimized,
            "gpu_launches": launches,
            "roofline": roofline,
            "cpu_baseline": cpu_baseline,
        }))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
