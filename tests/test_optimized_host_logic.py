"""CPU test of OptimizedUNet's host orchestration (which per-op C-ABI call reads which tensor, channel window and order):
`ops.*` is swapped for the torch stand-ins of tests/opt_standins.py -- restatements of the semantics include/deglare.h documents --
and the module's own `_run` / `_backward` / autograd bridge must then reproduce the oracle's forward and all 76 gradients.
The CUDA kernels themselves are tested on the GPU (tests/test_gpu_optimized.py)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import torch_unet as tpo

sys.path.insert(0, os.path.dirname(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import opt_standins  # noqa: E402
from make_golden import det_state_dict  # noqa: E402

dg = pytest.importorskip("image_enhancement_deglaring_b200")


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def _net(golden, monkeypatch):
    from image_enhancement_deglaring_b200 import ops
    opt_standins.install(monkeypatch, ops)
    g = golden("opt_rand.npz")
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    sd = {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=1234).items()}
    net = dg.OptimizedUNet()
    net.load_state_dict(sd, strict=True)
    return net, sd


@pytest.mark.parametrize("shape,seed", [((2, 1, 32, 32), 7), ((1, 1, 16, 48), 11)])
def test_orchestration_reproduces_oracle_gradients(golden, monkeypatch, shape, seed):
    net, sd = _net(golden, monkeypatch)
    x = _rand(shape, seed)
    gy = torch.randn(*shape, generator=torch.Generator().manual_seed(9)) / x.numel()
    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    out = tpo.optimized_forward(x, params)
    ref = dict(zip(params, torch.autograd.grad((out * gy).sum(), list(params.values()))))
    keep = {}
    y = net._run(x, keep)
    assert float((y - out.detach()).abs().max()) <= 1e-4 * max(1.0, float(out.detach().abs().max()))
    flat = torch.zeros(sum(p.numel() for p in net.parameters()))
    net._backward(keep, gy, flat)
    off = 0
    for k, p in net.named_parameters():
        got = flat[off:off + p.numel()].view_as(p)
        off += p.numel()
        r = ref[k]
        assert float((got - r).abs().max()) <= 1e-9 + 2e-4 * float(r.abs().max()), k


def test_autograd_bridge_returns_gradients_in_parameter_order(golden, monkeypatch):
    from image_enhancement_deglaring_b200.train import train_forward
    net, sd = _net(golden, monkeypatch)
    x, t = _rand((1, 1, 32, 32), 3), _rand((1, 1, 32, 32), 4)
    r = tpo.train_step(sd, x, t, forward=tpo.optimized_forward, max_norm=0.0)
    y = train_forward(net, x)
    loss = torch.nn.L1Loss()(y, t)
    loss.backward(retain_graph=True)
    assert abs(float(loss.detach()) - r["loss"]) <= 1e-5 * max(1.0, r["loss"])
    for k, p in net.named_parameters():
        ref = r["grads"][k]
        assert p.grad is not None and p.grad.shape == ref.shape, k
        assert float((p.grad - ref).abs().max()) <= 2e-5 + 1e-3 * float(ref.abs().max()), k
    with pytest.raises(RuntimeError, match="backward through the same forward twice"):
        loss.backward()              # the saved activations were released by the first backward
    with pytest.raises(RuntimeError, match="CUDA"):
        net(x)                       # the public forward still refuses CPU tensors: no CPU fallback in the product


# ---- data parallel (SURVEY 8e): the mean all-reduce of the flat gradient sits at the END of the bridge's backward ------------------
def _opt_ddp_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from image_enhancement_deglaring_b200 import ops
    from image_enhancement_deglaring_b200.train import train_forward
    for name in opt_standins.STANDINS:
        setattr(ops, name, getattr(opt_standins, name))
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "opt_rand.npz"), allow_pickle=False)
    tmpl = {k: tuple(int(v) for v in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    sd = {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=1234).items()}
    net = dg.OptimizedUNet()
    net.load_state_dict(sd, strict=True)
    x, t = _rand((2, 1, 16, 32), 3), _rand((2, 1, 16, 32), 4)
    y = train_forward(net, x[rank:rank + 1])      # one image per rank
    torch.nn.L1Loss()(y, t[rank:rank + 1]).backward()
    flat = torch.cat([p.grad.reshape(-1) for p in net.parameters()])
    gathered = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(gathered, flat)
    assert torch.equal(gathered[0], gathered[1])          # every rank holds the averaged gradient after backward
    if rank == 0:
        torch.save(flat, out)
    dist.destroy_process_group()


def test_bridge_averages_gradients_over_two_ranks(golden, tmp_path):
    out = str(tmp_path / "flat.pt")
    mp.spawn(_opt_ddp_worker, args=(2, 29500 + (os.getpid() % 2000) + 7, out), nprocs=2, join=True)
    got = torch.load(out)
    g = golden("opt_rand.npz")
    tmpl = {k: tuple(int(v) for v in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    sd = {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=1234).items()}
    x, t = _rand((2, 1, 16, 32), 3), _rand((2, 1, 16, 32), 4)
    # equal shards: the mean over ranks of the per-rank mean losses is the global-batch loss of optimized_train.py:223
    r = tpo.train_step(sd, x, t, forward=tpo.optimized_forward, max_norm=0.0)
    want = torch.cat([r["grads"][k].reshape(-1) for k in sd if k in dict(dg.OptimizedUNet().named_parameters())])
    assert got.shape == want.shape
    assert float((got - want).abs().max()) <= 2e-5 + 1e-3 * float(want.abs().max())


def test_data_gradient_fallback_chain(golden, monkeypatch):
    """16-bit tier dispatch of the conv data gradient: mma.sync kernel where it has the channel pair, else the tcgen05 kernel where it
    has a plan, else the generic kernel -- a refusal (rc 3, raised before any launch) is remembered per pair / shape and must not
    change the result.  Stand-ins refuse like the library does and count who served what."""
    from image_enhancement_deglaring_b200 import ops
    from image_enhancement_deglaring_b200.model_optimized import OptimizedUNet
    net, sd = _net(golden, monkeypatch)
    net.storage = "fp16"            # steers the dispatch; the stand-ins round the stored raws to fp16 like the kernels do
    monkeypatch.setattr(ops, "pack_conv3x3_tc", lambda w, dtype, stream=None: w)      # "a packing exists": hand the fp32 taps through
    monkeypatch.setattr(OptimizedUNet, "_tc_dgrad_ok", {})
    monkeypatch.setattr(OptimizedUNet, "_t5_dgrad_ok", {})
    served = {"tc": 0, "t5": 0, "generic": 0, "refused": 0}

    def via_forward_weights(dR, w_packed, cin):     # w_packed [3,3,cin,cout] (forward layout): flip + swap = the dgrad conv
        wflip = w_packed.flip(0, 1).permute(0, 1, 3, 2).contiguous()
        N, H, W, _ = dR.shape
        return opt_standins.conv3x3_dgrad_generic(dR, wflip, cin, N, H, W)

    def tc(dR, w_packed, cin, cout, stream=None):
        if max(cin, cout) > 128:
            served["refused"] += 1
            raise RuntimeError("libdeglare error 3: dgrad: no tensor-core kernel for %d -> %d channels" % (cin, cout))
        served["tc"] += 1
        return via_forward_weights(dR, w_packed, cin)

    def t5(dR, wflip, cin, cout, stream=None):
        if cin < 32:
            served["refused"] += 1
            raise RuntimeError("libdeglare error 3: wide dgrad: no tcgen05 plan for %d -> %d channels" % (cin, cout))
        served["t5"] += 1
        N, H, W, _ = dR.shape
        return opt_standins.conv3x3_dgrad_generic(dR, wflip, cin, N, H, W)

    def generic(dR, wflip, cin, N, H, W, out=None, stream=None):
        served["generic"] += 1
        return opt_standins.conv3x3_dgrad_generic(dR, wflip, cin, N, H, W)

    monkeypatch.setattr(ops, "conv3x3_dgrad", tc)
    monkeypatch.setattr(ops, "conv3x3_dgrad_wide", t5)
    monkeypatch.setattr(ops, "conv3x3_dgrad_generic", generic)
    x = _rand((1, 1, 32, 32), 5)
    gy = torch.randn(1, 1, 32, 32, generator=torch.Generator().manual_seed(9)) / x.numel()
    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    ref = dict(zip(params, torch.autograd.grad((tpo.optimized_forward(x, params) * gy).sum(), list(params.values()))))
    # the same tier with every data gradient on the generic kernel (path = 1): the dispatch must not change the arithmetic
    net.path = 1
    keep = {}
    net._run(x, keep)
    base = torch.zeros(sum(p.numel() for p in net.parameters()))
    net._backward(keep, gy, base)
    assert served == {"tc": 0, "t5": 0, "generic": 21, "refused": 0}, served
    served["generic"] = 0
    net.path = 0
    for rnd in range(2):            # the second pass runs from the remembered refusals: nobody is asked twice
        keep = {}
        net._run(x, keep)
        flat = torch.zeros(sum(p.numel() for p in net.parameters()))
        net._backward(keep, gy, flat)
        assert float((flat - base).abs().max()) <= 1e-6 * float(base.abs().max()), rnd
        off = 0
        for k, p in net.named_parameters():
            got = flat[off:off + p.numel()].view_as(p)
            off += p.numel()
            assert float((got - ref[k]).abs().max()) <= 1e-9 + 3e-2 * float(ref[k].abs().max()), (rnd, k)   # fp16 storage of the raws
        if rnd == 0:
            # 21 convs have a data gradient (all but enc1.0); the 256-channel pairs go to tcgen05, nothing needs the generic kernel
            assert served["tc"] + served["t5"] + served["generic"] == 21 and served["t5"] == 4 and served["generic"] == 0, served
            first = dict(served)
    assert served["refused"] == first["refused"] and served["t5"] == 2 * first["t5"], (first, served)
