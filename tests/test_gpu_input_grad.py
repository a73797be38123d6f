"""Input-image gradients and frozen-parameter training through LightweightUNet's native backward (dg_lw_backward_select): dL/dx
against the autograd oracle, only the requested parameter gradients, and a backward that skips frozen work and stops below the
lowest request.  Oracles: oracle/torch_unet.py under CPU autograd in float64."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import torch_unet as tpo

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import det_state_dict  # noqa: E402

pytestmark = pytest.mark.gpu

dg = pytest.importorskip("image_enhancement_deglaring_b200")
from image_enhancement_deglaring_b200 import _lib  # noqa: E402


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def _gy(shape, seed):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) / float(np.prod(shape))


def _net(sd, **kw):
    net = dg.LightweightUNet(**kw)
    net.load_state_dict(sd, strict=True)
    return net.cuda().train()


def _det_sd(seed, **kw):
    tmpl = {k: tuple(v.shape) for k, v in dg.LightweightUNet(**kw).state_dict().items()}
    return {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=seed).items()}


def _oracle_dx(sd, x, gy, params=False):
    """dL/dx (and, with params, every parameter gradient) of sum(forward(x) * gy), float64 CPU autograd."""
    xd = x.double().requires_grad_(True)
    p = {k: v.double().requires_grad_(params) for k, v in sd.items()}
    out = tpo.lightweight_forward(xd, p)
    keys = list(p) if params else []
    g = torch.autograd.grad((out * gy.double()).sum(), [xd] + [p[k] for k in keys])
    return g[0], dict(zip(keys, g[1:]))


def _rel(a, ref):
    return float((a.double().cpu() - ref.double().cpu()).norm() / ref.double().norm())


def _maxrel(a, ref):
    return float((a.double().cpu() - ref.double().cpu()).abs().max() / ref.double().abs().max())


# (name, constructor arguments, shape, metric, bound); the values measured on one B200 are in the test's docstring
CASES = [
    ("fp32-path1-64", dict(path=1), (2, 1, 64, 64), "maxrel", 2e-4),
    ("fp32-path1-48x80", dict(path=1), (3, 1, 48, 80), "maxrel", 2e-4),
    ("fp32-in3-out2-fs12", dict(in_channels=3, out_channels=2, features_start=12), (2, 3, 64, 64), "maxrel", 2e-4),
    ("fp16", dict(storage="fp16"), (2, 1, 128, 160), "rel", 2e-2),
    ("bf16", dict(storage="bf16"), (2, 1, 128, 160), "rel", 8e-2),
    ("fs64-fp16", dict(features_start=64, storage="fp16"), (1, 1, 48, 160), "rel", 2e-2),
]


@pytest.mark.parametrize("name,kw,shape,metric,bound", CASES, ids=[c[0] for c in CASES])
def test_input_gradient_matches_oracle(best_sd, name, kw, shape, metric, bound):
    """x.grad for an explicit random dL/dy against float64 autograd of the oracle, the parameters trainable as well.  Bounds are
    the per-tensor bounds of the parameter-gradient tests: fp32 tiers max-abs <= 2e-4 max|ref|, fp16 storage relative L2 <= 2e-2,
    bf16 storage <= 8e-2.  Measured on one NVIDIA B200 (1000 W): fp32 5.9e-7 / 8.1e-7 / 3.8e-6 (in=3, fs=12), fp16 8.7e-3,
    bf16 1.6e-2, fs=64 fp16 6.2e-3 -- every bound holds with margin, none had to move."""
    shipped = kw.get("features_start", 8) == 8 and kw.get("in_channels", 1) == 1 and kw.get("out_channels", 1) == 1
    sd = best_sd if shipped else _det_sd(7, **{k: v for k, v in kw.items() if k in ("in_channels", "out_channels", "features_start")})
    net = _net(sd, **kw)
    x = _rand(shape, 11)
    gy = _gy((shape[0], net.out_channels) + shape[2:], 12)
    xc = x.cuda().requires_grad_(True)
    net(xc).backward(gy.cuda())
    ref, _ = _oracle_dx(sd, x, gy)
    assert xc.grad is not None and xc.grad.shape == x.shape and xc.grad.dtype == torch.float32
    err = _maxrel(xc.grad, ref) if metric == "maxrel" else _rel(xc.grad, ref)
    print(f"{name}: dx {metric} err {err:.3e} (bound {bound})")
    assert err <= bound, (name, err)
    assert all(p.grad is not None for p in net.parameters())


@pytest.mark.parametrize("fused", [False, True])
def test_mixed_request_golden_step(best_sd, golden, fused):
    """x and every parameter require a gradient: the golden training step's parameter gradients keep the bounds of
    test_gradients_match_golden_step, and x.grad matches the oracle, with nn.L1Loss and with the fused dg.L1Loss."""
    g = golden("lw_train.npz")
    net = _net(best_sd, path=1)
    x, t = _rand((2, 1, 64, 64), 0), _rand((2, 1, 64, 64), 1)
    xc = x.cuda().requires_grad_(True)
    crit = dg.L1Loss() if fused else torch.nn.L1Loss()
    loss = crit(net(xc), t.cuda())
    loss.backward()
    assert abs(float(loss) - float(g["loss"])) <= 1e-5
    for k, p in net.named_parameters():
        ref = g["grad/" + k]
        err = float(np.abs(p.grad.cpu().numpy() - ref).max())
        assert err <= 2e-5 + 2e-4 * float(np.abs(ref).max()), (k, err)
    xd = x.double().requires_grad_(True)
    out = tpo.lightweight_forward(xd, {k: v.double() for k, v in best_sd.items()})
    (out - t.double()).abs().mean().backward()
    assert _maxrel(xc.grad, xd.grad) <= 2e-4


@pytest.mark.parametrize("storage,bound", [("fp32", 1e-6), ("fp16", 1e-3)])
def test_frozen_network_input_gradient(best_sd, storage, bound, monkeypatch):
    """net.requires_grad_(False): no parameter gets a .grad, no data-parallel all-reduce runs, and x.grad equals the mixed
    request's x.grad (fp32: the statistics sums use atomics, so up to summation order; fp16: without the weight gradient the bf16
    dR copy may be chosen for more layers).  A trainable conv in front of the frozen net gets the oracle pipeline's gradient."""
    from image_enhancement_deglaring_b200 import train as train_mod
    kw = dict(path=1) if storage == "fp32" else dict(storage=storage)
    x = _rand((2, 1, 64, 64), 3)
    gy = _gy((2, 1, 64, 64), 4).cuda()
    mixed = _net(best_sd, **kw)
    xm = x.cuda().requires_grad_(True)
    mixed(xm).backward(gy)

    def no_sync(*a, **k):
        raise AssertionError("sync_gradients called for a frozen network")
    monkeypatch.setattr(train_mod, "sync_gradients", no_sync)
    net = _net(best_sd, **kw).requires_grad_(False)
    xf = x.cuda().requires_grad_(True)
    net(xf).backward(gy)
    assert all(p.grad is None for p in net.parameters())
    assert _rel(xf.grad, xm.grad) <= bound
    # trainable pre-processing in front of the frozen de-glarer.  Its conv is torch's own (cuDNN), which by default runs fp32
    # convolutions in TF32 (10-bit mantissa); switched off so that the fp32 bound measures the native backward, not cuDNN
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", False)
    pre = torch.nn.Conv2d(1, 1, 3, padding=1)
    with torch.no_grad():
        pre.weight.copy_(torch.tensor([[[[0.05, 0.1, 0.05], [0.1, 0.4, 0.1], [0.05, 0.1, 0.05]]]]))
        pre.bias.fill_(0.02)
    pre_c = torch.nn.Conv2d(1, 1, 3, padding=1).cuda()
    pre_c.load_state_dict(pre.state_dict())
    net(pre_c(x.cuda())).backward(gy)
    assert all(p.grad is None for p in net.parameters())
    w = pre.weight.detach().double().requires_grad_(True)
    b = pre.bias.detach().double().requires_grad_(True)
    out = tpo.lightweight_forward(F.conv2d(x.double(), w, b, padding=1), {k: v.double() for k, v in best_sd.items()})
    (out * gy.cpu().double()).sum().backward()
    tol = 2e-4 if storage == "fp32" else 2e-2
    assert _rel(pre_c.weight.grad, w.grad) <= tol and _rel(pre_c.bias.grad, b.grad) <= tol


def _decoder_only(net):
    for name, p in net.named_parameters():
        p.requires_grad_(not name.startswith(("enc", "bottleneck")))


def _head_only(net):
    for name, p in net.named_parameters():
        p.requires_grad_(name.startswith("output_conv"))


def _backward_launches(net, x, gy):
    y = net(x)
    n0 = _lib.launch_count()
    y.backward(gy)
    return _lib.launch_count() - n0


@pytest.mark.parametrize("storage", ["fp32", "fp16"])
def test_truncation_and_skipping_are_real(best_sd, storage):
    """Fewer kernels for fewer gradients: full > decoder-only > head-only; the frozen-network backward runs no weight-gradient
    kernel at all (torch.profiler); decoder-only gradients match the oracle and frozen tensors get no .grad."""
    kw = dict(path=1) if storage == "fp32" else dict(storage=storage)
    x = _rand((2, 1, 64, 64), 5)
    gy = _gy((2, 1, 64, 64), 6)
    counts = []
    for setup in (lambda n: None, _decoder_only, _head_only):
        net = _net(best_sd, **kw)
        setup(net)
        counts.append(_backward_launches(net, x.cuda(), gy.cuda()))
    assert counts[0] > counts[1] > counts[2] >= 1, counts

    net = _net(best_sd, **kw)
    _decoder_only(net)
    net(x.cuda()).backward(gy.cuda())
    _, ref = _oracle_dx(best_sd, x, gy, params=True)
    for k, p in net.named_parameters():
        if k.startswith(("enc", "bottleneck")):
            assert p.grad is None, k
        elif storage == "fp32":
            assert float((p.grad.cpu().double() - ref[k]).abs().max()) <= 2e-5 + 2e-4 * float(ref[k].abs().max()), k
        else:
            assert float((p.grad.cpu().double() - ref[k]).norm()) <= 2e-2 * float(ref[k].norm()) + 1e-7, k

    frozen = _net(best_sd, **kw).requires_grad_(False)
    xc = x.cuda().requires_grad_(True)
    y = frozen(xc)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        y.backward(gy.cuda())
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("first_dgrad" in n for n in names), sorted(set(names))
    assert not [n for n in names if "wgrad" in n], sorted(set(names))


def _direct_backward(net, x, gy, select_mask=None):
    """dg_lw_forward, then dg_lw_backward (select_mask None) or dg_lw_backward_select with that mask and no grad_x; returns the
    flat gradient and the backward's launch count."""
    lib = _lib.load()
    N, _, H, W = x.shape
    stream = torch.cuda.current_stream().cuda_stream
    pc = net._refresh(train=True)
    ws = torch.empty(net.workspace_bytes(N, H, W), dtype=torch.uint8, device="cuda")
    y = torch.empty_like(gy)
    _lib.check(lib.dg_lw_forward(C.byref(pc), x.data_ptr(), y.data_ptr(), N, H, W, ws.data_ptr(), ws.numel(), None, None, stream))
    nb, cnt = C.c_size_t(0), C.c_size_t(0)
    _lib.check(lib.dg_lw_backward_workspace_bytes(C.byref(pc), N, H, W, C.byref(nb)))
    _lib.check(lib.dg_lw_num_params(C.byref(pc), C.byref(cnt)))
    bws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    flat = torch.full((cnt.value,), float("nan"), device="cuda")
    n0 = _lib.launch_count()
    if select_mask is None:
        _lib.check(lib.dg_lw_backward(C.byref(pc), x.data_ptr(), gy.data_ptr(), N, H, W, ws.data_ptr(), ws.numel(), bws.data_ptr(),
                                      bws.numel(), flat.data_ptr(), stream))
    else:
        req = _lib.DgLwBwdRequest()
        req.grad_y, req.grads, req.param_mask = gy.data_ptr(), flat.data_ptr(), select_mask
        _lib.check(lib.dg_lw_backward_select(C.byref(pc), x.data_ptr(), C.byref(req), N, H, W, ws.data_ptr(), ws.numel(),
                                             bws.data_ptr(), bws.numel(), stream))
    launches = _lib.launch_count() - n0
    torch.cuda.synchronize()
    return flat, launches


@pytest.mark.parametrize("storage", ["fp32", "fp16"])
def test_select_full_mask_launches_like_dg_lw_backward(best_sd, storage):
    """Every bit set and no grad_x: the new entry point launches exactly what dg_lw_backward launches and writes the same flat
    gradient (up to atomics order).  A partial mask writes its tensors and leaves every other element untouched."""
    net = _net(best_sd, storage=storage)
    x, gy = _rand((2, 1, 64, 64), 8).cuda(), _gy((2, 1, 64, 64), 9).cuda()
    ref, n_ref = _direct_backward(net, x, gy)
    got, n_got = _direct_backward(net, x, gy, (1 << 64) - 1)
    assert n_got == n_ref, (n_got, n_ref)
    assert bool(torch.isfinite(ref).all())
    assert float((got - ref).norm()) <= 1e-5 * float(ref.norm())
    sizes = [p.numel() for p in net.parameters()]
    offs = np.cumsum([0] + sizes)
    names = [k for k, _ in net.named_parameters()]
    mask = sum(1 << names.index(k) for k in ("dec1.0.weight", "dec1.1.weight", "dec1.1.bias", "output_conv.bias"))
    part, n_part = _direct_backward(net, x, gy, mask)
    assert n_part < n_ref
    for k in range(64):
        s = part[offs[k]:offs[k + 1]]
        if (mask >> k) & 1:
            assert float((s - ref[offs[k]:offs[k + 1]]).norm()) <= 2e-2 * float(ref[offs[k]:offs[k + 1]].norm()) + 1e-7, k
        else:
            assert bool(torch.isnan(s).all()), k


def test_two_stream_split_input_gradient(best_sd):
    """Batch 16 takes the two-stream split by default: x.grad equals the single-stream x.grad up to summation order."""
    lib = _lib.load()
    x, gy = _rand((16, 1, 64, 64), 13).cuda(), _gy((16, 1, 64, 64), 14).cuda()
    res = []
    old = lib.dg_set_batch_split(0)
    try:
        for split in (0, old):
            lib.dg_set_batch_split(split)
            net = _net(best_sd, storage="fp16")
            xc = x.clone().requires_grad_(True)
            net(xc).backward(gy)
            res.append(xc.grad.clone())
    finally:
        lib.dg_set_batch_split(old)
    assert old == 16
    assert _rel(res[1], res[0]) <= 1e-6


@pytest.mark.parametrize("cin", [1, 3])
@pytest.mark.parametrize("cout", [8, 12, 16, 64])
def test_first_conv_dgrad_kernel(cin, cout):
    """dg_conv_first_dgrad alone against float64 autograd of F.conv2d (padding 1), W and H not multiples of any tile size."""
    N, H, W = 2, 20, 70
    g = torch.Generator().manual_seed(cin * 100 + cout)
    w = torch.randn(cout, cin, 3, 3, generator=g) / (3 * cin ** 0.5)
    dR = torch.randn(N, cout, H, W, generator=g)
    xd = torch.zeros(N, cin, H, W, dtype=torch.float64, requires_grad=True)
    F.conv2d(xd, w.double(), padding=1).backward(dR.double())
    dR_nhwc = dR.permute(0, 2, 3, 1).contiguous().cuda()
    w_packed = w.permute(2, 3, 1, 0).contiguous().cuda()     # [3][3][cin][cout]
    dx = torch.full((N, cin, H, W), float("nan"), device="cuda")
    _lib.check(_lib.load().dg_conv_first_dgrad(dR_nhwc.data_ptr(), w_packed.data_ptr(), dx.data_ptr(), N, H, W, cin, cout,
                                               torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert _maxrel(dx, xd.grad) <= 1e-5
