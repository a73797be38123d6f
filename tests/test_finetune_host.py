"""CPU test of partially frozen training's host logic: OptimizedUNet's selective `_backward` over the torch stand-ins of
tests/opt_standins.py (only requested gradients, computed from only the calls a request reads), and the gradient sink's and
GraphedTrainStep's rules for an optimizer over the trainable subset.  The kernels themselves run in tests/test_gpu_finetune_graph.py."""
import os
import sys

import pytest
import torch

from oracle import torch_unet as tpo

sys.path.insert(0, os.path.dirname(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import opt_standins  # noqa: E402
from make_golden import det_state_dict  # noqa: E402

dg = pytest.importorskip("image_enhancement_deglaring_b200")


def _head1x1_bwd(src, weight, grad_y, N, H, W, dtype, G, P, dW, dB, stream=None, eps=opt_standins.EPS):
    """dg_head1x1_bwd with the NULL dW / dB the header allows: that gradient is not computed."""
    sW = dW if dW is not None else torch.zeros(weight.shape)
    sB = dB if dB is not None else torch.zeros(weight.shape[0])
    opt_standins.head1x1_bwd(src, weight, grad_y, N, H, W, dtype, G, P, sW, sB)


def _channel_attention_bwd(act_sum, plane, w1, w2, dscale, dw1, dw2, want_add=True, stream=None):
    """dg_channel_attention_bwd with NULL dw1 / dw2 (both or neither) and NULL add; at least one output requested."""
    assert (dw1 is None) == (dw2 is None) and (dw1 is not None or want_add)
    sw1 = dw1 if dw1 is not None else torch.zeros(w1.shape)
    sw2 = dw2 if dw2 is not None else torch.zeros(w2.shape)
    add = opt_standins.channel_attention_bwd(act_sum, plane, w1, w2, dscale, sw1, sw2)
    return add if want_add else None


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def _net(golden, monkeypatch):
    from image_enhancement_deglaring_b200 import ops
    opt_standins.install(monkeypatch, ops)
    monkeypatch.setattr(ops, "head1x1_bwd", _head1x1_bwd)
    monkeypatch.setattr(ops, "channel_attention_bwd", _channel_attention_bwd)
    g = golden("opt_rand.npz")
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    sd = {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=1234).items()}
    net = dg.OptimizedUNet()
    net.load_state_dict(sd, strict=True)
    return net, sd


def _record(monkeypatch, calls):
    """Log every backward op the orchestration issues, with the tensors that say which layer it serves."""
    from image_enhancement_deglaring_b200 import ops
    for name in ("conv3x3_wgrad", "conv3x3_dgrad_generic", "act_bwd", "gn_bwd_apply", "scale_bwd_sum", "channel_attention_bwd",
                 "head1x1_bwd", "grad_gather"):
        def wrap(*a, _f=getattr(ops, name), _n=name, **k):
            calls.append((_n, a, k))
            return _f(*a, **k)
        monkeypatch.setattr(ops, name, wrap)


DECODER = lambda k: not k.startswith(("enc", "bottleneck", "attention"))   # noqa: E731
HEAD = lambda k: k.startswith("output.")                                     # noqa: E731
ATT2 = lambda k: k.startswith("attention2.")                                 # noqa: E731
DEC_CONVS = [f"dec{k}.{i}" for k in (1, 2, 3, 4) for i in (0, 3)] + [f"upconv{k}.1" for k in (1, 2, 3, 4)]
# which conv weight gradients, conv data gradients and attention backward levels a request may run: the units the request
# reads, derived by hand from src/optimized_model.py:118-158 (a data gradient only where a requested tensor lies below the conv)
EXPECT = {
    "decoder": (DEC_CONVS, [c for c in DEC_CONVS if c != "upconv4.1"], []),
    "head": ([], [], []),
    "attention2": ([], ["dec1.3", "dec1.0", "upconv1.1", "dec2.3", "dec2.0"], [2]),
}
SUBSETS = {"decoder": DECODER, "head": HEAD, "attention2": ATT2}


@pytest.mark.parametrize("subset", list(SUBSETS))
def test_selective_backward_computes_only_what_requests_read(golden, monkeypatch, subset):
    net, sd = _net(golden, monkeypatch)
    shape = (2, 1, 32, 32)
    x = _rand(shape, 7)
    gy = torch.randn(*shape, generator=torch.Generator().manual_seed(9)) / x.numel()
    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    ref = dict(zip(params, torch.autograd.grad((tpo.optimized_forward(x, params) * gy).sum(), list(params.values()))))
    names = [k for k, _ in net.named_parameters()]
    want = [k for k in names if SUBSETS[subset](k)]
    keep = {}
    net._run(x, keep)
    sizes = {k: p.numel() for k, p in net.named_parameters()}
    offs, off = {}, 0
    for k in names:
        offs[k] = off
        off += sizes[k]
    flat = torch.full((off,), float("nan"))
    for k in want:
        flat[offs[k]:offs[k] + sizes[k]] = 0.0
    calls = []
    _record(monkeypatch, calls)
    net._backward(keep, gy, flat, want)
    for k in names:
        got = flat[offs[k]:offs[k] + sizes[k]]
        if k in want:
            r = ref[k].reshape(-1)
            assert float((got - r).abs().max()) <= 1e-9 + 2e-4 * float(r.abs().max()), k
        else:
            assert bool(torch.isnan(got).all()), k            # a frozen range is never touched
    # which layer each call served
    at = {offs[k]: k for k in names}
    flips = {v[0].data_ptr(): c for c, v in net._packs_bwd().items()}
    raws = {v["raw"].data_ptr(): c for c, v in keep.items() if isinstance(v, dict) and "raw" in v}
    wgrad = sorted(at[(k["out"].data_ptr() - flat.data_ptr()) // 4][:-len(".weight")] for n, _, k in calls if n == "conv3x3_wgrad")
    dgrad = sorted(flips[a[1].data_ptr()] for n, a, _ in calls if n == "conv3x3_dgrad_generic")
    att = sorted(a[0].shape[1] for n, a, _ in calls if n == "channel_attention_bwd")
    e_wgrad, e_dgrad, e_att = EXPECT[subset]
    assert wgrad == sorted(e_wgrad), wgrad
    assert dgrad == sorted(e_dgrad), dgrad
    assert att == [16 * 2 ** (lvl - 1) for lvl in e_att], att                  # attention{l} squeezes 16 * 2^(l-1) channels
    assert len([n for n, _, _ in calls if n == "scale_bwd_sum"]) == len(e_att)
    # an activation backward runs only for a conv whose output gradient something reads
    acts = {raws[a[0].data_ptr()] for n, a, _ in calls if n == "act_bwd"}
    assert acts == (set(e_dgrad) | set(e_wgrad)) - {"dec1.3"}, sorted(acts)
    # a frozen GroupNorm gets no dgamma / dbeta; the head gets no dW / dB when frozen
    for n, a, kw in calls:
        if n == "gn_bwd_apply":
            gn = raws[a[0].data_ptr()].rsplit(".", 1)
            gn = f"{gn[0]}.{int(gn[1]) + 1}"
            assert (a[11] is not None) == (gn + ".weight" in want) and (a[12] is not None) == (gn + ".bias" in want), gn
        if n == "head1x1_bwd":
            assert (a[9] is not None) == ("output.weight" in want) and (a[10] is not None) == ("output.bias" in want)
        if n == "channel_attention_bwd":
            assert (a[5] is not None) == (subset == "attention2") and kw.get("want_add", True) is False


def test_selective_backward_compact_layout_and_bridge(golden, monkeypatch):
    """`flat` holding only the requested tensors (the optimizer's bucket over the trainable subset) gets the same values as the
    full layout, and the autograd bridge returns gradients only for parameters that require one."""
    from image_enhancement_deglaring_b200.train import train_forward
    net, sd = _net(golden, monkeypatch)
    x = _rand((1, 1, 32, 32), 3)
    gy = torch.randn(1, 1, 32, 32, generator=torch.Generator().manual_seed(4)) / x.numel()
    sizes = {k: p.numel() for k, p in net.named_parameters()}
    want = [k for k in sizes if DECODER(k)]
    keep = {}
    net._run(x, keep)
    full = torch.zeros(sum(sizes.values()))
    net._backward(keep, gy, full, want)
    keep = {}
    net._run(x, keep)
    compact = torch.zeros(sum(sizes[k] for k in want))
    net._backward(keep, gy, compact, want)
    off = {}
    o = 0
    for k in sizes:
        off[k] = o
        o += sizes[k]
    assert torch.equal(compact, torch.cat([full[off[k]:off[k] + sizes[k]] for k in want]))
    with pytest.raises(ValueError):
        net._backward(keep, gy, torch.zeros(7), want)
    for k, p in net.named_parameters():
        p.requires_grad_(DECODER(k))
    y = train_forward(net, x)
    (y * gy).sum().backward()
    for k, p in net.named_parameters():
        if DECODER(k):
            assert torch.allclose(p.grad.reshape(-1), full[off[k]:off[k] + sizes[k]], rtol=1e-6, atol=1e-12), k
        else:
            assert p.grad is None, k


def _bucket(params, order):
    """A fresh FusedAdamW-style flat bucket whose views are the .grads of `order`."""
    from image_enhancement_deglaring_b200.train import _zero_grads
    flat = torch.empty(sum(p.numel() for p in order))
    _zero_grads(flat, order)
    return flat


def test_flat_grad_sink_accepts_the_trainable_subset_only():
    from image_enhancement_deglaring_b200.train import _flat_grad_sink

    def fresh():
        ps = [torch.nn.Parameter(torch.zeros(n)) for n in (3, 5, 2, 4)]
        ps[0].requires_grad_(False)
        ps[2].requires_grad_(False)
        return ps
    ps = fresh()
    flat = _bucket(ps, [ps[1], ps[3]])
    assert _flat_grad_sink(ps) is flat                           # trainable subset, in order, frozen ones absent
    assert _flat_grad_sink(ps, [False, True, False, True]) is flat
    ps = fresh()
    _bucket(ps, [ps[3], ps[1]])
    assert _flat_grad_sink(ps) is None                           # out of parameters() order
    ps = fresh()
    _bucket(ps, [ps[0], ps[1], ps[3]])
    assert _flat_grad_sink(ps) is None                           # covers a frozen tensor
    ps = fresh()
    flat = _bucket(ps, [ps[1], ps[3]])
    ps[2].grad = flat[:2]                                         # a frozen tensor's .grad inside the bucket
    assert _flat_grad_sink(ps) is None
    ps = fresh()
    flat = _bucket(ps, [ps[1], ps[3]])
    flat.add_(1.0)                                                # no longer known to be zero
    assert _flat_grad_sink(ps) is None
    for p in ps:
        p.requires_grad_(True)
    assert _flat_grad_sink(ps) is None                           # every parameter trainable: the bucket misses two
    assert _flat_grad_sink(ps, [True] * 4) is None
    flat = _bucket(ps, ps)
    assert _flat_grad_sink(ps) is flat


def test_graphed_step_requires_the_optimizer_over_exactly_the_trainable_parameters():
    from image_enhancement_deglaring_b200.train import _check_trainable
    net = torch.nn.Sequential(torch.nn.Linear(2, 3), torch.nn.Linear(3, 1))
    ps = list(net.parameters())
    _check_trainable(net, ps)
    net[0].requires_grad_(False)
    _check_trainable(net, ps[2:])
    with pytest.raises(ValueError, match=r"0\.weight \(frozen\)"):
        _check_trainable(net, ps)                                 # an optimizer over a frozen parameter
    with pytest.raises(ValueError, match="1.bias"):
        _check_trainable(net, ps[2:3])                            # missing a trainable one
    with pytest.raises(ValueError, match="position 0"):
        _check_trainable(net, ps[3:] + ps[2:3])                   # out of order
    with pytest.raises(ValueError, match="not a parameter"):
        _check_trainable(net, [torch.nn.Parameter(torch.zeros(1))] + ps[3:])
    net.requires_grad_(False)
    with pytest.raises(ValueError, match="no trainable"):
        _check_trainable(net, [])


def test_gather_index_of_every_request_stays_alive():
    """A captured step gathers with the index it was built with: a later request on the same module must not replace it."""
    from image_enhancement_deglaring_b200.train import _gather_index
    net = torch.nn.Sequential(torch.nn.Linear(2, 3), torch.nn.Linear(3, 1))
    ps = list(net.parameters())
    a = _gather_index(net, ps, [False, True, True, False], torch.device("cpu"))
    assert a.tolist() == list(range(6, 12))
    b = _gather_index(net, ps, [False, False, False, True], torch.device("cpu"))
    assert b.tolist() == [12]
    assert _gather_index(net, ps, [False, True, True, False], torch.device("cpu")) is a
