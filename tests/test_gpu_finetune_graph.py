"""Fine-tuning a partially frozen network on the GPU: GraphedTrainStep over the trainable subset (LightweightUNet through
dg_lw_backward_select, OptimizedUNet through its selective per-op backward), OptimizedUNet's eager selective backward against the
float64 autograd oracle, the work the frozen layers skip, and the relaxed per-op entry points (NULL head / attention outputs)."""
import os
import sys

import pytest
import torch

from oracle import torch_unet as tpo

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import TRAIN_LR, TRAIN_WD, det_state_dict  # noqa: E402

pytestmark = pytest.mark.gpu

dg = pytest.importorskip("image_enhancement_deglaring_b200")
from image_enhancement_deglaring_b200 import _lib, ops  # noqa: E402
from image_enhancement_deglaring_b200.train import FusedAdamW, GraphedTrainStep, L1Loss  # noqa: E402

# Launch counts of the all-trainable steps, recorded on an NVIDIA B200 at the parent commit 72cf362 ("Build each LightweightUNet
# conv's descriptor in one place"): a fully trainable net must keep exactly the launches it had before subsets were supported.
PARENT_LAUNCHES = {
    ("lw", "eager"): 72,
    ("lw", "graphed"): 648,
    ("opt", "eager"): 103,
    ("opt", "graphed"): 532,
}


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def _lw(sd, **kw):
    net = dg.LightweightUNet(**kw)
    net.load_state_dict(sd, strict=True)
    return net.cuda().train()


def _opt_sd(golden):
    g = golden("opt_rand.npz")
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    return {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=1234).items()}


def _opt(sd, **kw):
    net = dg.OptimizedUNet(**kw)
    net.load_state_dict(sd, strict=True)
    return net.cuda().train()


LW_DECODER = lambda k: not k.startswith(("enc", "bottleneck"))                 # noqa: E731
OPT_DECODER = lambda k: not k.startswith(("enc", "bottleneck", "attention"))   # noqa: E731
OPT_ENCODER = lambda k: k.startswith(("enc", "bottleneck"))                    # noqa: E731
OPT_HEAD = lambda k: k.startswith("output.")                                   # noqa: E731
OPT_ATT2 = lambda k: k.startswith("attention2.")                               # noqa: E731


def _freeze(net, trainable):
    for k, p in net.named_parameters():
        p.requires_grad_(trainable(k))
    return net


# ---- 1. LightweightUNet decoder-only: graphed == eager ---------------------------------------------------------------------
@pytest.mark.parametrize("kw", [dict(path=1), dict(storage="fp16")], ids=["fp32", "fp16"])
def test_lightweight_decoder_only_graphed_step_equals_eager_loop(best_sd, kw):
    """test_cuda_graph_training_step_equals_eager_loop with the encoder and bottleneck frozen: the optimizer holds the decoder only,
    the captured step computes only its gradients, and the frozen tensors stay bit-identical to the checkpoint."""
    fp32 = kw.get("path") == 1
    xs = [_rand((4, 1, 64, 96), 70 + i).cuda() for i in range(4)]
    ts = [_rand((4, 1, 64, 96), 80 + i).cuda() for i in range(4)]
    lrs = [TRAIN_LR, TRAIN_LR, TRAIN_LR * 0.5, TRAIN_LR * 0.5]

    def run(graphed):
        net = _freeze(_lw(best_sd, **kw), LW_DECODER)
        opt = FusedAdamW(net.parameters(), lr=TRAIN_LR, weight_decay=TRAIN_WD, max_grad_norm=1.0, capturable=graphed)
        crit = L1Loss()
        if graphed:   # an eager step whose autograd graph is still alive when the capture happens; its effect is undone
            keep_p, keep_m = opt.flat_p.clone(), (opt.exp_avg.clone(), opt.exp_avg_sq.clone())
            opt.zero_grad(set_to_none=True)
            alive = crit(net(xs[3]), ts[3])
            alive.backward()
            opt.step()
            with torch.no_grad():
                opt.flat_p.copy_(keep_p); opt.exp_avg.copy_(keep_m[0]); opt.exp_avg_sq.copy_(keep_m[1]); opt._step_dev.zero_()
        step = GraphedTrainStep(net, opt, crit, xs[0].shape) if graphed else None
        losses = []
        for x, t, lr in zip(xs, ts, lrs):
            opt.param_groups[0]["lr"] = lr
            if graphed:
                losses.append(float(step(x, t)))
            else:
                opt.zero_grad(set_to_none=True)
                loss = crit(net(x), t)
                loss.backward()
                opt.step()
                losses.append(float(loss))
        st = opt.state_dict()
        trainable = {i for i, p in enumerate(opt.param_groups[0]["params"]) if p.requires_grad}
        net.eval()
        with torch.no_grad():
            y = net(xs[0]).cpu()
        return losses, {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}, st, trainable, y

    la, pa, sa, _, ya = run(False)
    lb, pb, sb, trainable, yb = run(True)
    for a, b in zip(la, lb):
        assert abs(a - b) <= 2e-4 * abs(a), (la, lb)
    for k in pa:
        if not LW_DECODER(k):
            assert torch.equal(pa[k], best_sd[k]) and torch.equal(pb[k], best_sd[k]), k
            continue
        d = (pa[k] - pb[k]).abs()
        assert float(d.max()) <= 2 * TRAIN_LR, k
        if fp32:
            assert float((d > 2e-5).float().mean()) <= 2e-3, k
        moved = float((pa[k] - best_sd[k]).norm())
        assert float((pa[k] - pb[k]).norm()) <= (0.02 if fp32 else 0.1) * moved + 1e-6, k
    assert set(sb["state"]) == trainable and len(trainable) == sum(LW_DECODER(k) for k, _ in dg.LightweightUNet().named_parameters())
    assert all(int(float(s["step"])) == 4 for s in sb["state"].values())
    assert int(float(sa["state"][min(sa["state"])]["step"])) == 4
    assert float((ya - yb).abs().max()) <= (2e-3 if fp32 else 5e-3)
    with torch.no_grad():
        y0 = _lw(best_sd, **kw).eval()(xs[0]).cpu()
    assert float((yb - y0).abs().max()) > 10 * float((ya - yb).abs().max()) + 1e-4


# ---- 2. OptimizedUNet decoder-only / head-only: graphed == eager ------------------------------------------------------------
@pytest.mark.parametrize("subset", ["decoder", "head"])
def test_optimized_subset_graphed_step_equals_eager_loop(golden, subset):
    """test_optimized_cuda_graph_training_step_equals_eager_loop over a trainable subset, with its tolerances; frozen tensors stay
    bit-identical."""
    trainable = {"decoder": OPT_DECODER, "head": OPT_HEAD}[subset]
    sd = _opt_sd(golden)
    xs = [_rand((2, 1, 32, 48), 30 + i).cuda() for i in range(3)]
    ts = [_rand((2, 1, 32, 48), 40 + i).cuda() for i in range(3)]
    crit = torch.nn.L1Loss()
    a = _freeze(_opt(sd), trainable)
    oa = FusedAdamW(a.parameters(), lr=TRAIN_LR, weight_decay=TRAIN_WD, max_grad_norm=1.0)
    la = []
    for x, t in zip(xs, ts):
        oa.zero_grad(set_to_none=True)
        loss = crit(a(x), t)
        loss.backward()
        oa.step()
        la.append(float(loss.detach()))
    b = _freeze(_opt(sd), trainable)
    ob = FusedAdamW(b.parameters(), lr=TRAIN_LR, weight_decay=TRAIN_WD, max_grad_norm=1.0, capturable=True)
    step = GraphedTrainStep(b, ob, crit, xs[0].shape)
    lb = [float(step(x, t)) for x, t in zip(xs, ts)]
    for u, v in zip(la, lb):
        assert abs(u - v) <= 2e-5 * max(1.0, abs(u)), (la, lb)
    for (k, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        if not trainable(k):
            assert torch.equal(pa.detach().cpu(), sd[k]) and torch.equal(pb.detach().cpu(), sd[k]), k
            continue
        d = (pa.detach() - pb.detach()).abs()
        assert float(d.max()) <= 2 * TRAIN_LR, k
        moved = float((pa.detach().cpu() - sd[k]).norm())
        assert moved > 0, k
        assert float(d.norm()) <= 0.05 * moved + 1e-6, k
    with torch.no_grad():
        ya, yb = a.eval()(xs[0]).cpu(), b.eval()(xs[0]).cpu()
    assert float((ya - yb).abs().max()) <= 5e-3 * max(1.0, float(ya.abs().max()))


def test_two_graphed_subsets_on_one_net_replay_independently(best_sd):
    """Staged fine-tuning of one LightweightUNet: a graphed step over the decoder convs (A) and one over the head (B) are both
    captured, B after A; A replayed afterwards still walks the eager loop's trajectory (its captured gather index stays alive),
    and replaying B moves the head only."""
    head = lambda k: k.startswith("output_conv")                                   # noqa: E731
    dec = lambda k: LW_DECODER(k) and not head(k)                                   # noqa: E731
    xs = [_rand((4, 1, 64, 96), 90 + i).cuda() for i in range(4)]
    ts = [_rand((4, 1, 64, 96), 95 + i).cuda() for i in range(4)]
    crit = L1Loss()
    ref = _freeze(_lw(best_sd, path=1), dec)
    oref = FusedAdamW(ref.parameters(), lr=TRAIN_LR, weight_decay=TRAIN_WD, max_grad_norm=1.0)
    la = []
    for x, t in zip(xs, ts):
        oref.zero_grad(set_to_none=True)
        loss = crit(ref(x), t)
        loss.backward()
        oref.step()
        la.append(float(loss.detach()))
    net = _lw(best_sd, path=1)
    # both optimizers exist before either capture: each re-points its parameters into its own flat buffer once
    oa = FusedAdamW(_freeze(net, dec).parameters(), lr=TRAIN_LR, weight_decay=TRAIN_WD, max_grad_norm=1.0, capturable=True)
    ob = FusedAdamW(_freeze(net, head).parameters(), lr=TRAIN_LR, weight_decay=TRAIN_WD, max_grad_norm=1.0, capturable=True)
    step_a = GraphedTrainStep(_freeze(net, dec), oa, crit, xs[0].shape)
    step_b = GraphedTrainStep(_freeze(net, head), ob, crit, xs[0].shape)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    lb = [float(step_a(x, t)) for x, t in zip(xs, ts)]
    for u, v in zip(la, lb):
        assert abs(u - v) <= 2e-4 * abs(u), (la, lb)
    pa = {k: v.detach().cpu().clone() for k, v in ref.state_dict().items()}
    pb = {k: v.detach().cpu().clone() for k, v in net.state_dict().items()}
    for k in pa:
        if not dec(k):
            assert torch.equal(pb[k], best_sd[k]), k
            continue
        d = (pa[k] - pb[k]).abs()
        assert float(d.max()) <= 2 * TRAIN_LR, k
        assert float((d > 2e-5).float().mean()) <= 2e-3, k
        assert float(d.norm()) <= 0.02 * float((pa[k] - best_sd[k]).norm()) + 1e-6, k
    float(step_b(xs[0], ts[0]))
    after = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    for k in after:
        assert torch.equal(after[k], pb[k]) != head(k), k


# ---- 3. construction errors ---------------------------------------------------------------------------------------------------
def test_graphed_step_construction_errors(best_sd):
    shape = (2, 1, 32, 32)
    net = _lw(best_sd)
    opt = FusedAdamW(net.parameters(), capturable=True)            # over every parameter ...
    _freeze(net, LW_DECODER)                                         # ... then the encoder is frozen: the optimizer holds frozen ones
    with pytest.raises(ValueError, match="frozen"):
        GraphedTrainStep(net, opt, L1Loss(), shape)
    net = _freeze(_lw(best_sd), LW_DECODER)
    opt = FusedAdamW([p for k, p in net.named_parameters() if LW_DECODER(k) and k != "output_conv.bias"], capturable=True)
    with pytest.raises(ValueError, match="output_conv.bias"):     # missing a trainable one
        GraphedTrainStep(net, opt, L1Loss(), shape)
    net = _lw(best_sd)
    opt = FusedAdamW(net.parameters(), capturable=True)
    net.requires_grad_(False)
    with pytest.raises(ValueError, match="no trainable"):
        GraphedTrainStep(net, opt, L1Loss(), shape)
    net = _freeze(_lw(best_sd), LW_DECODER)
    with pytest.raises(RuntimeError, match="capturable"):
        GraphedTrainStep(net, FusedAdamW(net.parameters()), L1Loss(), shape)


# ---- 4. OptimizedUNet eager selective backward against the oracle -----------------------------------------------------------
@pytest.mark.parametrize("storage", ["fp32", "fp16"])
@pytest.mark.parametrize("subset", ["decoder", "head", "attention2"])
def test_optimized_selective_backward_matches_oracle(golden, storage, subset):
    """Requested gradients within test_optimized_backward_matches_oracle_fp32's per-tensor bound (fp32) or rel-L2 1.5e-2 (fp16
    storage); frozen tensors get no .grad."""
    trainable = {"decoder": OPT_DECODER, "head": OPT_HEAD, "attention2": OPT_ATT2}[subset]
    sd = _opt_sd(golden)
    shape = (2, 1, 64, 64)
    x = _rand(shape, 7)
    gy = torch.randn(*shape, generator=torch.Generator().manual_seed(9)) / x.numel()
    params = {k: v.detach().double().clone().requires_grad_(True) for k, v in sd.items()}
    ref = dict(zip(params, torch.autograd.grad((tpo.optimized_forward(x.double(), params) * gy.double()).sum(),
                                               list(params.values()))))
    net = _freeze(_opt(sd, storage=storage), trainable)
    net(x.cuda()).backward(gy.cuda())
    num = den = 0.0
    for k, p in net.named_parameters():
        if not trainable(k):
            assert p.grad is None, k
            continue
        g, r = p.grad.cpu().double(), ref[k]
        if storage == "fp32":
            assert float((g - r).abs().max()) <= 1e-10 + 3e-4 * float(r.abs().max()), k
        num += float(((g - r) ** 2).sum())
        den += float((r ** 2).sum())
    assert den > 0
    if storage == "fp16":
        assert (num / den) ** 0.5 <= 1.5e-2, (num / den) ** 0.5


# ---- 5. the skipping is real ------------------------------------------------------------------------------------------------------
def _backward_launches(net, x, gy):
    y = net(x)
    n0 = _lib.launch_count()
    y.backward(gy)
    return _lib.launch_count() - n0


def test_launches_follow_the_request(best_sd, golden):
    x, gy = _rand((2, 1, 64, 64), 5).cuda(), (torch.randn(2, 1, 64, 64, generator=torch.Generator().manual_seed(6)) / 8192).cuda()
    osd = _opt_sd(golden)
    for make, dec, head in ((lambda: _lw(best_sd, storage="fp16"), LW_DECODER, lambda k: k.startswith("output_conv")),
                            (lambda: _opt(osd, storage="fp16"), OPT_DECODER, OPT_HEAD)):
        counts = [_backward_launches(_freeze(make(), sel), x, gy) for sel in (lambda k: True, dec, head)]
        assert counts[0] > counts[1] > counts[2] >= 1, counts


def _kernels(net, x, gy):
    y = net(x)
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        y.backward(gy)
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_optimized_decoder_only_backward_runs_no_encoder_or_attention_kernel(golden):
    """Profiled decoder-only backward (fp16 tier: weight gradients on the named tensor-core kernels): no attention backward
    (se_bwd, scale_bwd_sum), and its weight-gradient kernels are exactly the full backward's minus an encoder-only backward's."""
    sd = _opt_sd(golden)
    x, gy = _rand((2, 1, 64, 64), 5).cuda(), (torch.randn(2, 1, 64, 64, generator=torch.Generator().manual_seed(6)) / 8192).cuda()
    runs = {name: _kernels(_freeze(_opt(sd, storage="fp16"), sel), x, gy)
            for name, sel in (("full", lambda k: True), ("decoder", OPT_DECODER), ("encoder", OPT_ENCODER))}
    dec = runs["decoder"]
    assert not [n for n in dec if "se_bwd" in n or "scale_bwd_sum" in n], sorted(set(dec))
    assert any("se_bwd" in n for n in runs["full"]) and any("scale_bwd_sum" in n for n in runs["full"])

    def wgrads(names):
        return sorted(n for n in names if "wgrad" in n)
    assert len(wgrads(runs["full"])) >= 12 and wgrads(dec)
    assert sorted(wgrads(dec) + wgrads(runs["encoder"])) == wgrads(runs["full"])


def _graph_launches(net, opt, crit, shape):
    n0 = _lib.launch_count()
    GraphedTrainStep(net, opt, crit, shape)      # 3 warm-up steps and the captured one
    return _lib.launch_count() - n0


def launch_counts(best_sd, osd):
    """Eager backward and GraphedTrainStep construction launches of fully trainable nets (the shapes of the graphed-step tests)."""
    x, gy = _rand((4, 1, 64, 96), 1).cuda(), (torch.randn(4, 1, 64, 96, generator=torch.Generator().manual_seed(2)) / 24576).cuda()
    xo, gyo = x[:2, :, :32, :48].contiguous(), gy[:2, :, :32, :48].contiguous()
    out = {("lw", "eager"): _backward_launches(_lw(best_sd, storage="fp16"), x, gy),
           ("opt", "eager"): _backward_launches(_opt(osd), xo, gyo)}
    net = _lw(best_sd, storage="fp16")
    out[("lw", "graphed")] = _graph_launches(net, FusedAdamW(net.parameters(), lr=TRAIN_LR, max_grad_norm=1.0, capturable=True),
                                             L1Loss(), x.shape)
    net = _opt(osd)
    out[("opt", "graphed")] = _graph_launches(net, FusedAdamW(net.parameters(), lr=TRAIN_LR, max_grad_norm=1.0, capturable=True),
                                              torch.nn.L1Loss(), xo.shape)
    return out


def test_all_trainable_launches_unchanged(best_sd, golden):
    got = launch_counts(best_sd, _opt_sd(golden))
    assert got == PARENT_LAUNCHES, (got, PARENT_LAUNCHES)


# ---- 6. relaxed per-op entry points -----------------------------------------------------------------------------------------
def test_relaxed_entry_points_match_the_full_call_bit_for_bit():
    gen = torch.Generator().manual_seed(3)
    N, H, W, C, groups = 2, 32, 32, 16, 4
    raw = torch.randn(N, H, W, C, generator=gen).cuda()
    stats = torch.stack((raw.double().sum(dim=(1, 2)), (raw.double() ** 2).sum(dim=(1, 2))), dim=-1).contiguous()
    gamma = (1 + 0.2 * torch.randn(C, generator=gen)).cuda()
    beta = (0.2 * torch.randn(C, generator=gen)).cuda()
    w = torch.randn(1, C, generator=gen).cuda()
    gy = torch.randn(N, 1, H, W, generator=gen).cuda()
    src = ops.make_src(raw, C, stats=stats, gamma=gamma, beta=beta, groups=groups)

    def head(dW, dB):
        G = torch.empty(N, H, W, C, device="cuda")
        P = torch.zeros(N, C, 2, dtype=torch.float64, device="cuda")
        ops.head1x1_bwd(src, w, gy, N, H, W, ops.DG_F32, G, P, dW, dB)
        return G, P
    G0, P0 = head(torch.zeros(1, C, device="cuda"), torch.zeros(1, device="cuda"))
    G1, P1 = head(None, None)
    assert torch.equal(G0, G1) and torch.equal(P0, P1)

    hid = 8
    act_sum = torch.rand(N, C, generator=gen, dtype=torch.float64).cuda() * (H * W)
    w1, w2 = torch.randn(hid, C, generator=gen).cuda(), torch.randn(C, hid, generator=gen).cuda()
    dscale = torch.randn(N, C, generator=gen, dtype=torch.float64).cuda()
    dw1, dw2 = torch.zeros(hid, C, device="cuda"), torch.zeros(C, hid, device="cuda")
    add = ops.channel_attention_bwd(act_sum, float(H * W), w1, w2, dscale, dw1, dw2)
    assert torch.equal(ops.channel_attention_bwd(act_sum, float(H * W), w1, w2, dscale, None, None), add)
    ew1, ew2 = torch.zeros_like(dw1), torch.zeros_like(dw2)
    assert ops.channel_attention_bwd(act_sum, float(H * W), w1, w2, dscale, ew1, ew2, want_add=False) is None
    assert torch.allclose(ew1, dw1, rtol=1e-6, atol=0) and torch.allclose(ew2, dw2, rtol=1e-6, atol=0)   # atomics order only
    with pytest.raises(RuntimeError):
        ops.channel_attention_bwd(act_sum, float(H * W), w1, w2, dscale, dw1, None)
    with pytest.raises(RuntimeError):
        ops.channel_attention_bwd(act_sum, float(H * W), w1, w2, dscale, None, None, want_add=False)
