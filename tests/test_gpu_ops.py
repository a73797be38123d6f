"""GPU parity of each fused op (through the C-ABI) against the oracle's decomposition."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import torch_unet as tpo

pytestmark = pytest.mark.gpu

ops = pytest.importorskip("image_enhancement_deglaring_b200.ops")

TOL = {ops.DG_F32: 2e-5, ops.DG_F16: 2e-3, ops.DG_BF16: 1.6e-2}   # relative to max|ref|
DTYPES = [ops.DG_F32, ops.DG_F16, ops.DG_BF16]


def _rs(seed):
    return np.random.RandomState(seed)


def _nhwc(t, dtype):
    """NCHW fp32 CPU -> NHWC storage-dtype CUDA, and the value the kernel will actually see (NCHW fp32 CPU)."""
    q = t.permute(0, 2, 3, 1).contiguous().to(ops.TORCH_DTYPE[dtype]).cuda()
    seen = q.float().cpu().permute(0, 3, 1, 2).contiguous()
    return q, seen


def _stats(seen):
    s = torch.stack((seen.double().sum(dim=(2, 3)), (seen.double() ** 2).sum(dim=(2, 3))), dim=2)
    return s.cuda().contiguous()


def _gn_params(rs, c):
    return (torch.from_numpy((1 + 0.3 * rs.standard_normal(c)).astype(np.float32)),
            torch.from_numpy((0.3 * rs.standard_normal(c)).astype(np.float32)))


def _check(out_nhwc, stats, ref, dtype, what):
    got = out_nhwc.float().cpu().permute(0, 3, 1, 2)
    scale = max(1.0, float(ref.abs().max()))
    err = float((got - ref).abs().max())
    assert err <= TOL[dtype] * scale, f"{what}: max err {err:.3e} (scale {scale:.2f})"
    # statistics are those of the STORED (rounded) values
    want = torch.stack((got.double().sum(dim=(2, 3)), (got.double() ** 2).sum(dim=(2, 3))), dim=2)
    serr = float((stats.cpu() - want).abs().max() / max(1.0, float(want.abs().max())))
    assert serr <= 1e-5, f"{what}: stats rel err {serr:.3e}"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cin,cout,H,W", [(1, 8, 32, 64), (3, 12, 16, 48), (1, 16, 48, 40)])
def test_conv_image_source(dtype, cin, cout, H, W):
    rs = _rs(1)
    N = 2
    x = torch.from_numpy(rs.rand(N, cin, H, W).astype(np.float32))
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * 0.4).astype(np.float32))
    src = ops.make_src(x.cuda(), cin, xform=ops.DG_X_IMAGE, silu=False)
    out, st = ops.conv3x3_fused([src], ops.pack_conv3x3(w.cuda()), cout, N, H, W, dtype, path=1)
    torch.cuda.synchronize()
    _check(out, st, F.conv2d(x, w, None, 1, 1), dtype, "image conv")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cin,cout,groups,H,W", [(8, 8, 8, 64, 64), (16, 16, 8, 32, 96), (32, 32, 8, 16, 16),
                                                   (64, 64, 8, 8, 32), (128, 128, 8, 4, 4), (12, 12, 6, 16, 32),
                                                   (16, 16, 1, 16, 16), (8, 8, 8, 40, 33)])
def test_conv_same_gn_silu(dtype, cin, cout, groups, H, W):
    rs = _rs(2)
    N = 2
    raw = torch.from_numpy((rs.standard_normal((N, cin, H, W)) * 3 + 1).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * (1.0 / np.sqrt(9 * cin))).astype(np.float32))
    src = ops.make_src(q, cin, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=groups)
    out, st = ops.conv3x3_fused([src], ops.pack_conv3x3(w.cuda()), cout, N, H, W, dtype, path=1)
    torch.cuda.synchronize()
    ref = F.conv2d(tpo.gn_silu(seen, groups, g, b), w, None, 1, 1)
    _check(out, st, ref, dtype, "same conv")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("cin,cout,H,W", [(8, 16, 32, 32), (64, 128, 4, 8), (12, 24, 8, 24)])
def test_conv_pool_source(dtype, cin, cout, H, W):
    rs = _rs(3)
    N = 2
    groups = 4
    raw = torch.from_numpy((rs.standard_normal((N, cin, 2 * H, 2 * W)) * 2 - 0.5).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * (1.0 / np.sqrt(9 * cin))).astype(np.float32))
    src = ops.make_src(q, cin, xform=ops.DG_X_POOL2, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=groups)
    act_sum = torch.zeros((N, cin), dtype=torch.float64, device="cuda")
    out, st = ops.conv3x3_fused([src], ops.pack_conv3x3(w.cuda()), cout, N, H, W, dtype, act_sum=act_sum, path=1)
    torch.cuda.synchronize()
    act = tpo.gn_silu(seen, groups, g, b)
    _check(out, st, F.conv2d(F.avg_pool2d(act, 2, 2), w, None, 1, 1), dtype, "pool conv")
    want = act.double().sum(dim=(2, 3))
    assert float((act_sum.cpu() - want).abs().max()) <= 1e-4 * max(1.0, float(want.abs().max()))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("c,H,W", [(8, 64, 64), (16, 32, 32), (64, 8, 8), (12, 16, 32), (160, 4, 4)])
def test_conv_convt_cat(dtype, c, H, W):
    """dec block first conv: ConvTranspose2d(2c->c) of the activated low-res tensor, cat (up, skip), conv 2c->c."""
    rs = _rs(4)
    N = 2
    gl = 4
    low = torch.from_numpy((rs.standard_normal((N, 2 * c, H // 2, W // 2)) * 2).astype(np.float32))
    skip = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2 + 0.3).astype(np.float32))
    ql, seen_l = _nhwc(low, dtype)
    qs, seen_s = _nhwc(skip, dtype)
    g1, b1 = _gn_params(rs, 2 * c)
    g2, b2 = _gn_params(rs, c)
    ctw = torch.from_numpy((rs.standard_normal((2 * c, c, 2, 2)) * (1.0 / np.sqrt(2 * c))).astype(np.float32))
    ctb = torch.from_numpy((rs.standard_normal(c) * 0.2).astype(np.float32))
    w = torch.from_numpy((rs.standard_normal((c, 2 * c, 3, 3)) * (1.0 / np.sqrt(18 * c))).astype(np.float32))
    s0 = ops.make_src(ql, 2 * c, xform=ops.DG_X_CONVT2, stats=_stats(seen_l), gamma=g1.cuda(), beta=b1.cuda(),
                      groups=gl, ct_w=ops.pack_convt2x2(ctw.cuda()), ct_b=ctb.cuda(), ct_cout=c)
    s1 = ops.make_src(qs, c, stats=_stats(seen_s), gamma=g2.cuda(), beta=b2.cuda(), groups=gl)
    out, st = ops.conv3x3_fused([s0, s1], ops.pack_conv3x3(w.cuda()), c, N, H, W, dtype, path=1)
    torch.cuda.synchronize()
    up = F.conv_transpose2d(tpo.gn_silu(seen_l, gl, g1, b1), ctw, ctb, stride=2)
    ref = F.conv2d(torch.cat((up, tpo.gn_silu(seen_s, gl, g2, b2)), 1), w, None, 1, 1)
    _check(out, st, ref, dtype, "convT+cat conv")


@pytest.mark.parametrize("dtype", [ops.DG_F32, ops.DG_F16])
def test_conv_up2_and_scaled_skip(dtype):
    """OptimizedUNet pieces: nearest x2 source (src/optimized_model.py:112) and SE-scaled skip (:199-202)."""
    rs = _rs(5)
    N, c, H, W = 2, 16, 16, 32
    low = torch.from_numpy((rs.standard_normal((N, 2 * c, H // 2, W // 2)) * 2).astype(np.float32))
    ql, seen_l = _nhwc(low, dtype)
    g1, b1 = _gn_params(rs, 2 * c)
    w = torch.from_numpy((rs.standard_normal((c, 2 * c, 3, 3)) * 0.06).astype(np.float32))
    s0 = ops.make_src(ql, 2 * c, xform=ops.DG_X_UP2, stats=_stats(seen_l), gamma=g1.cuda(), beta=b1.cuda(), groups=8)
    out, st = ops.conv3x3_fused([s0], ops.pack_conv3x3(w.cuda()), c, N, H, W, dtype, path=1)
    torch.cuda.synchronize()
    ref = F.conv2d(F.interpolate(tpo.gn_silu(seen_l, 8, g1, b1), scale_factor=2, mode="nearest"), w, None, 1, 1)
    _check(out, st, ref, dtype, "up2 conv")

    a = torch.from_numpy((rs.standard_normal((N, c, H, W))).astype(np.float32))
    s = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2).astype(np.float32))
    qa, seen_a = _nhwc(a, dtype)
    qs, seen_s = _nhwc(s, dtype)
    ga, ba = _gn_params(rs, c)
    gs, bs = _gn_params(rs, c)
    scale = torch.from_numpy(rs.rand(N, c).astype(np.float32))
    w2 = torch.from_numpy((rs.standard_normal((c, 2 * c, 3, 3)) * 0.06).astype(np.float32))
    sa = ops.make_src(qa, c, stats=_stats(seen_a), gamma=ga.cuda(), beta=ba.cuda(), groups=4)
    ss = ops.make_src(qs, c, stats=_stats(seen_s), gamma=gs.cuda(), beta=bs.cuda(), groups=4, scale=scale.cuda())
    out, st = ops.conv3x3_fused([sa, ss], ops.pack_conv3x3(w2.cuda()), c, N, H, W, dtype, path=1)
    torch.cuda.synchronize()
    cat = torch.cat((tpo.gn_silu(seen_a, 4, ga, ba), tpo.gn_silu(seen_s, 4, gs, bs) * scale[:, :, None, None]), 1)
    _check(out, st, F.conv2d(cat, w2, None, 1, 1), dtype, "cat(scaled skip) conv")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("c,oc", [(8, 1), (16, 1), (12, 2)])
def test_head_and_l1(dtype, c, oc):
    rs = _rs(6)
    N, H, W = 2, 48, 32
    groups = 4
    raw = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, c)
    w = torch.from_numpy((rs.standard_normal((oc, c, 1, 1)) * 0.3).astype(np.float32))
    bias = torch.from_numpy(rs.standard_normal(oc).astype(np.float32))
    tgt = torch.from_numpy(rs.rand(N, oc, H, W).astype(np.float32))
    src = ops.make_src(q, c, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=groups)
    l1 = torch.zeros(1, dtype=torch.float64, device="cuda")
    out = ops.head1x1(src, w.reshape(oc, c).contiguous().cuda(), bias.cuda(), N, H, W, dtype, target=tgt.cuda(), l1_sum=l1)
    torch.cuda.synchronize()
    ref = F.conv2d(tpo.gn_silu(seen, groups, g, b), w, bias)
    err = float((out.cpu() - ref).abs().max())
    assert err <= 2e-5 * max(1.0, float(ref.abs().max())), f"head err {err:.3e}"
    want = float((ref - tgt).abs().double().sum())
    assert abs(float(l1.item()) - want) <= 1e-4 * want


def test_errors_are_loud():
    with pytest.raises(RuntimeError):
        ops.make_src(torch.zeros(4), 1)  # CPU tensor
    x = torch.zeros(1, 1, 15, 16, device="cuda")
    w = torch.zeros(3, 3, 2, 8, device="cuda")
    low = torch.zeros(1, 7, 8, 2, device="cuda")
    src = ops.make_src(low, 2, xform=ops.DG_X_UP2, silu=False)
    with pytest.raises(RuntimeError, match="even"):
        ops.conv3x3_fused([src], w, 8, 1, 15, 16, ops.DG_F32)
    del x


# ---- tensor-core (HMMA) path: every LightweightUNet(features_start=8) layer configuration -------------------
TC_DTYPES = [ops.DG_F16, ops.DG_BF16]


def _tc_check(out_tc, st_tc, out_ref, st_ref, dtype, what):
    """TC path vs generic path on identical stored inputs: same math up to fp32 summation order and one
    16-bit rounding of the activated tile -> agree within a few storage ulps of the largest value."""
    a, b = out_tc.float(), out_ref.float()
    scale = max(1.0, float(b.abs().max()))
    err = float((a - b).abs().max())
    tol = (6e-3 if dtype == ops.DG_F16 else 4e-2) * scale
    assert err <= tol, f"{what}: TC vs generic max err {err:.3e} (scale {scale:.2f})"
    serr = float((st_tc - st_ref).abs().max() / max(1.0, float(st_ref.abs().max())))
    assert serr <= 2e-2, f"{what}: stats rel err {serr:.3e}"
    got = a.double()
    want = torch.stack((got.sum(dim=(1, 2)), (got ** 2).sum(dim=(1, 2))), dim=2)
    # TC statistics are taken from the fp32 accumulators, the stored copy is rounded once more
    s2 = float((st_tc - want).abs().max() / max(1.0, float(want.abs().max())))
    assert s2 <= (6e-4 if dtype == ops.DG_F16 else 5e-3), f"{what}: stats do not match stored values ({s2:.3e})"


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("cin,cout,H,W", [(8, 8, 64, 128), (16, 16, 32, 64), (32, 32, 32, 32), (64, 64, 16, 32),
                                            (128, 128, 8, 32), (8, 8, 48, 80), (16, 16, 24, 40), (128, 128, 2, 2),
                                            (64, 64, 6, 10)])
def test_tc_same(dtype, cin, cout, H, W):
    rs = _rs(11)
    N = 2
    raw = torch.from_numpy((rs.standard_normal((N, cin, H, W)) * 3 + 1).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * (1.0 / np.sqrt(9 * cin))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    wtc = ops.pack_conv3x3_tc(wp, dtype)
    st = _stats(seen)
    src = ops.make_src(q, cin, stats=st, gamma=g.cuda(), beta=b.cuda(), groups=8)
    o_ref, s_ref = ops.conv3x3_fused([src], wp, cout, N, H, W, dtype, path=1)
    o_tc, s_tc = ops.conv3x3_fused([src], wp, cout, N, H, W, dtype, path=2, weight_tc=wtc)
    torch.cuda.synchronize()
    _tc_check(o_tc, s_tc, o_ref, s_ref, dtype, f"tc same {cin}->{cout}")
    ref = F.conv2d(tpo.gn_silu(seen, 8, g, b), w, None, 1, 1)
    err = float((o_tc.float().cpu().permute(0, 3, 1, 2) - ref).abs().max())
    assert err <= (6e-3 if dtype == ops.DG_F16 else 4e-2) * max(1.0, float(ref.abs().max())), f"vs oracle {err:.3e}"


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("cin,cout,H,W", [(8, 16, 32, 64), (16, 32, 16, 32), (32, 64, 16, 32), (64, 128, 8, 32),
                                            (8, 16, 24, 40), (64, 128, 1, 1)])
def test_tc_pool(dtype, cin, cout, H, W):
    rs = _rs(12)
    N = 2
    raw = torch.from_numpy((rs.standard_normal((N, cin, 2 * H, 2 * W)) * 2 - 0.5).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * (1.0 / np.sqrt(9 * cin))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    wtc = ops.pack_conv3x3_tc(wp, dtype)
    src = ops.make_src(q, cin, xform=ops.DG_X_POOL2, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=8)
    o_ref, s_ref = ops.conv3x3_fused([src], wp, cout, N, H, W, dtype, path=1)
    o_tc, s_tc = ops.conv3x3_fused([src], wp, cout, N, H, W, dtype, path=2, weight_tc=wtc)
    torch.cuda.synchronize()
    _tc_check(o_tc, s_tc, o_ref, s_ref, dtype, f"tc pool {cin}->{cout}")


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("c,H,W", [(8, 64, 128), (16, 32, 64), (32, 16, 32), (64, 16, 32), (8, 48, 80), (16, 24, 40),
                                     (64, 2, 2), (32, 6, 10)])
def test_tc_convt_cat(dtype, c, H, W):
    rs = _rs(13)
    N = 2
    low = torch.from_numpy((rs.standard_normal((N, 2 * c, H // 2, W // 2)) * 2).astype(np.float32))
    skip = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2 + 0.3).astype(np.float32))
    ql, seen_l = _nhwc(low, dtype)
    qs, seen_s = _nhwc(skip, dtype)
    g1, b1 = _gn_params(rs, 2 * c)
    g2, b2 = _gn_params(rs, c)
    ctw = torch.from_numpy((rs.standard_normal((2 * c, c, 2, 2)) * (1.0 / np.sqrt(2 * c))).astype(np.float32))
    ctb = torch.from_numpy((rs.standard_normal(c) * 0.2).astype(np.float32))
    w = torch.from_numpy((rs.standard_normal((c, 2 * c, 3, 3)) * (1.0 / np.sqrt(18 * c))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    ctp = ops.pack_convt2x2(ctw.cuda())
    s0 = ops.make_src(ql, 2 * c, xform=ops.DG_X_CONVT2, stats=_stats(seen_l), gamma=g1.cuda(), beta=b1.cuda(),
                      groups=8, ct_w=ctp, ct_b=ctb.cuda(), ct_cout=c, ct_w_tc=ops.pack_convt2x2_tc(ctp, dtype))
    s1 = ops.make_src(qs, c, stats=_stats(seen_s), gamma=g2.cuda(), beta=b2.cuda(), groups=8)
    o_ref, s_ref = ops.conv3x3_fused([s0, s1], wp, c, N, H, W, dtype, path=1)
    o_tc, s_tc = ops.conv3x3_fused([s0, s1], wp, c, N, H, W, dtype, path=2, weight_tc=ops.pack_conv3x3_tc(wp, dtype))
    torch.cuda.synchronize()
    _tc_check(o_tc, s_tc, o_ref, s_ref, dtype, f"tc convT+cat {2 * c}->{c}")


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("cout,H,W", [(8, 64, 128), (16, 32, 64), (8, 48, 80), (8, 16, 16), (16, 2, 6)])
def test_tc_first_layer(dtype, cout, H, W):
    rs = _rs(14)
    N = 3
    x = torch.from_numpy(rs.rand(N, 1, H, W).astype(np.float32))
    w = torch.from_numpy((rs.standard_normal((cout, 1, 3, 3)) * 0.4).astype(np.float32))
    src = ops.make_src(x.cuda(), 1, xform=ops.DG_X_IMAGE, silu=False)
    out, st = ops.conv3x3_fused([src], ops.pack_conv3x3(w.cuda()), cout, N, H, W, dtype, path=2)
    torch.cuda.synchronize()
    ref = F.conv2d(x, w, None, 1, 1)
    got = out.float().cpu().permute(0, 3, 1, 2)
    err = float((got - ref).abs().max())
    assert err <= (4e-3 if dtype == ops.DG_F16 else 3e-2) * max(1.0, float(ref.abs().max())), f"first layer err {err:.3e}"
    want = torch.stack((got.double().sum(dim=(2, 3)), (got.double() ** 2).sum(dim=(2, 3))), dim=2)
    serr = float((st.cpu() - want).abs().max() / max(1.0, float(want.abs().max())))
    assert serr <= (6e-4 if dtype == ops.DG_F16 else 5e-3), f"first layer stats {serr:.3e}"


@pytest.mark.parametrize("dtype", TC_DTYPES)
def test_tc_tanh_silu_matches_oracle(dtype):
    """The tanh.approx SiLU of the staging prologue (h + h*tanh(h), h = y/2) against the fp32 oracle."""
    rs = _rs(15)
    N, cin, cout, H, W = 2, 16, 16, 32, 64
    raw = torch.from_numpy((rs.standard_normal((N, cin, H, W)) * 3 + 1).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * (1.0 / np.sqrt(9 * cin))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    wtc = ops.pack_conv3x3_tc(wp, dtype)
    src = ops.make_src(q, cin, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=8)
    o_t, _ = ops.conv3x3_fused([src], wp, cout, N, H, W, dtype, path=2, weight_tc=wtc)
    torch.cuda.synchronize()
    ref = F.conv2d(tpo.gn_silu(seen, 8, g, b), w, None, 1, 1)
    tol = (4e-3 if dtype == ops.DG_F16 else 3e-2) * max(1.0, float(ref.abs().max()))
    assert float((o_t.float().cpu().permute(0, 3, 1, 2) - ref).abs().max()) <= tol


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("c,H,W", [(64, 16, 32), (32, 16, 32), (16, 32, 64), (64, 2, 2), (32, 6, 10)])
def test_tc_standalone_convt_then_cat2(dtype, c, H, W):
    """Deep decoder levels: ConvTranspose as its own tensor-core GEMM, then the conv over (identity up, activated skip)."""
    rs = _rs(16)
    N = 2
    low = torch.from_numpy((rs.standard_normal((N, 2 * c, H // 2, W // 2)) * 2).astype(np.float32))
    skip = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2 + 0.3).astype(np.float32))
    ql, seen_l = _nhwc(low, dtype)
    qs, seen_s = _nhwc(skip, dtype)
    g1, b1 = _gn_params(rs, 2 * c)
    g2, b2 = _gn_params(rs, c)
    ctw = torch.from_numpy((rs.standard_normal((2 * c, c, 2, 2)) * (1.0 / np.sqrt(2 * c))).astype(np.float32))
    ctb = torch.from_numpy((rs.standard_normal(c) * 0.2).astype(np.float32))
    w = torch.from_numpy((rs.standard_normal((c, 2 * c, 3, 3)) * (1.0 / np.sqrt(18 * c))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    ctp = ops.pack_convt2x2(ctw.cuda())
    s0 = ops.make_src(ql, 2 * c, xform=ops.DG_X_CONVT2, stats=_stats(seen_l), gamma=g1.cuda(), beta=b1.cuda(),
                      groups=8, ct_w=ctp, ct_b=ctb.cuda(), ct_cout=c, ct_w_tc=ops.pack_convt2x2_tc(ctp, dtype))
    up = ops.convt2x2_fused(s0, N, H, W, dtype)
    torch.cuda.synchronize()
    up_ref = F.conv_transpose2d(tpo.gn_silu(seen_l, 8, g1, b1), ctw, ctb, stride=2)
    tol = (6e-3 if dtype == ops.DG_F16 else 4e-2) * max(1.0, float(up_ref.abs().max()))
    assert float((up.float().cpu().permute(0, 3, 1, 2) - up_ref).abs().max()) <= tol
    su = ops.make_src(up, c, silu=False)
    s1 = ops.make_src(qs, c, stats=_stats(seen_s), gamma=g2.cuda(), beta=b2.cuda(), groups=8)
    o_ref, st_ref = ops.conv3x3_fused([su, s1], wp, c, N, H, W, dtype, path=1)
    o_tc, st_tc = ops.conv3x3_fused([su, s1], wp, c, N, H, W, dtype, path=2, weight_tc=ops.pack_conv3x3_tc(wp, dtype))
    torch.cuda.synchronize()
    _tc_check(o_tc, st_tc, o_ref, st_ref, dtype, f"tc cat2 {2 * c}->{c}")
    ref = F.conv2d(torch.cat((up.float().cpu().permute(0, 3, 1, 2), tpo.gn_silu(seen_s, 8, g2, b2)), 1), w, None, 1, 1)
    assert float((o_tc.float().cpu().permute(0, 3, 1, 2) - ref).abs().max()) <= (6e-3 if dtype == ops.DG_F16 else 4e-2) * max(
        1.0, float(ref.abs().max()))


def _deep_case(rs, dtype, mode, cin, cout, N, H, W, groups=8):
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) * (1.0 / np.sqrt(9 * cin))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    wtc = ops.pack_conv3x3_tc(wp, dtype)
    if mode == "cat2":
        up = torch.from_numpy((rs.standard_normal((N, cout, H, W)) * 1.5).astype(np.float32))
        skip = torch.from_numpy((rs.standard_normal((N, cout, H, W)) * 2 + 0.3).astype(np.float32))
        qu, seen_u = _nhwc(up, dtype)
        qs, seen = _nhwc(skip, dtype)
        g, b = _gn_params(rs, cout)
        srcs = [ops.make_src(qu, cout, silu=False), ops.make_src(qs, cout, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=groups)]
        act = torch.cat((seen_u, tpo.gn_silu(seen, groups, g, b)), 1)
    else:
        f = 2 if mode == "pool" else 1
        raw = torch.from_numpy((rs.standard_normal((N, cin, f * H, f * W)) * 3 + 1).astype(np.float32))
        q, seen = _nhwc(raw, dtype)
        g, b = _gn_params(rs, cin)
        srcs = [ops.make_src(q, cin, xform=ops.DG_X_POOL2 if mode == "pool" else ops.DG_X_SAME, stats=_stats(seen),
                             gamma=g.cuda(), beta=b.cuda(), groups=groups)]
        act = tpo.gn_silu(seen, groups, g, b)
        if mode == "pool":
            act = F.avg_pool2d(act, 2, 2)
    ref = F.conv2d(act, w, None, 1, 1)
    return srcs, wp, wtc, ref


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("mode,cin,cout,H,W", [("same", 64, 64, 16, 64), ("same", 64, 64, 8, 32), ("same", 64, 64, 12, 40),
                                                 ("pool", 32, 64, 16, 32), ("pool", 32, 64, 6, 10), ("cat2", 64, 32, 16, 64),
                                                 ("cat2", 64, 32, 10, 36)])
def test_hmma_matches_generic(dtype, mode, cin, cout, H, W):
    """The mma.sync kernel (path 2 | 128: the tcgen05 kernel disabled) vs the generic kernel on identical inputs."""
    srcs, wp, wtc, _ = _deep_case(_rs(17), dtype, mode, cin, cout, 3, H, W)
    o_gen, s_gen = ops.conv3x3_fused(srcs, wp, cout, 3, H, W, dtype, path=1)
    o_hm, s_hm = ops.conv3x3_fused(srcs, wp, cout, 3, H, W, dtype, path=2 | 128, weight_tc=wtc)
    torch.cuda.synchronize()
    _tc_check(o_hm, s_hm, o_gen, s_gen, dtype, f"hmma {mode} {cin}->{cout}")


# every deep layer of LightweightUNet(features_start=8) at its real 512^2 geometry plus ragged / tiny shapes, then the channel
# sets of the wide variant (features_start=64: n-blocks, streamed K chunks, single-buffered accumulators)
T5_CASES = [("pool", 16, 32, 128, 128), ("same", 32, 32, 128, 128), ("cat2", 64, 32, 128, 128),
            ("pool", 32, 64, 64, 64), ("same", 64, 64, 64, 64), ("cat2", 128, 64, 64, 64),
            ("pool", 64, 128, 32, 32), ("same", 128, 128, 32, 32),
            ("same", 32, 32, 16, 16), ("same", 64, 64, 12, 40), ("pool", 32, 64, 6, 10), ("cat2", 64, 32, 10, 36),
            ("same", 128, 128, 2, 2), ("pool", 64, 128, 1, 1), ("same", 64, 64, 48, 80),
            ("same", 256, 256, 16, 16), ("pool", 128, 256, 16, 32), ("cat2", 512, 256, 16, 16), ("same", 512, 512, 8, 8),
            ("pool", 512, 1024, 4, 4), ("same", 1024, 1024, 4, 8), ("cat2", 1024, 512, 8, 8),
            # images wider than 128 columns are cut into column strips of 126 (+ 2 halo) columns: wide variant levels 1-2
            ("same", 64, 64, 24, 272), ("pool", 64, 128, 8, 160), ("cat2", 128, 64, 6, 130), ("same", 64, 64, 512, 512)]


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("mode,cin,cout,H,W", T5_CASES)
def test_t5_warp_specialised_tcgen05_conv(dtype, mode, cin, cout, H, W):
    """Round-2 tcgen05 kernel (path 2 | 256 = insist on it) vs the oracle's decomposition and vs the generic CUDA-core kernel."""
    N = 3 if H * W <= 4096 else 2
    srcs, wp, wtc, ref = _deep_case(_rs(18), dtype, mode, cin, cout, N, H, W)
    o_t5, s_t5 = ops.conv3x3_fused(srcs, wp, cout, N, H, W, dtype, path=2 | 256, weight_tc=wtc)
    torch.cuda.synchronize()
    got = o_t5.float().cpu().permute(0, 3, 1, 2)
    scale = max(1.0, float(ref.abs().max()))
    err = float((got - ref).abs().max())
    assert err <= (6e-3 if dtype == ops.DG_F16 else 4e-2) * scale, f"t5 {mode} {cin}->{cout} vs oracle: {err:.3e} (scale {scale:.2f})"
    # the epilogue's statistics are those of the STORED values
    want = torch.stack((got.double().sum(dim=(2, 3)), (got.double() ** 2).sum(dim=(2, 3))), dim=2)
    serr = float((s_t5.cpu() - want).abs().max() / max(1.0, float(want.abs().max())))
    assert serr <= 2e-5, f"t5 {mode} {cin}->{cout}: stats rel err {serr:.3e}"
    if cin * cout <= 128 * 128:
        o_gen, s_gen = ops.conv3x3_fused(srcs, wp, cout, N, H, W, dtype, path=1)
        torch.cuda.synchronize()
        _tc_check(o_t5, s_t5, o_gen, s_gen, dtype, f"t5 {mode} {cin}->{cout}")


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("c,H,W", [(64, 16, 32), (32, 16, 32), (64, 2, 2), (32, 6, 10), (128, 32, 32), (256, 16, 16), (512, 8, 8),
                                     (64, 128, 128), (64, 8, 520), (64, 512, 512)])
def test_t5_convtranspose(dtype, c, H, W):
    """ConvTranspose2d(2c -> c, k=2, s=2) + bias of the activated low-resolution tensor on the tcgen05 kernel (1-tap GEMM, N = 4c):
    upconv4 / upconv3 of the shipped model and every up-convolution of the wide variant."""
    rs = _rs(21)
    N = 2
    low = torch.from_numpy((rs.standard_normal((N, 2 * c, H // 2, W // 2)) * 2).astype(np.float32))
    ql, seen_l = _nhwc(low, dtype)
    g1, b1 = _gn_params(rs, 2 * c)
    ctw = torch.from_numpy((rs.standard_normal((2 * c, c, 2, 2)) * (1.0 / np.sqrt(2 * c))).astype(np.float32))
    ctb = torch.from_numpy((rs.standard_normal(c) * 0.2).astype(np.float32))
    ctp = ops.pack_convt2x2(ctw.cuda())
    s0 = ops.make_src(ql, 2 * c, xform=ops.DG_X_CONVT2, stats=_stats(seen_l), gamma=g1.cuda(), beta=b1.cuda(),
                      groups=8, ct_w=ctp, ct_b=ctb.cuda(), ct_cout=c, ct_w_tc=ops.pack_convt2x2_tc(ctp, dtype))
    up = ops.convt2x2_fused(s0, N, H, W, dtype, path=256)   # bit 8: insist on the tcgen05 kernel
    torch.cuda.synchronize()
    up_ref = F.conv_transpose2d(tpo.gn_silu(seen_l, 8, g1, b1), ctw, ctb, stride=2)
    tol = (6e-3 if dtype == ops.DG_F16 else 4e-2) * max(1.0, float(up_ref.abs().max()))
    err = float((up.float().cpu().permute(0, 3, 1, 2) - up_ref).abs().max())
    assert err <= tol, f"convT {2 * c}->{c}: {err:.3e}"
    if c <= 64:   # the mma.sync kernel (path bit 7) must agree
        up_h = ops.convt2x2_fused(s0, N, H, W, dtype, path=128)
        torch.cuda.synchronize()
        assert float((up.float() - up_h.float()).abs().max()) <= 0.5 * tol


def test_t5_is_the_default_for_deep_layers_and_can_be_disabled():
    srcs, wp, wtc, _ = _deep_case(_rs(19), ops.DG_F16, "same", 64, 64, 2, 16, 32)
    o_def, _ = ops.conv3x3_fused(srcs, wp, 64, 2, 16, 32, ops.DG_F16, weight_tc=wtc)
    o_t5, _ = ops.conv3x3_fused(srcs, wp, 64, 2, 16, 32, ops.DG_F16, path=2 | 256, weight_tc=wtc)
    o_hm, _ = ops.conv3x3_fused(srcs, wp, 64, 2, 16, 32, ops.DG_F16, path=2 | 128, weight_tc=wtc)
    torch.cuda.synchronize()
    assert torch.equal(o_def, o_t5)
    assert float((o_t5.float() - o_hm.float()).abs().max()) <= 2e-3 * max(1.0, float(o_hm.float().abs().max()))
    src8 = _deep_case(_rs(19), ops.DG_F16, "same", 8, 8, 2, 16, 32)
    with pytest.raises(RuntimeError, match="t5"):
        ops.conv3x3_fused(src8[0], src8[1], 8, 2, 16, 32, ops.DG_F16, path=2 | 256, weight_tc=src8[2])


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("N,H,W", [(2, 64, 128), (3, 48, 80), (1, 16, 64), (2, 16, 16), (5, 128, 192), (1, 512, 512)])
def test_ring_tma_kernel_matches_per_tile_kernel(dtype, N, H, W):
    """Persistent TMA-fed 8 -> 8 kernel (default) vs the per-tile mma.sync kernel (path bit 9) vs the oracle: same fp16 operands,
    same fp32 accumulation order inside an MMA -> they agree to a rounding of the stored value."""
    rs = _rs(23)
    raw = torch.from_numpy((rs.standard_normal((N, 8, H, W)) * 3 + 1).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, 8)
    w = torch.from_numpy((rs.standard_normal((8, 8, 3, 3)) * (1.0 / np.sqrt(72))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    wtc = ops.pack_conv3x3_tc(wp, dtype)
    src = ops.make_src(q, 8, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=8)
    o_ring, s_ring = ops.conv3x3_fused([src], wp, 8, N, H, W, dtype, path=2, weight_tc=wtc)
    o_tile, s_tile = ops.conv3x3_fused([src], wp, 8, N, H, W, dtype, path=2 | 512, weight_tc=wtc)
    torch.cuda.synchronize()
    scale = max(1.0, float(o_tile.float().abs().max()))
    assert float((o_ring.float() - o_tile.float()).abs().max()) <= (1e-3 if dtype == ops.DG_F16 else 8e-3) * scale
    assert float((s_ring - s_tile).abs().max() / max(1.0, float(s_tile.abs().max()))) <= 1e-5
    ref = F.conv2d(tpo.gn_silu(seen, 8, g, b), w, None, 1, 1)
    err = float((o_ring.float().cpu().permute(0, 3, 1, 2) - ref).abs().max())
    assert err <= (6e-3 if dtype == ops.DG_F16 else 4e-2) * max(1.0, float(ref.abs().max())), f"ring vs oracle {err:.3e}"
    got = o_ring.float().cpu().permute(0, 3, 1, 2).double()
    want = torch.stack((got.sum(dim=(2, 3)), (got ** 2).sum(dim=(2, 3))), dim=2)
    assert float((s_ring.cpu() - want).abs().max() / max(1.0, float(want.abs().max()))) <= 6e-4


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("N,H,W", [(2, 64, 128), (3, 48, 80), (1, 16, 64), (2, 16, 16), (2, 2, 2), (3, 34, 66), (1, 512, 512)])
def test_composite_decoder_kernel(dtype, N, H, W):
    """upconv1 + dec1.0 with the ConvTranspose folded into the conv taps (conv3x3_dec.cu: 2x2 composite taps per output parity
    class, border-corrected bias, TMA-fed) vs the oracle's ConvTranspose -> cat -> conv and vs the round-1 fused kernel."""
    rs = _rs(29)
    c = 8
    low = torch.from_numpy((rs.standard_normal((N, 2 * c, H // 2, W // 2)) * 2).astype(np.float32))
    skip = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2 + 0.3).astype(np.float32))
    ql, seen_l = _nhwc(low, dtype)
    qs, seen_s = _nhwc(skip, dtype)
    g1, b1 = _gn_params(rs, 2 * c)
    g2, b2 = _gn_params(rs, c)
    ctw = torch.from_numpy((rs.standard_normal((2 * c, c, 2, 2)) * (1.0 / np.sqrt(2 * c))).astype(np.float32))
    ctb = torch.from_numpy((rs.standard_normal(c) * 0.5).astype(np.float32))     # a bias large enough to expose border mistakes
    w = torch.from_numpy((rs.standard_normal((c, 2 * c, 3, 3)) * (1.0 / np.sqrt(18 * c))).astype(np.float32))
    wp = ops.pack_conv3x3(w.cuda())
    ctp = ops.pack_convt2x2(ctw.cuda())
    s0 = ops.make_src(ql, 2 * c, xform=ops.DG_X_CONVT2, stats=_stats(seen_l), gamma=g1.cuda(), beta=b1.cuda(),
                      groups=8, ct_w=ctp, ct_b=ctb.cuda(), ct_cout=c, ct_w_tc=ops.pack_convt2x2_tc(ctp, dtype))
    s1 = ops.make_src(qs, c, stats=_stats(seen_s), gamma=g2.cuda(), beta=b2.cuda(), groups=8)
    comp = ops.pack_dec_composite(ctp, ctb.cuda(), wp, dtype)
    assert comp is not None
    wtc = ops.pack_conv3x3_tc(wp, dtype)
    o_c, s_c = ops.conv3x3_fused([s0, s1], wp, c, N, H, W, dtype, path=2, weight_tc=wtc, weight_comp=comp)
    o_h, s_h = ops.conv3x3_fused([s0, s1], wp, c, N, H, W, dtype, path=2 | 1024, weight_tc=wtc, weight_comp=comp)
    torch.cuda.synchronize()
    up = F.conv_transpose2d(tpo.gn_silu(seen_l, 8, g1, b1), ctw, ctb, stride=2)
    ref = F.conv2d(torch.cat((up, tpo.gn_silu(seen_s, 8, g2, b2)), 1), w, None, 1, 1)
    scale = max(1.0, float(ref.abs().max()))
    tol = (6e-3 if dtype == ops.DG_F16 else 4e-2) * scale
    got = o_c.float().cpu().permute(0, 3, 1, 2)
    assert float((got - ref).abs().max()) <= tol, f"composite vs oracle {float((got - ref).abs().max()):.3e} (scale {scale:.2f})"
    assert float((o_c.float() - o_h.float()).abs().max()) <= tol
    want = torch.stack((got.double().sum(dim=(2, 3)), (got.double() ** 2).sum(dim=(2, 3))), dim=2)
    # statistics come from the fp32 accumulators, the stored copy is rounded once more: relative to the plane sums that is
    # ~2^-12 / sqrt(pixels) -- visible only on the tiny shapes
    assert float((s_c.cpu() - want).abs().max() / max(1.0, float(want.abs().max()))) <= (6e-4 if H * W >= 1024 else 5e-3)
    assert not torch.equal(o_c, o_h) or H * W <= 4      # really two different kernels


DGRAD_CASES = [(8, 8), (8, 16), (16, 16), (16, 32), (32, 32), (32, 64), (64, 64), (64, 128), (128, 128), (128, 64), (64, 32), (32, 16), (16, 8)]


@pytest.mark.parametrize("cin,cout", DGRAD_CASES)
@pytest.mark.parametrize("N,H,W", [(2, 32, 64), (3, 24, 40), (1, 8, 8)])
def test_dgrad_tc_matches_autograd(cin, cout, N, H, W):
    """dg_conv3x3_dgrad (dgrad_tc.cu: reads the forward weights' tensor-core packing transposed, bf16 operands) vs autograd of
    F.conv2d w.r.t. its input (src/model.py:93,96), every (C_in, C_out) pair of the shipped network."""
    rs = _rs(41 + cin + cout)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) / np.sqrt(9 * cin)).astype(np.float32))
    dR = torch.from_numpy(rs.standard_normal((N, cout, H, W)).astype(np.float32))
    x = torch.zeros(N, cin, H, W, requires_grad=True)
    F.conv2d(x, w, None, 1, 1).backward(dR)
    ref = x.grad
    wtc = ops.pack_conv3x3_tc(ops.pack_conv3x3(w.cuda()), ops.DG_BF16)
    got = ops.conv3x3_dgrad(dR.permute(0, 2, 3, 1).contiguous().cuda(), wtc, cin, cout).cpu().permute(0, 3, 1, 2)
    # bf16 rounding of both operands: relative 2^-8 per product, sqrt(9 cout) products per sum
    scale = float(ref.abs().max())
    assert float((got - ref).abs().max()) <= 1.5e-2 * scale, f"{float((got - ref).abs().max()):.3e} vs scale {scale:.3e}"
    rel = float((got - ref).norm() / ref.norm())
    assert rel <= 5e-3, rel
    # against the same product with operands rounded the way the kernel rounds them: tight
    xq = torch.zeros(N, cin, H, W, requires_grad=True)
    F.conv2d(xq, w.bfloat16().float(), None, 1, 1).backward(dR.bfloat16().float())
    assert float((got - xq.grad).abs().max()) <= 2e-5 * max(1.0, scale) * np.sqrt(9 * cout)


@pytest.mark.parametrize("cl,cu", [(128, 64), (64, 32), (32, 16), (16, 8)])
@pytest.mark.parametrize("N,H,W,interleaved", [(2, 32, 64, True), (3, 16, 24, False), (1, 8, 8, True)])
def test_convt_dgrad_tc_matches_autograd(cl, cu, N, H, W, interleaved):
    """dg_convt2x2_dgrad vs autograd of F.conv_transpose2d w.r.t. its input (src/model.py:47-53); the up-half gradient is read from
    the concat gradient either interleaved with the skip half (stride 2 C) or compact (stride C)."""
    rs = _rs(43 + cl)
    wt = torch.from_numpy((rs.standard_normal((cl, cu, 2, 2)) / np.sqrt(cl)).astype(np.float32))
    dUp = torch.from_numpy(rs.standard_normal((N, cu, H, W)).astype(np.float32))
    low = torch.zeros(N, cl, H // 2, W // 2, requires_grad=True)
    F.conv_transpose2d(low, wt, None, stride=2).backward(dUp)
    ref = low.grad
    nhwc = dUp.permute(0, 2, 3, 1).contiguous()
    dCat = torch.cat((nhwc, torch.full_like(nhwc, 7.0)), 3).contiguous() if interleaved else nhwc   # the skip half must be ignored
    wtc = ops.pack_convt2x2_tc(ops.pack_convt2x2(wt.cuda()), ops.DG_BF16)
    got = ops.convt2x2_dgrad(dCat.cuda(), wtc, cl, cu).cpu().permute(0, 3, 1, 2)
    scale = float(ref.abs().max())
    assert float((got - ref).abs().max()) <= 1.5e-2 * scale
    assert float((got - ref).norm() / ref.norm()) <= 5e-3
    lq = torch.zeros(N, cl, H // 2, W // 2, requires_grad=True)
    F.conv_transpose2d(lq, wt.bfloat16().float(), None, stride=2).backward(dUp.bfloat16().float())
    assert float((got - lq.grad).abs().max()) <= 2e-5 * max(1.0, scale) * np.sqrt(4 * cu)


@pytest.mark.parametrize("cin,cout,N,H,W", [(64, 64, 2, 32, 64), (128, 64, 1, 16, 32), (256, 128, 2, 8, 8), (256, 256, 1, 24, 40),
                                              (512, 1024, 1, 4, 4), (1024, 512, 2, 2, 2), (64, 128, 1, 16, 160), (32, 16, 1, 8, 8)])
def test_dgrad_wide_tcgen05_matches_autograd(cin, cout, N, H, W):
    """dg_conv3x3_dgrad_wide (conv3x3_t5.cu T5_IDENT: dR rounded to bf16, taps-flipped weights in the tensor-core packing, tcgen05
    implicit GEMM, fp32 out) vs autograd of F.conv2d w.r.t. its input (src/model.py:93,96) on the wide variant's channel sets."""
    rs = _rs(47 + cin + cout)
    w = torch.from_numpy((rs.standard_normal((cout, cin, 3, 3)) / np.sqrt(9 * cin)).astype(np.float32))
    dR = torch.from_numpy(rs.standard_normal((N, cout, H, W)).astype(np.float32))
    x = torch.zeros(N, cin, H, W, dtype=torch.float64, requires_grad=True)
    F.conv2d(x, w.double(), None, 1, 1).backward(dR.double())
    ref = x.grad.float()
    wflip_tc = ops.pack_conv3x3_tc(ops.flip_conv3x3(w.cuda()), ops.DG_BF16)
    got = ops.conv3x3_dgrad_wide(dR.permute(0, 2, 3, 1).contiguous().cuda(), wflip_tc, cin, cout).cpu().permute(0, 3, 1, 2)
    scale = float(ref.abs().max())
    assert float((got - ref).abs().max()) <= 1.5e-2 * scale, f"{float((got - ref).abs().max()):.3e} vs scale {scale:.3e}"
    assert float((got - ref).norm() / ref.norm()) <= 5e-3
    xq = torch.zeros(N, cin, H, W, dtype=torch.float64, requires_grad=True)
    F.conv2d(xq, w.bfloat16().double(), None, 1, 1).backward(dR.bfloat16().double())
    assert float((got - xq.grad.float()).abs().max()) <= 2e-5 * max(1.0, scale) * np.sqrt(9 * cout)


def test_dgrad_wide_refuses_what_it_has_no_plan_for():
    dR = torch.zeros(1, 8, 8, 32, device="cuda")
    w = torch.zeros(9 * 32 * 16 * 2, dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError, match="no tcgen05 plan"):
        ops.conv3x3_dgrad_wide(dR, w, 16, 32)        # 16 result channels: below the N = 32 minimum of the tcgen05 tile


def test_dgrad_refuses_uncovered_channel_sets():
    dR = torch.zeros(1, 8, 8, 24, device="cuda")
    w = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    with pytest.raises(RuntimeError, match="no tensor-core kernel"):
        ops.conv3x3_dgrad(dR, w, 24, 24)
    with pytest.raises(RuntimeError, match="no tensor-core kernel"):
        ops.convt2x2_dgrad(dR, w, 48, 24)


def test_tc_path_refuses_unsupported():
    w = torch.zeros(3, 3, 24, 24, device="cuda")
    raw = torch.zeros(1, 8, 8, 24, device="cuda", dtype=torch.float16)
    st = torch.ones(1, 24, 2, dtype=torch.float64, device="cuda")
    g = torch.ones(24, device="cuda")
    src = ops.make_src(raw, 24, stats=st, gamma=g, beta=g, groups=8)
    with pytest.raises(RuntimeError, match="tensor-core"):
        ops.conv3x3_fused([src], w, 24, 1, 8, 8, ops.DG_F16, path=2)


# ---- weight gradient: tensor-core kernel (bf16 operands, fp32 accumulate) vs generic kernel vs torch autograd ----------
def _wgrad_ref(act_in, dR_nchw, cout):
    """d/dW of sum(conv2d(act_in, W) * dR): the reference's autograd on the ACTIVATED input."""
    w = torch.zeros((cout, act_in.shape[1], 3, 3), dtype=torch.float64, requires_grad=True)
    (F.conv2d(act_in.double(), w, None, 1, 1) * dR_nchw.double()).sum().backward()
    return w.grad.float()


def _wgrad_check(dw_tc, dw_gen, ref, what):
    scale = float(ref.abs().max())
    e_gen = float((dw_gen.cpu() - ref).abs().max()) / scale
    e_tc = float((dw_tc.cpu() - ref).abs().max()) / scale
    assert e_gen <= 2e-3, f"{what}: generic wgrad rel err {e_gen:.3e}"
    # bf16 operands: 2^-9 relative rounding per factor, averaged over K = N*H*W products
    assert e_tc <= 1e-2, f"{what}: tensor-core wgrad rel err {e_tc:.3e} (generic {e_gen:.3e})"


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("cin,cout,H,W", [(8, 8, 64, 128), (16, 16, 32, 64), (32, 32, 32, 32), (64, 64, 16, 32),
                                            (128, 128, 8, 32), (8, 8, 48, 80), (32, 32, 6, 10),
                                            (256, 256, 8, 32), (512, 512, 4, 8), (1024, 1024, 2, 4)])   # wider variants (configs[4])
def test_wgrad_tc_same(dtype, cin, cout, H, W):
    rs = _rs(41)
    N = 3
    raw = torch.from_numpy((rs.standard_normal((N, cin, H, W)) * 2 + 0.5).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    dR = torch.from_numpy((rs.standard_normal((N, H, W, cout)) * 1e-6).astype(np.float32)).cuda()   # ~1/numel: underflows fp16
    src = ops.make_src(q, cin, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=8)
    dw_gen = ops.conv3x3_wgrad([src], dR, cin, cout, N, H, W, dtype, path=1)
    dw_tc = ops.conv3x3_wgrad([src], dR, cin, cout, N, H, W, dtype, path=2)
    torch.cuda.synchronize()
    ref = _wgrad_ref(tpo.gn_silu(seen, 8, g, b), dR.cpu().permute(0, 3, 1, 2), cout)
    _wgrad_check(dw_tc, dw_gen, ref, f"wgrad same {cin}->{cout}")


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("cin,cout,H,W", [(8, 16, 32, 64), (16, 32, 16, 32), (32, 64, 16, 32), (64, 128, 8, 32), (8, 16, 24, 40),
                                            (128, 256, 8, 32), (256, 512, 4, 8), (512, 1024, 2, 4)])
def test_wgrad_tc_pool(dtype, cin, cout, H, W):
    rs = _rs(42)
    N = 2
    raw = torch.from_numpy((rs.standard_normal((N, cin, 2 * H, 2 * W)) * 2 - 0.5).astype(np.float32))
    q, seen = _nhwc(raw, dtype)
    g, b = _gn_params(rs, cin)
    dR = torch.from_numpy((rs.standard_normal((N, H, W, cout)) * 1e-6).astype(np.float32)).cuda()
    src = ops.make_src(q, cin, xform=ops.DG_X_POOL2, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=8)
    dw_gen = ops.conv3x3_wgrad([src], dR, cin, cout, N, H, W, dtype, path=1)
    dw_tc = ops.conv3x3_wgrad([src], dR, cin, cout, N, H, W, dtype, path=2)
    torch.cuda.synchronize()
    ref = _wgrad_ref(F.avg_pool2d(tpo.gn_silu(seen, 8, g, b), 2), dR.cpu().permute(0, 3, 1, 2), cout)
    _wgrad_check(dw_tc, dw_gen, ref, f"wgrad pool {cin}->{cout}")


@pytest.mark.parametrize("dtype", TC_DTYPES)
@pytest.mark.parametrize("c,H,W", [(8, 64, 128), (16, 32, 64), (32, 16, 32), (64, 16, 32), (8, 48, 80), (128, 8, 32), (256, 4, 8),
                                   (512, 2, 4)])
def test_wgrad_tc_cat(dtype, c, H, W):
    """Decoder conv: input = cat(materialised ConvTranspose output, activated skip)."""
    rs = _rs(43)
    N = 2
    up = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 1.5).astype(np.float32))
    skip = torch.from_numpy((rs.standard_normal((N, c, H, W)) * 2 + 0.3).astype(np.float32))
    qu, seen_u = _nhwc(up, dtype)
    qs, seen_s = _nhwc(skip, dtype)
    g, b = _gn_params(rs, c)
    dR = torch.from_numpy((rs.standard_normal((N, H, W, c)) * 1e-6).astype(np.float32)).cuda()
    s0 = ops.make_src(qu, c, silu=False)
    s1 = ops.make_src(qs, c, stats=_stats(seen_s), gamma=g.cuda(), beta=b.cuda(), groups=8)
    dw_gen = ops.conv3x3_wgrad([s0, s1], dR, 2 * c, c, N, H, W, dtype, path=1)
    dw_tc = ops.conv3x3_wgrad([s0, s1], dR, 2 * c, c, N, H, W, dtype, path=2)
    torch.cuda.synchronize()
    ref = _wgrad_ref(torch.cat((seen_u, tpo.gn_silu(seen_s, 8, g, b)), 1), dR.cpu().permute(0, 3, 1, 2), c)
    _wgrad_check(dw_tc, dw_gen, ref, f"wgrad cat {2 * c}->{c}")


def test_wgrad_tc_refuses_what_it_does_not_cover():
    rs = _rs(44)
    q, seen = _nhwc(torch.from_numpy(rs.standard_normal((1, 24, 16, 16)).astype(np.float32)), ops.DG_F16)
    g, b = _gn_params(rs, 24)
    src = ops.make_src(q, 24, stats=_stats(seen), gamma=g.cuda(), beta=b.cuda(), groups=8)
    dR = torch.zeros((1, 16, 16, 24), device="cuda")
    with pytest.raises(RuntimeError):
        ops.conv3x3_wgrad([src], dR, 24, 24, 1, 16, 16, ops.DG_F16, path=2)
    ops.conv3x3_wgrad([src], dR, 24, 24, 1, 16, 16, ops.DG_F16, path=0)   # auto falls back to the generic kernel


# ---- per-op backward of GroupNorm + SiLU (dg_act_bwd, dg_gn_bwd_apply): shipped widths and the wide variant's (per-group prologue) ----
@pytest.mark.parametrize("dtype", [ops.DG_F32, ops.DG_F16])
@pytest.mark.parametrize("C,groups,H,W,pooled", [(16, 8, 16, 24, True), (128, 8, 8, 8, False), (256, 8, 8, 12, True), (1024, 8, 4, 4, False),
                                                   (512, 4, 6, 10, False), (12, 6, 8, 8, False)])
def test_act_and_groupnorm_backward_ops(dtype, C, groups, H, W, pooled):
    """G = (dA_a + AvgPool2d-backward(dA_b)) * SiLU'(y), P sums, then dR / dgamma / dbeta in place, against autograd of
    F.silu(F.group_norm(raw)) (src/model.py:94-98) consumed same-resolution and (optionally) through nn.AvgPool2d(2, 2)."""
    gen = torch.Generator().manual_seed(5 + C)
    N = 2
    raw = (torch.randn(N, H, W, C, generator=gen) * 1.5 + 0.3).to(ops.TORCH_DTYPE[dtype]).cuda()
    gamma = (1 + 0.2 * torch.randn(C, generator=gen)).cuda().requires_grad_(True)
    beta = (0.2 * torch.randn(C, generator=gen)).cuda().requires_grad_(True)
    dA = torch.randn(N, H, W, 2 * C, generator=gen).cuda()                 # one half of a concat gradient: channels C .. 2C
    dB = torch.randn(N, H // 2, W // 2, C, generator=gen).cuda() if pooled else None
    r = raw.float().requires_grad_(True)
    act = F.silu(F.group_norm(r.permute(0, 3, 1, 2), groups, gamma, beta, 1e-5))
    loss = (act * dA[..., C:].permute(0, 3, 1, 2)).sum()
    if pooled:
        loss = loss + (F.avg_pool2d(act, 2, 2) * dB.permute(0, 3, 1, 2)).sum()
    loss.backward()
    stats = torch.stack((raw.double().sum(dim=(1, 2)), (raw.double() ** 2).sum(dim=(1, 2))), dim=-1).contiguous()
    G = torch.empty(N, H, W, C, device="cuda")
    P = torch.zeros(N, C, 2, dtype=torch.float64, device="cuda")
    g, b = gamma.detach(), beta.detach()
    ops.act_bwd(raw, stats, g, b, groups, dtype, N, H, W, C, G, P, dA_a=dA, off_a=C, dA_b=dB)
    dgamma, dbeta = torch.zeros(C, device="cuda"), torch.zeros(C, device="cuda")
    ops.gn_bwd_apply(raw, stats, g, groups, dtype, N, H, W, C, P, G, dgamma, dbeta)
    for got, ref, what in ((G, r.grad, "dR"), (dgamma, gamma.grad, "dgamma"), (dbeta, beta.grad, "dbeta")):
        err = float((got - ref).abs().max())
        assert err <= 2e-4 * float(ref.abs().max()) + 1e-6, (what, err, float(ref.abs().max()))


# ---- the two device steps of the row-sharded whole-image path and the graph-capturable optimizer tail -----------------------------
@pytest.mark.parametrize("tdtype,code", [(torch.float32, 0), (torch.float16, 1), (torch.bfloat16, 2)])
@pytest.mark.parametrize("C,W,rows,c0,own0,own1,c1", [(8, 64, 20, 0, 2, 18, 20), (16, 48, 11, 1, 2, 10, 10), (12, 32, 9, 0, 0, 7, 9),
                                                     (128, 16, 6, 1, 2, 4, 5), (1024, 4, 5, 0, 1, 4, 5)])
def test_band_stats_subtracts_the_computed_halo_rows(tdtype, code, C, W, rows, c0, own0, own1, c1):
    """dg_band_stats: kernel statistics over the computed rows [c0, c1) minus the halo rows [c0, own0) and [own1, c1) = the sums
    over the owned rows, in double (whole_image.py; nn.GroupNorm over the whole image, src/model.py:94,97)."""
    import ctypes as C_
    from image_enhancement_deglaring_b200 import _lib
    g = torch.Generator().manual_seed(C + rows)
    t = (torch.randn(rows, W, C, generator=g) * 2).to(tdtype).cuda()
    d = t.double()
    full = torch.stack((d[c0:c1].sum((0, 1)), (d[c0:c1] ** 2).sum((0, 1))), -1)        # what the conv epilogue hands over
    want = torch.stack((d[own0:own1].sum((0, 1)), (d[own0:own1] ** 2).sum((0, 1))), -1)
    out = torch.empty_like(full)
    _lib.check(_lib.load().dg_band_stats(full.data_ptr(), t.data_ptr(), code, W, C, c0, own0, own1, c1, out.data_ptr(),
                                         torch.cuda.current_stream().cuda_stream))
    assert float((out - want).abs().max()) <= 1e-9 * max(1.0, float(full.abs().max()))
    with pytest.raises(RuntimeError):
        _lib.check(_lib.load().dg_band_stats(full.data_ptr(), t.data_ptr(), code, W, C, 3, 2, own1, c1, out.data_ptr(), None))


@pytest.mark.parametrize("C,groups,parts", [(8, 8, 1), (16, 8, 2), (12, 6, 3), (128, 8, 8), (1024, 8, 2)])
def test_gn_affine_from_gathered_partial_sums(C, groups, parts):
    """dg_gn_affine: partial (sum, sum of squares) blocks of all ranks, one every `stride` doubles, added in block order -> the
    GroupNorm affine (a, b) with y = x * a + b equal to F.group_norm on the full tensor."""
    from image_enhancement_deglaring_b200 import _lib
    g = torch.Generator().manual_seed(C + parts)
    H, W = 6 * parts, 10
    x = torch.randn(1, C, H, W, generator=g) * 1.5 + 0.3
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    want = F.group_norm(x, groups, gamma, beta, 1e-5)
    stride = 2 * C + 24                                   # packets carry rows behind the statistics
    buf = torch.zeros(parts, stride, dtype=torch.float64)
    for r in range(parts):
        band = x[0, :, r * 6:(r + 1) * 6].double()
        buf[r, :2 * C] = torch.stack((band.sum((1, 2)), (band ** 2).sum((1, 2))), -1).reshape(-1)
    buf[:, 2 * C:] = 1e30                                  # must not be read
    coef = torch.empty(C, 2, dtype=torch.float32, device="cuda")
    dbuf, dgamma, dbeta = buf.cuda(), gamma.cuda(), beta.cuda()      # named: the library only borrows the pointers
    _lib.check(_lib.load().dg_gn_affine(dbuf.data_ptr(), parts, stride, dgamma.data_ptr(), dbeta.data_ptr(), C, groups,
                                        float(H * W), 1e-5, coef.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    c = coef.cpu()
    got = x * c[:, 0].view(1, C, 1, 1) + c[:, 1].view(1, C, 1, 1)
    assert float((got - want).abs().max()) <= 2e-5
    with pytest.raises(RuntimeError):
        _lib.check(_lib.load().dg_gn_affine(buf.data_ptr(), parts, stride, gamma.data_ptr(), beta.data_ptr(), C, 5 if C % 5 else 7, float(H * W),
                                            1e-5, coef.data_ptr(), None))


def test_adamw_step_graph_equals_host_step_flavour():
    """dg_adamw_step_graph (step count and learning rate in device memory) performs exactly the update of dg_adamw_step, step after step."""
    from image_enhancement_deglaring_b200 import _lib
    lib = _lib.load()
    n = 10007
    g0 = torch.Generator().manual_seed(3)
    p0 = torch.randn(n, generator=g0)
    pa, pb = p0.clone().cuda(), p0.clone().cuda()
    ma, va, mb, vb = (torch.zeros(n, device="cuda") for _ in range(4))
    sa, sb = torch.zeros(1, dtype=torch.float64, device="cuda"), torch.zeros(1, dtype=torch.float64, device="cuda")
    step_dev = torch.zeros(1, dtype=torch.int32, device="cuda")
    lr_dev = torch.zeros(1, dtype=torch.float32, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for step, lr in enumerate((1e-3, 1e-3, 5e-4, 2e-3), start=1):
        gr = (torch.randn(n, generator=g0) * (10.0 if step == 2 else 0.01)).cuda()     # step 2 is clipped
        _lib.check(lib.dg_adamw_step(pa.data_ptr(), gr.data_ptr(), ma.data_ptr(), va.data_ptr(), n, sa.data_ptr(), 1.0, lr, 0.9, 0.999, 1e-8,
                                     0.01, step, 1.0, st))
        lr_dev.fill_(lr)
        _lib.check(lib.dg_adamw_step_graph(pb.data_ptr(), gr.data_ptr(), mb.data_ptr(), vb.data_ptr(), n, sb.data_ptr(), 1.0, lr_dev.data_ptr(),
                                           0.9, 0.999, 1e-8, 0.01, step_dev.data_ptr(), 1.0, st))
        assert int(step_dev.item()) == step
        # the gradient's sum of squares is reduced with double atomics (order noise ~1e-16), so the clip factor may move by an ulp
        assert float((pa - pb).abs().max()) <= 1e-7
        assert torch.allclose(ma, mb, rtol=1e-6, atol=0) and torch.allclose(va, vb, rtol=1e-6, atol=0)
        assert abs(float(sa.item()) - float(sb.item())) <= 1e-12 * float(sa.item())
