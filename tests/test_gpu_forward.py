"""GPU parity of the whole LightweightUNet forward (drop-in nn.Module over the C-ABI) against the
oracle and the reference-generated golden vectors.  Tolerances are BASELINE.json's north_star:
fp32 max-abs <= 2e-3 (we hold 2e-4), 16-bit <= 5e-3, PSNR >= 50 dB."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import torch_unet as tpo
from dg_testutil import psnr

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import det_state_dict  # noqa: E402

pytestmark = pytest.mark.gpu

dg = pytest.importorskip("image_enhancement_deglaring_b200")


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def _net(sd, **kw):
    net = dg.LightweightUNet(**kw)
    net.load_state_dict(sd, strict=True)
    return net.cuda().eval()


def test_png_golden_fp32(best_sd, golden):
    g = golden("lw_png.npz")
    net = _net(best_sd)
    for i in (1, 2):
        x = torch.from_numpy(g[f"x{i}_u8"].astype(np.float32) / 255.0)[None, None].cuda()
        with torch.no_grad():
            y = net(x)[0, 0].cpu().numpy()
        err = np.abs(y - g[f"y{i}"]).max()
        assert err <= 2e-4, f"png{i}: max-abs {err:.3e}"
        assert psnr(y, g[f"y{i}"]) >= 80.0


@pytest.mark.parametrize("storage,tol,min_psnr", [("fp16", 5e-3, 50.0), ("bf16", 3e-2, 50.0)])
def test_png_golden_16bit(best_sd, golden, storage, tol, min_psnr):
    # bf16 storage cannot meet 5e-3 on these weights (SURVEY.md section 7: 1.1e-2..1.4e-2 from storage rounding
    # alone); fp16 is the 16-bit tier that holds north_star's bound.  Both must hold PSNR >= 50 dB.
    g = golden("lw_png.npz")
    net = _net(best_sd, storage=storage)
    for i in (1, 2):
        x = torch.from_numpy(g[f"x{i}_u8"].astype(np.float32) / 255.0)[None, None].cuda()
        with torch.no_grad():
            y = net(x)[0, 0].cpu().numpy()
        err = np.abs(y - g[f"y{i}"]).max()
        p = psnr(y, g[f"y{i}"])
        print(f"{storage} png{i}: max-abs {err:.3e} psnr {p:.1f} dB")
        assert err <= tol, f"{storage} png{i}: max-abs {err:.3e}"
        assert p >= min_psnr


def test_random_golden_and_layer_taps(best_sd, golden):
    g = golden("lw_rand.npz")
    net = _net(best_sd)
    x = _rand((2, 1, 64, 64), 0).cuda()
    with torch.no_grad():
        y = net(x).cpu().numpy()
    order = ["enc1.0", "enc1.3", "enc2.0", "enc2.3", "enc3.0", "enc3.3", "enc4.0", "enc4.3", "bottleneck.0",
             "bottleneck.3", "dec4.0", "dec4.3", "dec3.0", "dec3.3", "dec2.0", "dec2.3", "dec1.0", "dec1.3"]
    report = []
    for idx, name in enumerate(order):
        raw, _ = net.raw_activation(idx, 2, 64, 64)
        ref = g["tap/" + name]
        report.append((name, float(np.abs(raw.cpu().numpy() - ref).max()), float(np.abs(ref).max())))
    bad = [r for r in report if r[1] > 2e-4 * max(1.0, r[2])]
    assert not bad, f"raw conv outputs off: {bad} (all: {report})"
    assert np.abs(y - g["y_2x64x64_seed0"]).max() <= 1e-4


@pytest.mark.parametrize("shape,seed,key", [((1, 1, 96, 80), 1, "y_1x96x80_seed1"), ((3, 1, 16, 16), 2, "y_3x16x16_seed2")])
def test_odd_shapes(best_sd, golden, shape, seed, key):
    g = golden("lw_rand.npz")
    net = _net(best_sd)
    with torch.no_grad():
        y = net(_rand(shape, seed).cuda()).cpu().numpy()
    assert np.abs(y - g[key]).max() <= 1e-4


@pytest.mark.parametrize("shape,seed", [((1, 1, 96, 80), 1), ((3, 1, 16, 16), 2), ((2, 1, 528, 32), 7), ((2, 1, 48, 1040), 8)])
def test_odd_shapes_16bit_tensor_core_path(best_sd, shape, seed):
    """Partial tiles, images smaller than a tile, and very wide / tall images through the tensor-core kernels."""
    x = _rand(shape, seed)
    with torch.no_grad():
        ref = tpo.lightweight_forward(x, best_sd).numpy()
    net = _net(best_sd, storage="fp16")
    with torch.no_grad():
        y = net(x.cuda()).cpu().numpy()
        y1 = _net(best_sd, storage="fp16", path=1)(x.cuda()).cpu().numpy()   # generic kernels, same storage
    assert np.abs(y - ref).max() <= 5e-3, shape
    assert psnr(y, ref) >= 50.0
    assert np.abs(y - y1).max() <= 5e-3


def test_full_size_batch_row_and_checksum(best_sd, golden):
    g = golden("lw_rand.npz")
    net = _net(best_sd)
    x = _rand((2, 1, 512, 512), 0).cuda()
    with torch.no_grad():
        y = net(x)
    assert np.abs(y[:, 0, 255, :].cpu().numpy() - g["y_2x512x512_seed0_row255"]).max() <= 2e-4
    s = g["y_2x512x512_seed0_stats"]
    yd = y.double()
    assert abs(float(yd.sum()) - s[0]) <= 1e-5 * abs(s[0]) + 1.0
    assert abs(float((yd ** 2).sum()) - s[1]) <= 1e-4 * abs(s[1])
    # batched forward == per-sample forward (GroupNorm statistics are per sample; SURVEY section 8e)
    with torch.no_grad():
        y1 = net(x[1:2].contiguous())
    assert float((y1 - y[1:2]).abs().max()) <= 1e-5


def test_variants_match_reference(golden):
    g = golden("lw_variants.npz")
    for fs, hw in ((16, 64), (64, 32)):
        tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g[f"keys_fs{fs}"], g[f"shapes_fs{fs}"])}
        sd = {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=100 + fs).items()}
        net = _net(sd, features_start=fs)
        with torch.no_grad():
            y = net(_rand((2, 1, hw, hw), 5).cuda()).cpu().numpy()
        ref = g[f"y_fs{fs}_2x{hw}x{hw}_seed5"]
        err = np.abs(y - ref).max()
        assert err <= 2e-4 * max(1.0, np.abs(ref).max()), f"fs={fs}: {err:.3e}"
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys_fs12"], g["shapes_fs12"])}
    sd = {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=112).items()}
    net = _net(sd, in_channels=3, out_channels=2, num_groups=8, features_start=12)
    with torch.no_grad():
        y = net(_rand((2, 3, 32, 48), 6).cuda()).cpu().numpy()
    ref = g["y_fs12_in3_out2_2x32x48_seed6"]
    assert np.abs(y - ref).max() <= 2e-4 * max(1.0, np.abs(ref).max())


def test_against_oracle_random_batches(best_sd):
    net = _net(best_sd)
    for shape, seed in (((4, 1, 128, 128), 11), ((2, 1, 256, 64), 12), ((1, 1, 32, 528), 13)):
        x = _rand(shape, seed)
        with torch.no_grad():
            ref = tpo.lightweight_forward(x, best_sd).numpy()
            y = net(x.cuda()).cpu().numpy()
        assert np.abs(y - ref).max() <= 2e-4, shape


def test_shape_and_device_errors(best_sd):
    net = _net(best_sd)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="multiples of 16"):
            net(torch.zeros(1, 1, 500, 500, device="cuda"))
        with pytest.raises(RuntimeError, match="CUDA"):
            net(torch.zeros(1, 1, 16, 16))
        with pytest.raises(RuntimeError):
            net(torch.zeros(1, 2, 16, 16, device="cuda"))


def test_state_dict_roundtrip_and_param_update(best_sd):
    net = _net(best_sd)
    sd2 = net.state_dict()
    assert list(sd2.keys()) == list(best_sd.keys()) or set(sd2.keys()) == set(best_sd.keys())
    for k in best_sd:
        assert sd2[k].dtype == torch.float32 and tuple(sd2[k].shape) == tuple(best_sd[k].shape)
        assert torch.equal(sd2[k].cpu(), best_sd[k])
    x = _rand((1, 1, 32, 32), 3).cuda()
    with torch.no_grad():
        y0 = net(x).clone()
        net.output_conv.bias.add_(0.25)      # in-place update must invalidate the packed cache
        y1 = net(x)
    assert float((y1 - y0 - 0.25).abs().max()) <= 1e-6


def test_infer_host_matches_device_forward(best_sd):
    from image_enhancement_deglaring_b200.session import InferenceSession
    net = _net(best_sd)
    sess = InferenceSession(net, chunk=2)
    x = _rand((5, 1, 64, 64), 21)
    out = sess.run([sess.get_outputs()[0].name], {sess.get_inputs()[0].name: x.numpy()})[0]
    with torch.no_grad():
        y = net(x.cuda()).cpu().numpy()
    assert out.shape == (5, 1, 64, 64) and out.dtype == np.float32
    assert np.abs(out - y).max() <= 1e-6


def _quantise(y):
    """api/app.py:190-193: clip to [0, 1], scale by 255 in float32, truncate to uint8."""
    return (np.clip(y, 0, 1) * 255).astype(np.uint8)


@pytest.mark.parametrize("storage", ["fp32", "fp16"])
def test_u8_io_is_bit_identical_to_quantised_fp32_io(best_sd, storage):
    """SURVEY 8f1: uint8 in / uint8 out folded into the first / last kernel must equal the host-side
    `u.astype(float32) / 255.0` -> forward -> `(clip(y, 0, 1) * 255).astype(uint8)` of api/app.py:153-193 exactly."""
    net = _net(best_sd, storage=storage)
    rs = np.random.RandomState(5)
    for shape in [(3, 1, 64, 96), (2, 1, 48, 80), (1, 1, 512, 512)]:
        u = rs.randint(0, 256, size=shape).astype(np.uint8)
        u[0, 0, :4, :8] = np.array([0, 255, 1, 254, 127, 128, 2, 253], dtype=np.uint8)
        xf = torch.from_numpy(u.astype(np.float32) / 255.0).cuda()
        with torch.no_grad():
            want = _quantise(net(xf).cpu().numpy())
            got = net.forward_u8(torch.from_numpy(u).cuda()).cpu().numpy()
        assert got.dtype == np.uint8 and got.shape == shape
        assert np.array_equal(got, want), f"{storage} {shape}: {int((got != want).sum())} pixels differ"


def test_u8_png_golden_within_one_level(best_sd, golden):
    """The reference's /infer output image for the two shipped PNGs: fp32 storage differs from the quantised reference
    output only where 255*y sits within float noise of an integer (<= 1 level, a handful of pixels); fp16 storage <= 2 levels."""
    g = golden("lw_png.npz")
    for storage, max_levels, max_frac in [("fp32", 1, 1e-3), ("fp16", 2, 0.5)]:
        net = _net(best_sd, storage=storage)
        for i in (1, 2):
            want = _quantise(g[f"y{i}"])
            got = net.forward_u8(torch.from_numpy(g[f"x{i}_u8"])[None, None].cuda())[0, 0].cpu().numpy()
            d = np.abs(got.astype(np.int32) - want.astype(np.int32))
            assert d.max() <= max_levels, f"{storage} png{i}: {d.max()} levels"
            assert (d > 0).mean() <= max_frac, f"{storage} png{i}: {(d > 0).mean():.4f} of the pixels differ"


def test_u8_session_matches_device_forward(best_sd):
    from image_enhancement_deglaring_b200.session import InferenceSession
    net = _net(best_sd, storage="fp16")
    sess = InferenceSession(net, chunk=2)
    u = np.random.RandomState(6).randint(0, 256, size=(5, 1, 64, 64)).astype(np.uint8)
    out = sess.run_u8(u)
    want = net.forward_u8(torch.from_numpy(u).cuda()).cpu().numpy()
    assert out.dtype == np.uint8 and np.array_equal(out, want)
    with pytest.raises(RuntimeError):
        sess.run_u8(u.astype(np.float32))
    with pytest.raises(RuntimeError):
        net.forward_u8(torch.from_numpy(u))  # CPU tensor


def test_infer_host_many_chunks_two_compute_streams(best_sd):
    """dg_lw_infer_host alternates two compute streams / workspaces over the chunks: every chunk count parity."""
    from image_enhancement_deglaring_b200.session import InferenceSession
    net = _net(best_sd, storage="fp16")
    x = _rand((7, 1, 64, 64), 22)
    with torch.no_grad():
        y = net(x.cuda()).cpu().numpy()
    for chunk in (1, 2, 3, 7, 16):
        sess = InferenceSession(net, chunk=chunk)
        out = sess.run(["output"], {"input": x.numpy()})[0]
        assert np.array_equal(out, y), f"chunk {chunk}"


def test_submit_wait_pipeline_across_calls(best_sd):
    """dg_lw_infer_host_submit / _wait: several calls in flight share the chunk pipeline (slots are reused ACROSS calls), float and
    uint8, batch sizes that are not a multiple of the chunk, more calls than tickets, a geometry change that drains the pipeline --
    every result equals the device-resident forward of the same batch, and a blocking call may follow at once."""
    from image_enhancement_deglaring_b200.session import InferenceSession
    net = _net(best_sd, storage="fp16")
    sess = InferenceSession(net, chunk=2)
    xs = [_rand((n, 1, 64, 96), 40 + i) for i, n in enumerate((5, 7, 2, 9, 1, 6, 3, 8, 5, 4, 7))]      # 11 calls > 8 tickets
    with torch.no_grad():
        want = [net(x.cuda()).cpu() for x in xs]
    pins = [(x.pin_memory(), torch.empty_like(x).pin_memory()) for x in xs]
    tickets = [sess.submit(px, py, chunk=2) for px, py in pins]
    for t in reversed(tickets):          # any order; early tickets may already be retired
        sess.wait(t)
    for (px, py), w in zip(pins, want):
        assert torch.equal(py, w)
    # uint8 twin, two in flight as bench.py does, then another image size (drains), then the blocking call
    us = [(torch.rand(6, 1, 64, 96, generator=torch.Generator().manual_seed(60 + i)) * 255).to(torch.uint8) for i in range(4)]
    pins8 = [(u.pin_memory(), torch.empty_like(u).pin_memory()) for u in us]
    pending = []
    for px, py in pins8:
        if len(pending) == 2:
            sess.wait(pending.pop(0))
        pending.append(sess.submit(px, py, chunk=4))
    big = _rand((3, 1, 128, 64), 77)
    pbig = (big.pin_memory(), torch.empty_like(big).pin_memory())
    pending.append(sess.submit(*pbig, chunk=4))
    for t in pending:
        sess.wait(t)
    for (px, py), u in zip(pins8, us):
        assert torch.equal(py, net.forward_u8(u.cuda()).cpu())
    with torch.no_grad():
        assert torch.equal(pbig[1], net(big.cuda()).cpu())
    out = sess.run(["output"], {"input": xs[0].numpy()})[0]
    assert np.array_equal(out, want[0].numpy())
    with pytest.raises(RuntimeError):
        sess.wait(10 ** 6)                # unknown ticket
    with pytest.raises(RuntimeError):
        sess.submit(pins[0][0], pins8[0][1])   # mixed dtypes


def test_tiled_high_resolution_equals_per_tile_forward(best_sd):
    """BASELINE.json configs[2] (definition A of SURVEY 8e): a 1024x1536 image as six independent 512x512 tiles equals the
    module applied to each tile on its own -- float and uint8 entry points."""
    from image_enhancement_deglaring_b200.tiling import infer_tiled, split_tiles
    net = _net(best_sd, storage="fp16")
    img = _rand((1024, 1536), 31).cuda()
    with torch.no_grad():
        full = infer_tiled(net, img, tile=512, batch=4)
        tiles, grid = split_tiles(img, 512)
        assert grid == (2, 3)
        for t in (0, 4):
            r, c = divmod(t, 3)
            one = net(tiles[t:t + 1])[0]
            assert torch.equal(full[:, 512 * r:512 * (r + 1), 512 * c:512 * (c + 1)], one)
        u = (img * 255).to(torch.uint8)
        full8 = infer_tiled(net.forward_u8, u, tile=512)
        assert full8.dtype == torch.uint8 and torch.equal(full8[:, :512, 1024:], net.forward_u8(split_tiles(u, 512)[0][2:3])[0])


def test_two_stream_batch_split_is_bit_identical(best_sd):
    """dg_lw_forward runs the halves of a large batch on two private streams (dg_set_batch_split): same bits as one stream,
    for the float and the uint8 entry points, odd batch included."""
    from image_enhancement_deglaring_b200 import _lib
    lib = _lib.load()
    net = _net(best_sd, storage="fp16")
    x = _rand((5, 1, 64, 96), 41).cuda()
    u = (x * 255).to(torch.uint8)
    old = lib.dg_set_batch_split(0)
    try:
        with torch.no_grad():
            y1, u1 = net(x).clone(), net.forward_u8(u).clone()
        assert lib.dg_set_batch_split(2) == 0
        with torch.no_grad():
            y2, u2 = net(x).clone(), net.forward_u8(u).clone()
            for _ in range(3):   # back-to-back calls reuse the fork / join events
                y3 = net(x)
        assert torch.equal(y1, y2) and torch.equal(u1, u2) and torch.equal(y1, y3)
    finally:
        lib.dg_set_batch_split(old)
    assert old == 16


def test_4096_square_image_as_64_tiles(best_sd):
    """BASELINE.json configs[2] at its full size: a 4096x4096 grayscale image = 64 tiles of 512x512 = one batch-64 forward
    (run as four batches of 16 here).  Every checked output tile equals the module applied to that tile alone, the marked tile included."""
    from image_enhancement_deglaring_b200.tiling import infer_tiled
    net = _net(best_sd, storage="fp16")
    img = _rand((4096, 4096), 51)
    img[3 * 512:4 * 512, 5 * 512:6 * 512] = 0.25          # tile (row 3, col 5) = tile index 29: constant input
    img = img.cuda()
    with torch.no_grad():
        out = infer_tiled(net, img, tile=512, batch=16)
        assert out.shape == (1, 4096, 4096)
        for r, c in ((0, 0), (3, 5), (7, 7)):
            alone = net(img[None, None, r * 512:(r + 1) * 512, c * 512:(c + 1) * 512])[0]
            assert torch.equal(out[:, r * 512:(r + 1) * 512, c * 512:(c + 1) * 512], alone), (r, c)
        # the marked (constant-input) tile is not confused with its random neighbours
        assert not torch.equal(out[:, 3 * 512:4 * 512, 5 * 512:6 * 512], out[:, 3 * 512:4 * 512, 4 * 512:5 * 512])


def test_whole_image_4096_exact_groupnorm_on_one_gpu(best_sd):
    """SURVEY 8e "definition B": the network applied to the WHOLE 4096x4096 image (GroupNorm statistics over the full image, receptive
    fields across what would be tile borders) -- one dg_lw_forward call with N = 1, H = W = 4096 (2.1 GB of fp16 workspace, every
    kernel on image-wide grids, the tcgen05 kernel on column strips) against the oracle; and it differs from the tiled result."""
    from image_enhancement_deglaring_b200.tiling import infer_tiled
    x = _rand((1, 1, 4096, 4096), 91)
    torch.set_num_threads(os.cpu_count() or 1)
    with torch.no_grad():
        ref = tpo.lightweight_forward(x, best_sd)
    for storage, tol in (("fp16", 5e-3), ("fp32", 2e-4)):
        net = _net(best_sd, storage=storage)
        with torch.no_grad():
            y = net(x.cuda())
            err = float((y.cpu() - ref).abs().max())
            assert err <= tol, f"{storage}: whole-image max-abs {err:.3e}"
            if storage == "fp16":
                assert psnr(y.cpu().numpy(), ref.numpy()) >= 50.0
                tiled = infer_tiled(net, x[0, 0].cuda(), tile=512, batch=16)
                assert float((tiled - y[0]).abs().max()) > 1e-3          # tiling is a different function (definition A)
        del net, y
        torch.cuda.empty_cache()


def test_headline_config_batch64_512_fp16_matches_oracle(best_sd):
    """The configuration bench.py quotes -- batch 64 x 1x512x512, fp16 storage, default two-stream split, every persistent kernel on
    full grids -- against the oracle on the same seeded inputs: max-abs <= 5e-3 and PSNR >= 50 dB per image (north_star)."""
    net = _net(best_sd, storage="fp16")
    x = _rand((64, 1, 512, 512), 77)
    with torch.no_grad():
        y = net(x.cuda()).cpu()
        y2 = net(x.cuda()).cpu()
    assert torch.equal(y, y2)                       # run-to-run reproducible
    torch.set_num_threads(os.cpu_count() or 1)
    worst, worst_psnr = 0.0, 1e9
    with torch.no_grad():
        for i in range(0, 64, 8):
            ref = tpo.lightweight_forward(x[i:i + 8], best_sd)
            for j in range(8):
                a, b = y[i + j, 0].numpy(), ref[j, 0].numpy()
                worst = max(worst, float(np.abs(a - b).max()))
                worst_psnr = min(worst_psnr, psnr(a, b))
    print(f"batch 64 fp16: worst max-abs {worst:.3e}, worst PSNR {worst_psnr:.1f} dB")
    assert worst <= 5e-3, worst
    assert worst_psnr >= 50.0, worst_psnr
    # ... and the batch is bit-identical to its images run alone (GroupNorm is per sample; statistics are batch-invariant)
    with torch.no_grad():
        for i in (0, 31, 32, 63):
            assert torch.equal(net(x[i:i + 1].cuda()).cpu(), y[i:i + 1]), i


def test_session_sees_weight_update_immediately(best_sd):
    """ADVICE r1: the host pipeline runs on library-private streams; packing kernels of freshly changed weights are enqueued on the
    caller's stream.  dg_lw_infer_host orders its streams after the caller's, so run() right after an in-place update is correct."""
    from image_enhancement_deglaring_b200.session import InferenceSession
    net = _net(best_sd, storage="fp16")
    sess = InferenceSession(net, chunk=4)
    x = _rand((8, 1, 64, 96), 5).numpy()
    for step in range(4):
        with torch.no_grad():
            for p in net.parameters():
                p.mul_(1.0 + 0.01 * (step + 1))      # bumps the version counters -> re-pack on the next call
        out = sess.run(["output"], {"input": x})[0]
        with torch.no_grad():
            want = net(torch.from_numpy(x).cuda()).cpu().numpy()
        assert np.array_equal(out, want), step
