"""Pin the CPU oracle against the golden vectors produced by the reference itself
(tests/golden/make_golden.py).  CPU only."""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import numpy_unet as npo
from oracle import torch_unet as tpo

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from make_golden import det_state_dict, TRAIN_LR, TRAIN_WD  # noqa: E402


def _rand(shape, seed):
    return torch.rand(*shape, generator=torch.Generator().manual_seed(seed))


def test_state_dict_is_the_published_model(best_sd):
    # README.md:10-11 -- 486,409 parameters, 1.86 MB
    assert len(best_sd) == 64
    assert sum(v.numel() for v in best_sd.values()) == 486409
    assert best_sd["enc1.0.weight"].shape == (8, 1, 3, 3)
    assert best_sd["upconv4.weight"].shape == (128, 64, 2, 2)
    assert best_sd["output_conv.weight"].shape == (1, 8, 1, 1)


def test_torch_oracle_matches_reference_png(best_sd, golden):
    g = golden("lw_png.npz")
    for i in (1, 2):
        x = torch.from_numpy(g[f"x{i}_u8"].astype(np.float32) / 255.0)[None, None]
        with torch.no_grad():
            y = tpo.lightweight_forward(x, best_sd)[0, 0].numpy()
        assert np.abs(y - g[f"y{i}"]).max() <= 1e-5


def test_torch_oracle_matches_reference_random_and_taps(best_sd, golden):
    g = golden("lw_rand.npz")
    taps = {}
    with torch.no_grad():
        y = tpo.lightweight_forward(_rand((2, 1, 64, 64), 0), best_sd, taps=taps)
    assert np.abs(y.numpy() - g["y_2x64x64_seed0"]).max() <= 1e-5
    names = [k for k in g.files if k.startswith("tap/")]
    assert len(names) == 23  # 18 conv3x3 + 4 convT + head
    for k in names:
        key = k[4:]
        if key == "output_conv":
            continue
        ref = g[k]
        assert np.abs(taps[key].numpy() - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max()), key
    with torch.no_grad():
        assert np.abs(tpo.lightweight_forward(_rand((1, 1, 96, 80), 1), best_sd).numpy()
                      - g["y_1x96x80_seed1"]).max() <= 1e-5
        assert np.abs(tpo.lightweight_forward(_rand((3, 1, 16, 16), 2), best_sd).numpy()
                      - g["y_3x16x16_seed2"]).max() <= 1e-5


def test_numpy_oracle_matches_reference(best_sd, golden):
    g = golden("lw_rand.npz")
    sd = {k: v.numpy() for k, v in best_sd.items()}
    x = _rand((2, 1, 64, 64), 0).numpy()
    y32 = npo.lightweight_unet_forward(x, sd)
    assert np.abs(y32 - g["y_2x64x64_seed0"]).max() <= 2e-5
    y64 = npo.lightweight_unet_forward(x.astype(np.float64), sd)
    assert np.abs(y64 - g["y_2x64x64_seed0"]).max() <= 2e-5
    x = _rand((3, 1, 16, 16), 2).numpy()
    assert np.abs(npo.lightweight_unet_forward(x, sd) - g["y_3x16x16_seed2"]).max() <= 2e-5


def test_numpy_oracle_full_size_row(best_sd, golden):
    g = golden("lw_rand.npz")
    sd = {k: v.numpy() for k, v in best_sd.items()}
    x = _rand((2, 1, 512, 512), 0)[:1].numpy()
    y = npo.lightweight_unet_forward(x, sd)
    assert np.abs(y[0, 0, 255] - g["y_2x512x512_seed0_row255"][0]).max() <= 2e-5


def test_oracles_match_reference_variants(golden):
    g = golden("lw_variants.npz")
    for fs, hw in ((16, 64), (64, 32)):
        tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g[f"keys_fs{fs}"], g[f"shapes_fs{fs}"])}
        sd = det_state_dict(tmpl, seed=100 + fs)
        x = _rand((2, 1, hw, hw), 5)
        with torch.no_grad():
            y = tpo.lightweight_forward(x, {k: torch.from_numpy(v) for k, v in sd.items()}).numpy()
        ref = g[f"y_fs{fs}_2x{hw}x{hw}_seed5"]
        assert np.abs(y - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys_fs12"], g["shapes_fs12"])}
    sd = det_state_dict(tmpl, seed=112)
    x = _rand((2, 3, 32, 48), 6)
    ref = g["y_fs12_in3_out2_2x32x48_seed6"]
    with torch.no_grad():
        y = tpo.lightweight_forward(x, {k: torch.from_numpy(v) for k, v in sd.items()}).numpy()
    assert np.abs(y - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())
    y = npo.lightweight_unet_forward(x.numpy(), sd)
    assert np.abs(y - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())
    # divisor search gives 6 groups for 12 channels, 8 for 24/48/96/192
    assert [npo._groups_lightweight(c, 8) for c in (12, 24, 48, 96, 192)] == [6, 8, 8, 8, 8]
    assert list(g["gn_groups_fs12"][:4]) == [6, 6, 8, 8]


def test_oracles_match_reference_optimized(golden):
    g = golden("opt_rand.npz")
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    assert len(tmpl) == 76 and int(g["n_params"]) == 2163969
    sd = det_state_dict(tmpl, seed=1234)
    assert abs(sum(float(np.abs(v).astype(np.float64).sum()) for v in sd.values()) - float(g["wsum"])) < 1e-6 * float(g["wsum"])
    tsd = {k: torch.from_numpy(v) for k, v in sd.items()}
    for shape, seed, key in (((2, 1, 64, 64), 3, "y_2x64x64_seed3"), ((1, 1, 48, 80), 4, "y_1x48x80_seed4")):
        x = _rand(shape, seed)
        ref = g[key]
        with torch.no_grad():
            y = tpo.optimized_forward(x, tsd).numpy()
        assert np.abs(y - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())
        y = npo.optimized_unet_forward(x.numpy(), sd)
        assert np.abs(y - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max())


def test_train_step_oracle_matches_reference(best_sd, golden):
    g = golden("lw_train.npz")
    x, t = _rand((2, 1, 64, 64), 0), _rand((2, 1, 64, 64), 1)
    r = tpo.train_step(best_sd, x, t, lr=TRAIN_LR, weight_decay=TRAIN_WD, max_norm=1.0)
    assert abs(r["loss"] - float(g["loss"])) <= 1e-6
    assert abs(r["total_norm"] - float(g["total_norm"])) <= 1e-4
    for k in best_sd:
        gr = g["grad/" + k]
        assert np.abs(r["grads"][k].numpy() - gr).max() <= 1e-5 + 1e-4 * np.abs(gr).max(), k
        assert np.abs(r["new_params"][k].numpy() - g["new/" + k]).max() <= 2e-6, k


def _opt_sd(golden):
    g = golden("opt_rand.npz")
    tmpl = {k: tuple(int(s) for s in sh.split(",")) for k, sh in zip(g["keys"], g["shapes"])}
    return {k: torch.from_numpy(v) for k, v in det_state_dict(tmpl, seed=1234).items()}


def test_optimized_train_step_oracle_matches_reference(golden):
    """tests/golden/make_opt_train_golden.py: the reference OptimizedUNet through optimized_train.py:220-233 (L1, backward, clip 1.0,
    AdamW) and through backward(gy) with an explicit output gradient."""
    g = golden("opt_train.npz")
    sd = _opt_sd(golden)
    x, t = _rand((2, 1, 64, 64), 7), _rand((2, 1, 64, 64), 8)
    r = tpo.train_step(sd, x, t, forward=tpo.optimized_forward, lr=TRAIN_LR, weight_decay=TRAIN_WD, max_norm=1.0)
    assert abs(r["loss"] - float(g["loss"])) <= 2e-6 * max(1.0, abs(float(g["loss"])))
    assert np.abs(r["out"].numpy() - g["y"]).max() <= 1e-4 * max(1.0, np.abs(g["y"]).max())
    assert abs(r["total_norm"] - float(g["total_norm"])) <= 1e-4 * float(g["total_norm"])
    for k in sd:
        got = r["grads"][k].numpy().reshape(-1)
        norm = float(g["gnorm/" + k])
        assert abs(np.sqrt((got.astype(np.float64) ** 2).sum()) - norm) <= 1e-4 * norm + 1e-7, k
        assert np.abs(got[:32] - g["ghead/" + k]).max() <= 1e-5 + 1e-3 * np.abs(g["ghead/" + k]).max(), k
        if "grad/" + k in g.files:
            ref = g["grad/" + k].reshape(-1)
            assert np.abs(got - ref).max() <= 1e-5 + 1e-3 * np.abs(ref).max(), k
        new = r["new_params"][k].numpy().reshape(-1)
        assert np.abs(new[:32] - g["newhead/" + k]).max() <= 2e-5, k
    # explicit output gradient
    gy = torch.randn(2, 1, 64, 64, generator=torch.Generator().manual_seed(9)) / (2 * 64 * 64)
    params = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
    grads = torch.autograd.grad((tpo.optimized_forward(x, params) * gy).sum(), list(params.values()))
    for k, gr in zip(params, grads):
        got = gr.numpy().reshape(-1)
        norm = float(g["gy_gnorm/" + k])
        assert abs(np.sqrt((got.astype(np.float64) ** 2).sum()) - norm) <= 1e-4 * norm + 1e-9, k
        assert np.abs(got[:32] - g["gy_ghead/" + k]).max() <= 1e-9 + 1e-3 * np.abs(g["gy_ghead/" + k]).max(), k


# ---- second oracle: the exported ONNX graph (what api/app.py:84,171 and evaluate.py:95,122 execute through onnxruntime) ----------
def test_onnx_artefact_interpreter_matches_reference_goldens(best_sd, golden, tmp_path):
    """oracle/onnx_interp.py evaluates the exported graph (opset 11, 229 nodes, eleven operator types) with the ONNX operator
    semantics: it must land on the outputs the reference MODULE produced (golden vectors), i.e. artefact == module == oracle.
    The graph is tests/golden/make_onnx_golden.py's export of the reference module, stored without its weights; the initializers
    are re-attached from weights/best_model.pth, each checked against the sha256 the export recorded."""
    import hashlib
    from oracle.onnx_interp import OnnxGraph
    store = golden("onnx_graph.npz")
    path = tmp_path / "best_model.onnx"
    path.write_bytes(store["model"].tobytes())
    g = OnnxGraph(str(path))
    assert not g.inits
    for name, key, shape, digest in zip(store["init_names"], store["init_keys"], store["init_shapes"], store["init_sha256"]):
        v = best_sd[key].numpy().reshape([int(s) for s in shape.split(",")])
        assert hashlib.sha256(v.astype("<f4").tobytes()).hexdigest() == digest, name
        g.inits[name] = v
    assert g.opset == 11 and g.inputs == ["input"] and g.outputs == ["output"] and len(g.nodes) == 229
    assert g.op_types() == ["Add", "AveragePool", "Concat", "Constant", "Conv", "ConvTranspose", "InstanceNormalization", "Mul",
                            "Reshape", "Shape", "Sigmoid"]
    png = golden("lw_png.npz")
    for i in (1, 2):   # the two sample images through the /infer preprocessing (api/app.py:136-157)
        x = png[f"x{i}_u8"].astype(np.float32)[None, None] / 255.0
        assert np.abs(g.run(x)[0, 0] - png[f"y{i}"]).max() <= 1e-5
    rnd = golden("lw_rand.npz")
    assert np.abs(g.run(_rand((2, 1, 64, 64), 0).numpy()) - rnd["y_2x64x64_seed0"]).max() <= 1e-5
    assert np.abs(g.run(_rand((1, 1, 96, 80), 1).numpy()) - rnd["y_1x96x80_seed1"]).max() <= 1e-5      # dynamic axes
    # every raw conv / ConvTranspose output of the graph against the reference module's forward hooks
    taps = {}
    g.run(_rand((2, 1, 64, 64), 0).numpy(), taps=taps)
    assert len(taps) == 23
    for name, v in taps.items():     # "/enc1/enc1.0/Conv_output_0" -> "enc1.0";  "/upconv4/ConvTranspose_output_0" -> "upconv4"
        parts = name.strip("/").split("/")
        key = parts[-2] if len(parts) >= 2 else parts[0]
        key = "output_conv" if name == "output" else key
        ref = rnd["tap/" + key]        # all 23: 18 conv3x3, 4 ConvTranspose, the head
        assert np.abs(v.numpy() - ref).max() <= 1e-4 * max(1.0, np.abs(ref).max()), key
    # and against the restated oracle on an input neither golden file holds
    x = _rand((3, 1, 48, 32), 77)
    with torch.no_grad():
        want = tpo.lightweight_forward(x, best_sd).numpy()
    assert np.abs(g.run(x.numpy()) - want).max() <= 1e-5
    # the initializers are the 486,409 weights of weights/best_model.pth, every state_dict entry exactly once
    named = {k: v for k, v in g.inits.items() if not k.startswith("onnx::")}
    assert sum(v.size for v in g.inits.values() if v.dtype == np.float32) == 486409
    assert sorted(store["init_keys"]) == sorted(best_sd)
    for k, v in named.items():
        assert np.array_equal(v, best_sd[k].numpy()), k


def test_l1_grad_restatement():
    o = np.array([[0.2, 0.5], [0.7, 0.1]])
    t = np.array([[0.5, 0.5], [0.1, 0.4]])
    assert npo.l1_loss(o, t) == pytest.approx(0.3)
    assert np.array_equal(npo.l1_loss_grad(o, t), np.array([[-0.25, 0.0], [0.25, -0.25]]))


# ---- validation metrics oracle (SURVEY 8f4; skimage is absent: the restatement is checked against a direct evaluation) ----
def test_metrics_oracle_self_consistency():
    from oracle import metrics_np as M
    rs = np.random.RandomState(3)
    a = rs.rand(24, 31).astype(np.float32)
    b = np.clip(a + 0.1 * rs.standard_normal(a.shape), 0, 1).astype(np.float32)
    assert abs(M.ssim(a, a) - 1.0) < 1e-6
    assert abs(M.ssim(a, b) - M.ssim_bruteforce(a, b)) < 2e-5          # float32 filter outputs vs float64 windows
    assert abs(M.ssim(a, b) - M.ssim(b, a)) < 1e-6                      # symmetric
    mse = float(np.mean((a.astype(np.float64) - b.astype(np.float64)) ** 2))
    assert abs(M.psnr(a, b) - 10 * np.log10(1.0 / mse)) < 1e-9
    flat = np.full((16, 16), 0.5, np.float32)
    assert abs(M.ssim(flat, flat * 0.5) - (2 * 0.5 * 0.25 + 1e-4) / (0.25 + 0.0625 + 1e-4)) < 1e-6   # luminance term only
