"""CPU-only tests: the C-ABI library loads and exports every declared symbol, the nn.Module surface matches the
reference's state_dict contract, errors are loud without a GPU, and the multi-rank host logic works over gloo."""
import os
import re
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    from image_enhancement_deglaring_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "deglare.h")).read()
    declared = set(re.findall(r"\b(dg_[a-z0-9_]+)\s*\(", hdr))
    assert {"dg_conv3x3_fused", "dg_head1x1", "dg_lw_forward", "dg_lw_infer_host"} <= declared
    lib = _lib.load()
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/deglare.h but not exported"
    assert declared == set(_lib.SYMBOLS), (declared ^ set(_lib.SYMBOLS))
    assert lib.dg_version() >= 100
    # nothing may launch without a GPU; the counter is per process and GPU tests may already have run in this one, so it is read
    # in a fresh process that sees no device
    import subprocess
    out = subprocess.run([sys.executable, "-c", "from image_enhancement_deglaring_b200 import _lib; print(_lib.load().dg_launch_count())"],
                         cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    assert int(out.stdout.split()[-1]) == 0


def test_struct_layouts_match_header_sizes(tmp_path):
    """The ctypes mirrors must have the size the C compiler gives the structs of include/deglare.h (gcc compiles the header as C)."""
    import ctypes as C
    import subprocess
    from image_enhancement_deglaring_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text('#include "deglare.h"\n#include <stdio.h>\nint main(void){printf("%zu %zu %zu %zu\\n", sizeof(dg_src), '
                   'sizeof(dg_conv3x3_args), sizeof(dg_head_args), sizeof(dg_lw_params)); return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(v) for v in subprocess.check_output([str(exe)], text=True).split()]
    assert sizes == [C.sizeof(_lib.DgSrc), C.sizeof(_lib.DgConv3x3Args), C.sizeof(_lib.DgHeadArgs), C.sizeof(_lib.DgLwParams)]
    assert C.sizeof(_lib.DgSrc) == 9 * 8 + 6 * 4


_REMOVED_PATH_BITS_PROBE = r"""
import ctypes as C, json
from image_enhancement_deglaring_b200 import _lib
lib = _lib.load()
buf = (C.c_float * 4096)()   # placeholder for every pointer: none may be dereferenced
res = {}
for path in (4, 8, 16, 32, 64, 2048, 0, 2 | 128):
    p = _lib.DgLwParams()
    p.in_channels, p.out_channels, p.features_start, p.dtype, p.path = 1, 1, 8, _lib.DG_F16, path
    rc = lib.dg_lw_workspace_bytes(C.byref(p), 1, 16, 16, C.byref(C.c_size_t(0)))
    res[path] = [rc, lib.dg_last_error_string().decode()]
    if path & 0x87c:
        a = _lib.DgConv3x3Args()
        a.nsrc, a.dtype, a.N, a.H, a.W, a.cout, a.eps, a.path = 1, _lib.DG_F16, 1, 16, 16, 8, 1e-5, path
        a.weight = a.out = a.out_stats = C.addressof(buf)
        a.src[0].raw, a.src[0].channels, a.src[0].groups, a.src[0].xform = C.addressof(buf), 8, 1, _lib.DG_X_SAME
        res[path] += [lib.dg_conv3x3_fused(C.byref(a), None), lib.dg_last_error_string().decode()]
comp = {}
for cl, cu in ((16, 8), (32, 16), (64, 32), (128, 64)):
    n = C.c_size_t(0)
    rc = lib.dg_dec_composite_bytes(cl, cu, C.byref(n))
    comp[f"{cl},{cu}"] = [rc, n.value, lib.dg_last_error_string().decode() if rc else ""]
print(json.dumps({"path": res, "comp": comp}))
"""


def test_removed_path_bits_are_rejected():
    """Path bits 2-6 and 11 no longer select anything: dg_conv3x3_fused and the dg_lw_* planner return 2 and name the bit, before
    any CUDA call -- run in a process that sees no CUDA device, where a call that reached the runtime would fail differently.  With
    bit 11 went the tcgen05 decoder mode's composite packing: dg_dec_composite_bytes covers (16, 8) only."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, "-c", _REMOVED_PATH_BITS_PROBE], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    probe = json.loads(out.stdout.splitlines()[-1])
    res = {int(k): v for k, v in probe["path"].items()}
    for bit in (2, 3, 4, 5, 6, 11):
        ws_rc, ws_err, conv_rc, conv_err = res[1 << bit]
        assert conv_rc == 2 and f"path {1 << bit} sets bit {bit}," in conv_err, (bit, conv_rc, conv_err)
        assert ws_rc == 2 and f"path {1 << bit} sets bit {bit}," in ws_err, (bit, ws_rc, ws_err)
    assert res[0][0] == 0 and res[2 | 128][0] == 0, res   # the surviving bits still plan a workspace
    comp = probe["comp"]
    assert comp["16,8"][0] == 0 and comp["16,8"][1] > 0, comp
    for pair in ("32,16", "64,32", "128,64"):
        assert comp[pair][0] == 3 and "(16, 8)" in comp[pair][2], (pair, comp[pair])


def test_module_surface_matches_reference_contract(best_sd, golden):
    import image_enhancement_deglaring_b200 as dg
    net = dg.LightweightUNet()
    assert dg.count_parameters(net) == 486409                     # README.md:10
    assert abs(dg.get_model_size_mb(net) - 1.8555) < 1e-3         # README.md:11
    assert list(net.state_dict().keys()) == [k for k in net.state_dict()]
    assert set(net.state_dict().keys()) == set(best_sd.keys())
    res = net.load_state_dict(best_sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    for k, v in net.state_dict().items():
        assert v.dtype == torch.float32 and tuple(v.shape) == tuple(best_sd[k].shape)
    # constructor arguments of src/model.py:14, including the group-divisor search for odd widths
    g = golden("lw_variants.npz")
    odd = dg.LightweightUNet(in_channels=3, out_channels=2, num_groups=8, features_start=12)
    assert list(odd.state_dict().keys()) == list(g["keys_fs12"])
    assert [",".join(map(str, v.shape)) for v in odd.state_dict().values()] == list(g["shapes_fs12"])
    assert [m.num_groups for m in odd.modules() if isinstance(m, torch.nn.GroupNorm)] == list(g["gn_groups_fs12"])
    assert "GroupNorm(8, 8" in str(net) and "ConvTranspose2d(128, 64" in str(net)


def test_optimized_surface_matches_reference_contract(golden):
    import image_enhancement_deglaring_b200 as dg
    g = golden("opt_rand.npz")
    net = dg.OptimizedUNet()
    assert list(net.state_dict().keys()) == list(g["keys"])                       # 76 keys, same order
    assert [",".join(map(str, v.shape)) for v in net.state_dict().values()] == list(g["shapes"])
    assert dg.count_parameters(net) == int(g["n_params"]) == 2163969
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="CUDA"):
            net(torch.zeros(1, 1, 16, 16))


def test_no_cpu_fallback():
    import image_enhancement_deglaring_b200 as dg
    net = dg.LightweightUNet()
    with torch.no_grad():
        with pytest.raises(RuntimeError, match="CUDA"):
            net(torch.zeros(1, 1, 16, 16))
    from image_enhancement_deglaring_b200.session import InferenceSession
    with pytest.raises(RuntimeError, match="CUDA"):
        InferenceSession(net)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "image_enhancement_deglaring_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), fn
    # outside tests/ and oracle/ itself, only bench.py (cpu_baseline / --impl reference) and __graft_entry__.smoke() may use it
    allowed = {"bench.py", "__graft_entry__.py"}
    for d, _, files in os.walk(ROOT):
        rel = os.path.relpath(d, ROOT)
        if rel.split(os.sep)[0] in ("tests", "oracle", ".git", "gpurun_out", "baseline") or "__pycache__" in rel:
            continue
        for fn in files:
            if fn.endswith(".py") and os.path.join(rel, fn).lstrip("./") not in allowed:
                src = open(os.path.join(d, fn)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), os.path.join(rel, fn)


def test_shard_range_partitions_exactly():
    from image_enhancement_deglaring_b200.parallel import shard_range
    for n in (0, 1, 7, 64, 65):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        shard_range(4, 2, 2)


def _ddp_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from image_enhancement_deglaring_b200.parallel import FlatGradBucket, shard_range
    torch.manual_seed(0)
    lin = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 1))
    bucket = FlatGradBucket(lin.parameters())
    x = torch.arange(40, dtype=torch.float32).reshape(8, 5) / 40.0
    lo, hi = shard_range(8, rank, world)
    bucket.zero_()
    lin(x[lo:hi]).abs().mean().backward()
    # every .grad must still alias the flat bucket after backward
    off = 0
    for p in bucket.params:
        assert p.grad.data_ptr() == bucket.flat[off:off + p.numel()].data_ptr()
        off += p.numel()
    flat = bucket.allreduce_mean().clone()
    if rank == 0:
        torch.save(flat, out)
    dist.destroy_process_group()


def test_gradient_bucket_allreduce_world2(tmp_path):
    port = 29500 + (os.getpid() % 2000)
    out = str(tmp_path / "flat.pt")
    mp.spawn(_ddp_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out)
    torch.manual_seed(0)
    lin = torch.nn.Sequential(torch.nn.Linear(5, 3), torch.nn.Linear(3, 1))
    x = torch.arange(40, dtype=torch.float32).reshape(8, 5) / 40.0
    # mean over equal shards of per-shard mean losses == global mean loss
    lin(x).abs().mean().backward()
    want = torch.cat([p.grad.flatten() for p in lin.parameters()])
    assert torch.allclose(got, want, atol=1e-6)


# ---- 4096^2-style tiling (BASELINE.json configs[2]): tiles are independent units sharded over ranks --------------
def _fake_forward(t):
    """Stands in for the CUDA module on CPU: per-tile, position-dependent, so a misplaced tile cannot cancel out."""
    ramp = torch.arange(t.shape[-1], dtype=t.dtype)
    return t * 2.0 + ramp + t.mean(dim=(1, 2, 3), keepdim=True)


def test_tiles_roundtrip_and_order():
    from image_enhancement_deglaring_b200.tiling import infer_tiled, merge_tiles, split_tiles
    img = torch.arange(3 * 8 * 12, dtype=torch.float32).reshape(3, 8, 12)
    tiles, grid = split_tiles(img, tile=4)
    assert tiles.shape == (6, 3, 4, 4) and grid == (2, 3)
    assert torch.equal(tiles[4], img[:, 4:8, 4:8])            # row-major: tile 4 = (row 1, col 1)
    assert torch.equal(merge_tiles(tiles, grid), img)
    single = infer_tiled(_fake_forward, img[0], tile=4, batch=4)  # 2-D input -> one channel; 6 tiles in calls of 4 + 2
    want = merge_tiles(_fake_forward(split_tiles(img[0], 4)[0]), grid)
    assert torch.equal(single, want)
    with pytest.raises(RuntimeError):
        split_tiles(torch.zeros(10, 12), tile=4)


def _fake_forward_2ch(t):
    f = t.float() / 255.0
    return torch.cat((f, 1.0 - f), 1)


def _tile_worker(rank, world, port, out):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from image_enhancement_deglaring_b200.tiling import infer_tiled
    res = {}
    for name, (h, w) in {"even": (8, 16), "ragged": (12, 4), "fewer_tiles_than_ranks": (4, 4)}.items():
        img = torch.arange(h * w, dtype=torch.float32).reshape(h, w) / 7.0
        res[name] = infer_tiled(_fake_forward, img, tile=4, rank=rank, world=world)
        part, span, _ = infer_tiled(_fake_forward, img, tile=4, rank=rank, world=world, gather=False)
        assert part.shape[0] == span[1] - span[0]
    # more ranks than tiles AND a forward that changes dtype and channel count (uint8 in -> 2 float channels out): the empty
    # shard must take the OUTPUT's shape / dtype or all_gather mismatches across ranks
    u8 = (torch.arange(16, dtype=torch.float32).reshape(4, 4)).to(torch.uint8)
    res["u8_to_2ch_float"] = infer_tiled(_fake_forward_2ch, u8, tile=4, rank=rank, world=world)
    res["u8_to_2ch_float_declared"] = infer_tiled(_fake_forward_2ch, u8, tile=4, rank=rank, world=world, out_channels=2,
                                                  out_dtype=torch.float32)
    # data-parallel gradient exchange: mean over ranks of the flat bucket (train.sync_gradients; gloo has no AVG -> sum + scale)
    from image_enhancement_deglaring_b200.train import sync_gradients
    flat = torch.arange(10, dtype=torch.float32) * (rank + 1)
    res["sync"] = sync_gradients(flat.clone())
    res["nosync"] = sync_gradients(flat.clone(), enabled=False)
    torch.save(res, f"{out}.{rank}")
    dist.destroy_process_group()


def test_tiled_inference_sharded_world2(tmp_path):
    from image_enhancement_deglaring_b200.tiling import infer_tiled
    port = 31500 + (os.getpid() % 2000)
    out = str(tmp_path / "tiles.pt")
    mp.spawn(_tile_worker, args=(2, port, out), nprocs=2, join=True)
    r0, r1 = torch.load(out + ".0"), torch.load(out + ".1")
    for name, (h, w) in {"even": (8, 16), "ragged": (12, 4), "fewer_tiles_than_ranks": (4, 4)}.items():
        img = torch.arange(h * w, dtype=torch.float32).reshape(h, w) / 7.0
        want = infer_tiled(_fake_forward, img, tile=4)
        assert torch.equal(r0[name], want) and torch.equal(r1[name], want), name
    u8 = (torch.arange(16, dtype=torch.float32).reshape(4, 4)).to(torch.uint8)
    want = infer_tiled(_fake_forward_2ch, u8, tile=4)
    for key in ("u8_to_2ch_float", "u8_to_2ch_float_declared"):
        assert want.dtype == torch.float32 and want.shape == (2, 4, 4)
        assert torch.equal(r0[key], want) and torch.equal(r1[key], want), key
    base = torch.arange(10, dtype=torch.float32)
    assert torch.allclose(r0["sync"], base * 1.5) and torch.allclose(r1["sync"], base * 1.5)      # mean of (1x, 2x)
    assert torch.equal(r0["nosync"], base) and torch.equal(r1["nosync"], base * 2)


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU oracle port timed on the host cores) prints ONE JSON line carrying the contract's
    keys; it needs no GPU, so the line is checked here on a tiny workload."""
    import json
    import subprocess
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--ref-batch", "1", "--hw", "64"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "unet_deglare_512x512_images_per_sec" and d["unit"] == "images/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0
    # "reference" = the unmodified reference module from oracle/_ref (oracle/build_ref.py, build container -> GPU box), else the port
    want_kind = "reference" if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "model.py")) else "port"
    assert d["cpu_baseline"]["kind"] == want_kind and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["config"]["onnxruntime_cpu"].startswith("onnxruntime")
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
