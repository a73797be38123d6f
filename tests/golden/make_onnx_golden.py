#!/usr/bin/env python
"""The ONNX graph behind tests/test_oracle.py::test_onnx_artefact_interpreter_matches_reference_goldens, without its weights.

The shipped `best_model.onnx` (graph + the 486,409 weights that tools/onnx_weights.py turned into weights/best_model.pth) is not
part of this repository.  This script exports the same network the way scripts/export_to_onnx.py did -- src/model.py's
LightweightUNet module layout, torch.onnx's TorchScript exporter, opset 11, dynamic N / H / W, input "input", output "output" --
from weights/best_model.pth, and stores:

    model        the ModelProto bytes with every initializer removed from the graph (~40 KB instead of ~2 MB)
    init_names   initializer names in graph order
    init_keys    the state_dict key each initializer holds (GroupNorm gamma / beta are the anonymous onnx::Mul_N / onnx::Add_N
                 tensors of shape [C,1,1], keyed by the module path of the node that consumes them, as tools/onnx_weights.py does)
    init_shapes  their shapes, "a,b,c"
    init_sha256  sha256 of each initializer's little-endian float32 bytes

The test re-attaches the initializers from weights/best_model.pth and checks each against its hash.

    python tests/golden/make_onnx_golden.py      # writes tests/golden/onnx_graph.npz
"""
import hashlib
import io
import os
import re
import sys
import tempfile

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import onnx_interp as oi          # noqa: E402
from oracle.torch_unet import groups_lightweight  # noqa: E402


def _block(cin, c, g):
    return nn.Sequential(nn.Conv2d(cin, c, 3, padding=1, bias=False), nn.GroupNorm(g, c), nn.SiLU(),
                         nn.Conv2d(c, c, 3, padding=1, bias=False), nn.GroupNorm(g, c), nn.SiLU())


class LightweightUNet(nn.Module):
    """src/model.py's module layout (names, order, bias-free convs), so the exported node and initializer names are the shipped ones."""

    def __init__(self, features_start=8, num_groups=8):
        super().__init__()
        f = [features_start << i for i in range(5)]
        g = [groups_lightweight(c, num_groups) for c in f]
        self.enc1, self.enc2 = _block(1, f[0], g[0]), _block(f[0], f[1], g[1])
        self.enc3, self.enc4 = _block(f[1], f[2], g[2]), _block(f[2], f[3], g[3])
        self.bottleneck = _block(f[3], f[4], g[4])
        for lvl in (4, 3, 2, 1):
            setattr(self, f"upconv{lvl}", nn.ConvTranspose2d(f[lvl], f[lvl - 1], 2, stride=2))
            setattr(self, f"dec{lvl}", _block(2 * f[lvl - 1], f[lvl - 1], g[lvl - 1]))
        self.output_conv = nn.Conv2d(f[0], 1, 1)

    def forward(self, x):
        e1 = self.enc1(x)
        e2 = self.enc2(F.avg_pool2d(e1, 2))
        e3 = self.enc3(F.avg_pool2d(e2, 2))
        e4 = self.enc4(F.avg_pool2d(e3, 2))
        d = self.bottleneck(F.avg_pool2d(e4, 2))
        for lvl, skip in ((4, e4), (3, e3), (2, e2), (1, e1)):
            d = getattr(self, f"dec{lvl}")(torch.cat((getattr(self, f"upconv{lvl}")(d), skip), 1))
        return self.output_conv(d)


def export(sd):
    m = LightweightUNet()
    m.load_state_dict(sd, strict=True)
    m.eval()
    # The exporter loads the `onnx` package only to insert custom onnx-script functions; this graph has none, so that step is the
    # identity and the script runs where the package is not installed.
    from torch.onnx._internal.torchscript_exporter import onnx_proto_utils
    onnx_proto_utils._add_onnxscript_fn = lambda proto, custom_opsets: proto
    buf = io.BytesIO()
    axes = {0: "batch", 2: "height", 3: "width"}
    torch.onnx.export(m, torch.rand(1, 1, 512, 512), buf, dynamo=False, opset_version=11, input_names=["input"],
                      output_names=["output"], dynamic_axes={"input": axes, "output": axes})
    return buf.getvalue()


def _varint_bytes(v):
    out = bytearray()
    while True:
        b = v & 0x7F
        v >>= 7
        out.append(b | (0x80 if v else 0))
        if not v:
            return bytes(out)


def _raw_fields(buf):
    """(field number, raw bytes of the whole field) for each field of one protobuf message."""
    pos = 0
    while pos < len(buf):
        start = pos
        key, pos = oi._varint(buf, pos)
        wt = key & 7
        if wt == 0:
            _, pos = oi._varint(buf, pos)
        elif wt == 1:
            pos += 8
        elif wt == 2:
            ln, pos = oi._varint(buf, pos)
            pos += ln
        elif wt == 5:
            pos += 4
        else:
            raise ValueError(f"unsupported wire type {wt}")
        yield key >> 3, bytes(buf[start:pos])


def strip_initializers(model):
    """ModelProto bytes -> the same bytes with GraphProto.initializer (field 5 of field 7) removed."""
    out = bytearray()
    for fno, raw in _raw_fields(memoryview(model)):
        if fno != 7:
            out += raw
            continue
        _, p = oi._varint(raw, 0)      # field key
        _, p = oi._varint(raw, p)      # length
        body = b"".join(r for f, r in _raw_fields(memoryview(raw)[p:]) if f != 5)
        out += _varint_bytes((7 << 3) | 2) + _varint_bytes(len(body)) + body
    return bytes(out)


def main():
    sd = torch.load(os.path.join(ROOT, "weights", "best_model.pth"))
    model = export(sd)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "best_model.onnx")
        with open(path, "wb") as fh:
            fh.write(model)
        g = oi.OnnxGraph(path)
    # anonymous GroupNorm affine initializers: consumer "/enc1/enc1.1/Mul_output_0" -> "enc1.1.weight" (Add -> ".bias")
    anon = {}
    pat = re.compile(r"^/\w+/(?P<mod>[\w.]+)/(?P<op>Mul|Add)_output_0$")
    for op, ins, outs, _ in g.nodes:
        m = pat.match(outs[0])
        for i in ins:
            if i.startswith("onnx::") and i in g.inits and m and op in ("Mul", "Add"):
                anon[i] = m.group("mod") + (".weight" if op == "Mul" else ".bias")
    names = list(g.inits)
    keys = [anon.get(n, n) for n in names]
    assert sorted(keys) == sorted(sd), set(keys) ^ set(sd)
    for n, k in zip(names, keys):
        assert np.array_equal(g.inits[n].reshape(-1), sd[k].numpy().reshape(-1)), n
    out = {
        "model": np.frombuffer(strip_initializers(model), dtype=np.uint8),
        "init_names": np.array(names), "init_keys": np.array(keys),
        "init_shapes": np.array([",".join(map(str, g.inits[n].shape)) for n in names]),
        "init_sha256": np.array([hashlib.sha256(g.inits[n].astype("<f4").tobytes()).hexdigest() for n in names]),
    }
    np.savez_compressed(os.path.join(HERE, "onnx_graph.npz"), **out)
    print("wrote onnx_graph.npz:", len(g.nodes), "nodes,", len(names), "initializers,", out["model"].size, "graph bytes")


if __name__ == "__main__":
    main()
