"""Second CPU oracle: an interpreter for the shipped `best_model.onnx` -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

What `/infer` really executes is not `src/model.py` but the exported graph: `api/app.py:84` builds an
`onnxruntime.InferenceSession` over `best_model.onnx` and `api/app.py:171` runs it (likewise `evaluate.py:95,122`).
onnxruntime (pinned 1.22.0, `api/requirements.txt:7`) is not installed here and cannot be, so this module stands in for it
(SURVEY 8c "optional second oracle"): it reads the protobuf directly (no `onnx` package either) and evaluates the graph's
eleven operator types with their ONNX opset-11 semantics in torch fp32 / fp64 on the CPU:

    Conv, ConvTranspose, InstanceNormalization, Reshape, Shape, Constant, Mul, Add, Sigmoid, AveragePool, Concat

(`nn.GroupNorm` is exported as Reshape -> InstanceNormalization(scale 1, bias 0) -> Reshape -> Mul(gamma) -> Add(beta);
`nn.SiLU` as Sigmoid + Mul.)  Parity status: the operator semantics are the published ONNX ones; the interpreter is pinned by
`tests/test_oracle.py::test_onnx_artefact_*` against the golden outputs the reference module itself produced on the same
weights (`tests/golden/lw_png.npz`, `lw_rand.npz`) -- i.e. the exported artefact, the PyTorch module and `oracle/torch_unet.py`
agree to 1e-5 on the two shipped sample images.

The shipped `best_model.onnx` is not part of this repository.  The test runs on the same network exported the same way (opset 11,
229 nodes), stored without its weights (`tests/golden/make_onnx_golden.py` -> `tests/golden/onnx_graph.npz`); the initializers
are re-attached from `weights/best_model.pth`, which tools/onnx_weights.py extracted from the shipped file.
"""
import struct

import numpy as np
import torch
import torch.nn.functional as F


# ---- minimal protobuf reader (wire format only; field numbers from onnx.proto3) -------------------------------------------
def _varint(buf, pos):
    out = shift = 0
    while True:
        b = buf[pos]
        pos += 1
        out |= (b & 0x7F) << shift
        if not b & 0x80:
            return out, pos
        shift += 7


def _fields(buf):
    pos, n = 0, len(buf)
    while pos < n:
        key, pos = _varint(buf, pos)
        fno, wt = key >> 3, key & 7
        if wt == 0:
            val, pos = _varint(buf, pos)
        elif wt == 1:
            val, pos = buf[pos:pos + 8], pos + 8
        elif wt == 2:
            ln, pos = _varint(buf, pos)
            val, pos = buf[pos:pos + ln], pos + ln
        elif wt == 5:
            val, pos = buf[pos:pos + 4], pos + 4
        else:
            raise ValueError(f"unsupported wire type {wt}")
        yield fno, wt, val


def _signed(v):
    return v - (1 << 64) if v >= (1 << 63) else v


def _packed_ints(wt, val, out):
    if wt == 0:
        out.append(_signed(val))
    else:
        p = 0
        while p < len(val):
            d, p = _varint(val, p)
            out.append(_signed(d))


_DTYPES = {1: np.float32, 7: np.int64, 6: np.int32, 11: np.float64}


def _tensor(buf):
    """TensorProto -> (name, ndarray)."""
    dims, name, raw, floats, ints, dtype = [], "", None, [], [], 1
    for fno, wt, val in _fields(buf):
        if fno == 1:
            _packed_ints(wt, val, dims)
        elif fno == 2:
            dtype = val
        elif fno == 4:
            floats.extend([struct.unpack("<f", val)[0]] if wt == 5 else struct.unpack(f"<{len(val) // 4}f", val))
        elif fno == 7:
            _packed_ints(wt, val, ints)
        elif fno == 8:
            name = bytes(val).decode()
        elif fno == 9:
            raw = bytes(val)
    if dtype not in _DTYPES:
        raise ValueError(f"tensor {name!r}: unsupported ONNX data type {dtype}")
    if raw is not None:
        arr = np.frombuffer(raw, dtype=np.dtype(_DTYPES[dtype]).newbyteorder("<")).astype(_DTYPES[dtype])
    elif dtype == 1:
        arr = np.asarray(floats, dtype=np.float32)
    else:
        arr = np.asarray(ints, dtype=_DTYPES[dtype])
    return name, arr.reshape(dims)


def _attribute(buf):
    """AttributeProto -> (name, python value)."""
    name, f, i, s, t, floats, ints = "", None, None, None, None, [], []
    for fno, wt, val in _fields(buf):
        if fno == 1:
            name = bytes(val).decode()
        elif fno == 2:
            f = struct.unpack("<f", val)[0]
        elif fno == 3:
            i = _signed(val)
        elif fno == 4:
            s = bytes(val).decode()
        elif fno == 5:
            t = _tensor(val)[1]
        elif fno == 7:
            floats.extend([struct.unpack("<f", val)[0]] if wt == 5 else struct.unpack(f"<{len(val) // 4}f", val))
        elif fno == 8:
            _packed_ints(wt, val, ints)
    for v in (t, s, f, i):
        if v is not None:
            return name, v
    return name, (ints if ints else floats)


def _node(buf):
    ins, outs, op, attrs = [], [], None, {}
    for fno, _, val in _fields(buf):
        if fno == 1:
            ins.append(bytes(val).decode())
        elif fno == 2:
            outs.append(bytes(val).decode())
        elif fno == 4:
            op = bytes(val).decode()
        elif fno == 5:
            k, v = _attribute(val)
            attrs[k] = v
    return op, ins, outs, attrs


def _value_name(buf):
    for fno, _, val in _fields(buf):
        if fno == 1:
            return bytes(val).decode()
    return ""


class OnnxGraph:
    """The parsed artefact: initializers, nodes in graph (= topological) order, graph input / output names."""

    def __init__(self, path):
        with open(path, "rb") as fh:
            model = memoryview(fh.read())
        graph = None
        self.opset = None
        for fno, _, val in _fields(model):
            if fno == 7:
                graph = val
            elif fno == 8:   # opset_import
                for f2, _, v2 in _fields(val):
                    if f2 == 2:
                        self.opset = v2
        if graph is None:
            raise ValueError("no GraphProto in file")
        self.inits, self.nodes, self.inputs, self.outputs = {}, [], [], []
        for fno, _, val in _fields(graph):
            if fno == 1:
                self.nodes.append(_node(val))
            elif fno == 5:
                name, arr = _tensor(val)
                self.inits[name] = arr
            elif fno == 11:
                self.inputs.append(_value_name(val))
            elif fno == 12:
                self.outputs.append(_value_name(val))
        self.inputs = [n for n in self.inputs if n not in self.inits]

    def op_types(self):
        return sorted({n[0] for n in self.nodes})

    # ---- evaluation: ONNX opset-11 operator semantics --------------------------------------------------------------------
    def run(self, x, dtype=torch.float32, taps=None):
        """x: ndarray / tensor [N,1,H,W] -> ndarray [N,1,H,W] (what `session.run(None, {input: x})[0]` returns)."""
        env = {k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in self.inits.items()}
        env = {k: (v.to(dtype) if v.is_floating_point() else v) for k, v in env.items()}
        env[self.inputs[0]] = torch.as_tensor(x).to(dtype)
        with torch.no_grad():
            for op, ins, outs, at in self.nodes:
                a = [env[i] if i else None for i in ins]
                env[outs[0]] = self._eval(op, a, at, dtype)
                if taps is not None and op in ("Conv", "ConvTranspose"):
                    taps[outs[0]] = env[outs[0]]
        return env[self.outputs[0]].float().numpy()

    @staticmethod
    def _eval(op, a, at, dtype):
        if op == "Conv":
            pads = at.get("pads", [0, 0, 0, 0])
            if pads[0] != pads[2] or pads[1] != pads[3]:
                raise NotImplementedError("asymmetric Conv pads")
            return F.conv2d(a[0], a[1], a[2] if len(a) > 2 else None, stride=tuple(at.get("strides", [1, 1])),
                            padding=(pads[0], pads[1]), dilation=tuple(at.get("dilations", [1, 1])), groups=at.get("group", 1))
        if op == "ConvTranspose":
            pads = at.get("pads", [0, 0, 0, 0])
            if any(pads) or any(at.get("output_padding", [0, 0])):
                raise NotImplementedError("padded ConvTranspose")
            return F.conv_transpose2d(a[0], a[1], a[2] if len(a) > 2 else None, stride=tuple(at.get("strides", [1, 1])),
                                      dilation=tuple(at.get("dilations", [1, 1])), groups=at.get("group", 1))
        if op == "InstanceNormalization":     # per (n, c) over the remaining axes, biased variance, eps inside the sqrt
            x = a[0]
            axes = tuple(range(2, x.dim()))
            mean = x.mean(dim=axes, keepdim=True)
            var = ((x - mean) ** 2).mean(dim=axes, keepdim=True)
            shape = (1, -1) + (1,) * (x.dim() - 2)
            return (x - mean) / torch.sqrt(var + at.get("epsilon", 1e-5)) * a[1].reshape(shape) + a[2].reshape(shape)
        if op == "Reshape":                    # 0 copies the input dimension, -1 is inferred
            shape = [int(v) for v in a[1].tolist()]
            shape = [a[0].shape[i] if v == 0 else v for i, v in enumerate(shape)]
            return a[0].reshape(shape)
        if op == "Shape":
            return torch.tensor(list(a[0].shape), dtype=torch.int64)
        if op == "Constant":
            v = torch.from_numpy(np.ascontiguousarray(at["value"]))
            return v.to(dtype) if v.is_floating_point() else v
        if op == "Mul":
            return a[0] * a[1]
        if op == "Add":
            return a[0] + a[1]
        if op == "Sigmoid":
            return torch.sigmoid(a[0])
        if op == "AveragePool":
            pads = at.get("pads", [0, 0, 0, 0])
            if any(pads) or at.get("ceil_mode", 0):
                raise NotImplementedError("padded / ceil-mode AveragePool")
            return F.avg_pool2d(a[0], tuple(at["kernel_shape"]), tuple(at.get("strides", at["kernel_shape"])))
        if op == "Concat":
            return torch.cat(a, dim=at["axis"])
        raise NotImplementedError(f"ONNX operator {op}")
