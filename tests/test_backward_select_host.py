"""CPU-only checks of dg_lw_backward_select: every malformed request is rejected before any CUDA call, and the ctypes mirror of
dg_lw_bwd_request has the size the C compiler gives it."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_PROBE = r"""
import ctypes as C, json
from image_enhancement_deglaring_b200 import _lib
lib = _lib.load()
buf = (C.c_float * 4096)()   # placeholder for every pointer: none may be dereferenced
ptr = C.addressof(buf)

def call(path=0, **fields):
    p = _lib.DgLwParams()
    p.in_channels, p.out_channels, p.features_start, p.dtype, p.path = 1, 1, 8, _lib.DG_F16, path
    r = _lib.DgLwBwdRequest()
    for k, v in fields.items():
        setattr(r, k, v)
    rc = lib.dg_lw_backward_select(C.byref(p), ptr, C.byref(r), 1, 16, 16, ptr, 1 << 40, ptr, 1 << 40, None)
    return [rc, lib.dg_last_error_string().decode()]

res = {
    "both_seeds": call(grad_y=ptr, y=ptr, target=ptr, grads=ptr, param_mask=1),
    "no_seed": call(grads=ptr, param_mask=1),
    "half_l1_seed": call(y=ptr, grads=ptr, param_mask=1),
    "mask_without_grads": call(grad_y=ptr, param_mask=1 << 40),
    "nothing": call(grad_y=ptr, grads=ptr),
    "null_request": [lib.dg_lw_backward_select(None, ptr, None, 1, 16, 16, ptr, 0, ptr, 0, None), lib.dg_last_error_string().decode()],
}
for bit in range(2, 7):
    res[f"path_bit_{bit}"] = call(path=1 << bit, grad_y=ptr, grad_x=ptr)
print(json.dumps(res))
"""


def test_backward_select_rejects_malformed_requests():
    """Both or neither gradient seed, a param_mask without a grads buffer, an empty request and a removed path bit all return 2
    with a message -- run in a process that sees no CUDA device, where a call that reached the runtime would fail differently."""
    out = subprocess.run([sys.executable, "-c", _PROBE], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    res = json.loads(out.stdout.splitlines()[-1])
    assert res["both_seeds"][0] == 2 and "exactly one gradient seed" in res["both_seeds"][1], res["both_seeds"]
    assert res["no_seed"][0] == 2 and "exactly one gradient seed" in res["no_seed"][1], res["no_seed"]
    assert res["half_l1_seed"][0] == 2 and "both y and target" in res["half_l1_seed"][1], res["half_l1_seed"]
    assert res["mask_without_grads"][0] == 2 and "without a grads buffer" in res["mask_without_grads"][1], res["mask_without_grads"]
    assert res["nothing"][0] == 2 and "nothing requested" in res["nothing"][1], res["nothing"]
    assert res["null_request"][0] == 2 and "null request" in res["null_request"][1], res["null_request"]
    for bit in range(2, 7):
        rc, err = res[f"path_bit_{bit}"]
        assert rc == 2 and f"path {1 << bit} sets bit {bit}," in err, (bit, rc, err)


def test_bwd_request_layout_matches_header(tmp_path):
    """sizeof(dg_lw_bwd_request) from gcc (the header compiled as C) equals its ctypes mirror, field offsets included."""
    from image_enhancement_deglaring_b200 import _lib
    src = tmp_path / "req.c"
    src.write_text('#include "deglare.h"\n#include <stddef.h>\n#include <stdio.h>\nint main(void){printf("%zu %zu %zu\\n", '
                   'sizeof(dg_lw_bwd_request), offsetof(dg_lw_bwd_request, param_mask), offsetof(dg_lw_bwd_request, grad_x)); '
                   'return 0;}\n')
    exe = tmp_path / "req"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    size, off_mask, off_gx = (int(v) for v in subprocess.check_output([str(exe)], text=True).split())
    assert size == C.sizeof(_lib.DgLwBwdRequest) == 7 * 8
    assert off_mask == _lib.DgLwBwdRequest.param_mask.offset and off_gx == _lib.DgLwBwdRequest.grad_x.offset
