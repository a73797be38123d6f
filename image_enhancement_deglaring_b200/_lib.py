"""ctypes binding of libdeglare.so (the C-ABI declared in include/deglare.h).

PyTorch is plumbing here: it owns device memory and streams; every FLOP of the hot path
runs in the hand-written sm_100a kernels of csrc/.  There is no CPU or eager fallback: if
the shared library is missing, loading raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libdeglare.so")

DG_F32, DG_F16, DG_BF16 = 0, 1, 2
DG_X_SAME, DG_X_POOL2, DG_X_UP2, DG_X_CONVT2, DG_X_IMAGE, DG_X_IMAGE_U8 = 0, 1, 2, 3, 4, 5
DG_MAX_BLOCKS = 10

DTYPE_CODES = {"fp32": DG_F32, "fp16": DG_F16, "bf16": DG_BF16}


class DgSrc(C.Structure):
    _fields_ = [
        ("raw", C.c_void_p), ("stats", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
        ("scale", C.c_void_p), ("ct_w", C.c_void_p), ("ct_b", C.c_void_p), ("ct_w_tc", C.c_void_p),
        ("coef", C.c_void_p),
        ("channels", C.c_int32), ("groups", C.c_int32), ("xform", C.c_int32), ("silu", C.c_int32),
        ("ct_cout", C.c_int32), ("reserved", C.c_int32),
    ]


class DgConv3x3Args(C.Structure):
    _fields_ = [
        ("src", DgSrc * 2), ("nsrc", C.c_int32), ("dtype", C.c_int32),
        ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("cout", C.c_int32),
        ("weight", C.c_void_p), ("weight_tc", C.c_void_p), ("out", C.c_void_p), ("out_stats", C.c_void_p),
        ("act_sum", C.c_void_p), ("eps", C.c_float), ("path", C.c_int32), ("weight_comp", C.c_void_p),
    ]


class DgHeadArgs(C.Structure):
    _fields_ = [
        ("src", DgSrc), ("dtype", C.c_int32), ("N", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
        ("cout", C.c_int32), ("weight", C.c_void_p), ("bias", C.c_void_p), ("out", C.c_void_p),
        ("target", C.c_void_p), ("l1_sum", C.c_void_p), ("eps", C.c_float), ("out_kind", C.c_int32),
    ]


class DgLwParams(C.Structure):
    _fields_ = [
        ("in_channels", C.c_int32), ("out_channels", C.c_int32), ("features_start", C.c_int32),
        ("dtype", C.c_int32), ("groups", C.c_int32 * DG_MAX_BLOCKS),
        ("conv_w", (C.c_void_p * 2) * DG_MAX_BLOCKS), ("gn_w", (C.c_void_p * 2) * DG_MAX_BLOCKS),
        ("gn_b", (C.c_void_p * 2) * DG_MAX_BLOCKS), ("up_w", C.c_void_p * 4), ("up_b", C.c_void_p * 4),
        ("conv_w_tc", (C.c_void_p * 2) * DG_MAX_BLOCKS), ("up_w_tc", C.c_void_p * 4),
        ("conv_w_flip", (C.c_void_p * 2) * DG_MAX_BLOCKS), ("up_w_t", C.c_void_p * 4),
        ("up_w_tc_bf16", C.c_void_p * 4), ("conv_w_tc_bf16", (C.c_void_p * 2) * DG_MAX_BLOCKS),
        ("head_w", C.c_void_p), ("head_b", C.c_void_p), ("path", C.c_int32), ("reserved", C.c_int32),
        ("dec_comp", C.c_void_p * 4), ("conv_w_flip_tc_bf16", (C.c_void_p * 2) * DG_MAX_BLOCKS),
        ("up_w_dgrad_tc_bf16", C.c_void_p * 4),
    ]


class DgLwBwdRequest(C.Structure):
    _fields_ = [
        ("grad_y", C.c_void_p), ("y", C.c_void_p), ("target", C.c_void_p), ("loss_grad", C.c_void_p),
        ("grads", C.c_void_p), ("param_mask", C.c_uint64), ("grad_x", C.c_void_p),
    ]


# every symbol include/deglare.h declares: name -> (restype, argtypes)
SYMBOLS = {
    "dg_conv3x3_fused": (C.c_int, [C.POINTER(DgConv3x3Args), C.c_void_p]),
    "dg_conv3x3_wgrad": (C.c_int, [C.POINTER(DgConv3x3Args), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p]),
    "dg_conv3x3_dgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p]),
    "dg_convt2x2_dgrad": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_void_p]),
    "dg_conv3x3_dgrad_wide": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                        C.c_int32, C.c_void_p]),
    "dg_head1x1": (C.c_int, [C.POINTER(DgHeadArgs), C.c_void_p]),
    "dg_pil_resize_u8": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_size_t, C.c_void_p]),
    "dg_cv2_resize_u8": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                   C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dg_augment": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                             C.c_uint64, C.c_void_p]),
    "dg_image_metrics": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_void_p,
                                   C.c_void_p]),
    "dg_lw_workspace_bytes": (C.c_int, [C.POINTER(DgLwParams), C.c_int32, C.c_int32, C.c_int32,
                                        C.POINTER(C.c_size_t)]),
    "dg_lw_forward": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dg_lw_layout": (C.c_int, [C.POINTER(DgLwParams), C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                               C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_int32),
                               C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dg_convt2x2_fused": (C.c_int, [C.POINTER(DgSrc), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_float,
                                    C.c_int32, C.c_void_p]),
    "dg_channel_attention": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_void_p, C.c_void_p]),
    "dg_head1x1_bwd": (C.c_int, [C.POINTER(DgHeadArgs), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dg_act_bwd": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                             C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                             C.c_float, C.c_void_p]),
    "dg_gn_bwd_apply": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
    "dg_grad_gather": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                 C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "dg_scale_bwd_sum": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32,
                                   C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
    "dg_channel_attention_bwd": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                           C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dg_lw_num_params": (C.c_int, [C.POINTER(DgLwParams), C.POINTER(C.c_size_t)]),
    "dg_lw_backward_workspace_bytes": (C.c_int, [C.POINTER(DgLwParams), C.c_int32, C.c_int32, C.c_int32,
                                                 C.POINTER(C.c_size_t)]),
    "dg_lw_backward": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "dg_l1_loss_sum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "dg_lw_backward_l1": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]),
    "dg_lw_backward_select": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.POINTER(DgLwBwdRequest), C.c_int32, C.c_int32,
                                        C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dg_conv_first_dgrad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_void_p]),
    "dg_adamw_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_float,
                                C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int32, C.c_float, C.c_void_p]),
    "dg_adamw_step_graph": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_float,
                                      C.c_void_p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_void_p, C.c_float, C.c_void_p]),
    "dg_lw_profile": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_size_t, C.c_void_p, C.POINTER(C.c_float)]),
    "dg_lw_host_scratch_bytes": (C.c_int, [C.POINTER(DgLwParams), C.c_int32, C.c_int32, C.c_int32,
                                           C.POINTER(C.c_size_t)]),
    "dg_lw_infer_host": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dg_lw_forward_u8": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                   C.c_void_p, C.c_size_t, C.c_void_p]),
    "dg_lw_infer_host_u8": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dg_lw_infer_host_submit": (C.c_int, [C.POINTER(DgLwParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                          C.c_int32, C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p, C.POINTER(C.c_int64)]),
    "dg_lw_infer_host_wait": (C.c_int, [C.c_int64]),
    "dg_band_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_void_p]),
    "dg_gn_affine": (C.c_int, [C.c_void_p, C.c_int32, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_float,
                               C.c_void_p, C.c_void_p]),
    "dg_tc_conv3x3_bytes": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "dg_pack_conv3x3_tc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "dg_tc_convt2x2_bytes": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "dg_pack_convt2x2_tc": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "dg_dec_composite_bytes": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    "dg_pack_dec_composite": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "dg_last_error_string": (C.c_char_p, []),
    "dg_version": (C.c_int, []),
    "dg_set_pdl": (C.c_int, [C.c_int]),
    "dg_set_batch_split": (C.c_int, [C.c_int]),
    "dg_launch_count": (C.c_uint64, []),
}

_lib = None


def load():
    """Load libdeglare.so (once).  Raises if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m image_enhancement_deglaring_b200.build` "
                "(the de-glaring UNet has no CPU / eager fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        if os.environ.get("DG_PDL") == "0":   # A/B switch for programmatic dependent launch
            lib.dg_set_pdl(0)
        if os.environ.get("DG_BATCH_SPLIT") is not None:   # A/B switch / threshold for the two-stream batch split
            lib.dg_set_batch_split(int(os.environ["DG_BATCH_SPLIT"]))
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise RuntimeError(f"libdeglare error {rc}: {load().dg_last_error_string().decode()}")


_generation = 0


def bump_generation():
    """Called by code that rewrites parameter memory without torch ops (FusedAdamW): modules key their packed-weight
    caches on this counter in addition to the tensors' own version counters."""
    global _generation
    _generation += 1


def generation():
    return _generation


def launch_count():
    return int(load().dg_launch_count())
