"""ctypes binding of libyogo_b200.so (include/yogo_b200.h).

There is deliberately no CPU or eager-PyTorch fallback: if the shared library is missing, or
the device is not sm_100, every product entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libyogo_b200.so")

YG_F32, YG_BF16, YG_U8 = 0, 1, 2
ACT_NONE, ACT_LRELU, ACT_SILU = 0, 1, 2
IMPL_AUTO, IMPL_SIMT, IMPL_TCGEN05 = 0, 1, 2

c_void_p, c_int, c_float, c_double, c_size_t, c_longlong = (
    C.c_void_p,
    C.c_int,
    C.c_float,
    C.c_double,
    C.c_size_t,
    C.c_longlong,
)


class FwdEpilogue(C.Structure):
    _fields_ = [
        ("scale", c_void_p),
        ("shift", c_void_p),
        ("act", c_int),
        ("dropscale", c_void_p),
        ("stats", c_void_p),
        ("preact", c_void_p),
        ("actmask", c_void_p),
    ]


class BwdEpilogue(C.Structure):
    _fields_ = [
        ("saved", c_void_p),
        ("act", c_int),
        ("dropscale", c_void_p),
        ("bn_scale", c_void_p),
        ("bn_shift", c_void_p),
        ("bn_mean", c_void_p),
        ("bn_invstd", c_void_p),
        ("bn_sums", c_void_p),
        ("actmask", c_void_p),
    ]


# name -> (restype, argtypes); mirrors include/yogo_b200.h one to one
_PROTOS = {
    "yg_version": (c_int, []),
    "yg_last_error": (C.c_char_p, []),
    "yg_device_check": (c_int, []),
    "yg_set_conv_impl": (c_int, [c_int]),
    "yg_get_conv_impl": (c_int, []),
    "yg_set_tc_options": (c_int, [c_int]),
    "yg_get_tc_options": (c_int, []),
    "yg_tc_debug_read": (c_int, [c_void_p, c_int]),
    "yg_launch_count": (C.c_ulonglong, []),
    "yg_conv_first_fwd": (
        c_int,
        [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, C.POINTER(FwdEpilogue), c_void_p],
    ),
    "yg_conv_first_bwd": (
        c_int,
        [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, C.POINTER(BwdEpilogue),
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_size_t, c_void_p],
    ),
    "yg_conv_first_bwd_workspace": (c_size_t, [c_int, c_int]),
    "yg_conv_first_gram": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "yg_conv_first_stats_from_gram": (c_int, [c_void_p, c_void_p, c_void_p, c_double, c_int, c_void_p, c_void_p]),
    "yg_conv_first_bwd_finalize": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_int, c_float, c_int,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "yg_conv_first_dgrad": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, C.POINTER(BwdEpilogue), c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "yg_conv_first_bn_means": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_int, c_void_p, c_void_p, c_void_p],
    ),
    "yg_conv_fwd": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, C.POINTER(FwdEpilogue), c_void_p],
    ),
    "yg_conv_dgrad": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, C.POINTER(BwdEpilogue), c_void_p],
    ),
    "yg_conv_wgrad_workspace": (c_size_t, [c_int] * 7),
    "yg_conv_wgrad": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
         c_void_p, c_size_t, c_void_p],
    ),
    "yg_bn_finalize": (
        c_int,
        [c_void_p, c_double, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p,
         c_void_p, c_int, c_void_p],
    ),
    "yg_bn_fold_eval": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int, c_void_p],
    ),
    "yg_bn_act_apply": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
    ),
    "yg_bn_stats": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "yg_bn_bwd_sums": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "yg_bn_bwd_apply": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_float, c_int, c_void_p],
    ),
    "yg_head_fwd": (
        c_int,
        [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
         c_float, c_float, c_int, c_void_p, c_void_p, c_void_p],
    ),
    "yg_head_bwd_workspace": (c_size_t, [c_int] * 5),
    "yg_head_bwd": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
         c_float, c_float, c_float, c_float, C.POINTER(BwdEpilogue), c_float, c_void_p, c_size_t, c_void_p],
    ),
    "yg_head_softmax_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "yg_yogo_loss_workspace": (c_size_t, [c_int] * 3),
    "yg_yogo_loss_fwd_bwd": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_float, c_float, c_float,
         c_void_p, c_size_t, c_void_p],
    ),
    "yg_format_preds_workspace": (c_size_t, [c_int] * 4),
    "yg_format_preds_batch": (
        c_int,
        [c_void_p, c_int, c_int, c_int, c_int, c_float, c_double, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_size_t, c_void_p],
    ),
    "yg_box_iou_cost": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "yg_compact_labels": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "yg_lsap_workspace_words": (c_longlong, [c_int, c_int]),
    "yg_lsap_batch": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "yg_match_batch": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "yg_confusion_batch": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "yg_coco_match_batch": (
        c_int,
        [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_longlong, C.POINTER(c_double), c_void_p,
         c_void_p, c_void_p, c_void_p],
    ),
    "yg_coco_accumulate": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_int, C.POINTER(c_double), c_void_p, c_void_p, c_void_p],
    ),
    "yg_score_rows_batch": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_longlong, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
         C.POINTER(c_float), c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "yg_roc_keys": (c_int, [c_void_p, c_longlong, c_int, c_void_p, c_void_p]),
    "yg_roc_curves": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_longlong, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "yg_flip_images":(c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "yg_flip_labels": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "yg_format_labels_batch": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "yg_dropout_scales": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "yg_dd_draw": (c_int, [c_void_p, c_void_p, c_float, c_float, c_int, c_int, c_void_p]),
    "yg_dd_gather_images": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "yg_dd_build_labels": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "yg_png_gray8_workspace": (c_size_t, [c_int, c_int, c_int, c_longlong]),
    "yg_png_decode_gray8": (
        c_int,
        [c_void_p, c_longlong, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "yg_adamw_flat_dev": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_void_p, c_void_p]),
    "yg_adamw_flat": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_void_p, c_longlong, c_float, c_float, c_float, c_float, c_float, c_longlong,
         c_float, c_void_p],
    ),
}

EXPORTED_SYMBOLS = tuple(_PROTOS)

_lib: Optional[C.CDLL] = None
_device_checked = False


class YogoB200Error(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (no GPU needed) and bind every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise YogoB200Error(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C yogo_b200/csrc`). yogo_b200 has no CPU / eager fallback."
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def lib() -> C.CDLL:
    """Library handle for compute calls: also verifies an sm_100 device once."""
    global _device_checked
    l = load()
    if not _device_checked:
        if not torch.cuda.is_available():
            raise YogoB200Error("yogo_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        rc = l.yg_device_check()
        if rc != 0:
            raise YogoB200Error(l.yg_last_error().decode())
        _device_checked = True
    return l


def check(rc: int) -> None:
    if rc != 0:
        raise YogoB200Error(f"yogo_b200 [{rc}]: {load().yg_last_error().decode()}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream() -> int:
    """The caller's current stream on the CURRENT device; every entry point runs under `on_device` so that the current
    device is the one the tensors live on."""
    return torch.cuda.current_stream().cuda_stream


def on_device(pick):
    """Decorator: run the wrapped entry point with the CUDA device of the tensor `pick(*args, **kwargs)` returns as the
    current device (kernel launches, cudaMemsetAsync, TMA descriptors and `stream()` all use the current device; ATen
    does this switch for every op of the reference).  Non-CUDA tensors pass through so that the callee raises its own
    'no CPU fallback' error."""
    import functools

    def deco(fn):
        @functools.wraps(fn)
        def wrapped(*args, **kwargs):
            t = pick(*args, **kwargs)
            if isinstance(t, torch.Tensor) and t.is_cuda and t.device.index != torch.cuda.current_device():
                with torch.cuda.device(t.device):
                    return fn(*args, **kwargs)
            return fn(*args, **kwargs)

        return wrapped

    return deco


def dtype_code(dt: torch.dtype) -> int:
    if dt == torch.float32:
        return YG_F32
    if dt == torch.bfloat16:
        return YG_BF16
    if dt == torch.uint8:
        return YG_U8
    raise YogoB200Error(f"unsupported dtype {dt}")


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise YogoB200Error(
            f"{what} must live on a CUDA device (got {t.device}); yogo_b200 runs on B200 only and has no CPU fallback"
        )


class Workspace:
    """Grow-only per-device scratch buffers keyed by purpose."""

    def __init__(self):
        self._bufs = {}

    def get(self, key: str, nbytes: int, device) -> torch.Tensor:
        k = (key, torch.device(device).index)
        buf = self._bufs.get(k)
        if buf is None or buf.numel() < nbytes:
            buf = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)
            self._bufs[k] = buf
        return buf


workspace = Workspace()


def set_conv_impl(impl: str) -> None:
    code = {"auto": IMPL_AUTO, "simt": IMPL_SIMT, "tcgen05": IMPL_TCGEN05}[impl]
    check(load().yg_set_conv_impl(code))


def get_conv_impl() -> str:
    return {IMPL_AUTO: "auto", IMPL_SIMT: "simt", IMPL_TCGEN05: "tcgen05"}[load().yg_get_conv_impl()]


FP32_X3_BIT = 1 << 21


def set_fp32_tensor_cores(on: bool) -> None:
    """fp32 tensors (`compute_dtype = torch.float32`) on the bf16 tensor cores through the split-bf16 "x3" convolutions of
    csrc/x3.cu (error ~2^-16 per product, ~13x faster than the exact SIMT kernels).  Off by default: the exact kernels are
    the fp32 parity path - LeakyReLU networks amplify any rounding difference wherever a pre-activation sits within that
    difference of the kink, so gradients of the x3 path agree with the reference to ~1e-2, not 1e-3 (its forward does, and so
    do the gradients of SiLU networks)."""
    lib_ = load()
    cur = lib_.yg_get_tc_options()
    check(lib_.yg_set_tc_options((cur | FP32_X3_BIT) if on else (cur & ~FP32_X3_BIT)))


def get_fp32_tensor_cores() -> bool:
    return bool(load().yg_get_tc_options() & FP32_X3_BIT)
