"""ctypes binding of libyl11.so (include/yl11.h) — the only door between the Python host code and the GPU.

There is deliberately no fallback: if the library is missing, or no sm_100 device is present, every compute
entry point raises.  `available()` lets CPU-only tooling (tests of host logic, docs) import the package.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

_LIB_PATH = Path(__file__).resolve().parent / "lib" / "libyl11.so"
_lib = None
_inited_devices: set[int] = set()

YL_BF16, YL_F32, YL_U8, YL_F16 = 0, 1, 2, 3
#: torch dtypes an image batch may arrive in -> yl_dtype (uint8 = image bytes, scaled by 1/255 on ingest)
INGEST_DTYPES = {torch.float32: YL_F32, torch.float16: YL_F16, torch.uint8: YL_U8}
ACT_NONE, ACT_SILU = 0, 1
IMPL_AUTO, IMPL_DIRECT, IMPL_TCGEN05 = 0, 1, 2


class YLError(RuntimeError):
    """Raised for every non-zero yl_status."""


class Tensor(C.Structure):
    """Mirror of `yl_tensor`: a channel slice of an NHWC buffer."""

    _fields_ = [
        ("data", C.c_void_p),
        ("n", C.c_int32),
        ("h", C.c_int32),
        ("w", C.c_int32),
        ("c", C.c_int32),
        ("cstride", C.c_int32),
        ("coff", C.c_int32),
        ("dtype", C.c_int32),
        ("_pad", C.c_int32),
    ]


class DetEpilogue(C.Structure):
    """Mirror of `yl_det_epilogue`."""

    _fields_ = [
        ("pred", C.c_void_p),
        ("mode", C.c_int32),
        ("reg_max", C.c_int32),
        ("nc", C.c_int32),
        ("A", C.c_int32),
        ("anchor0", C.c_int32),
        ("stride", C.c_float),
        ("conf", C.c_float),
        ("_pad", C.c_int32),
        ("cand_ws", C.c_void_p),
    ]


DET_NONE, DET_BOX, DET_CLS, DET_CLS_FILTER = 0, 1, 2, 3


class LbImage(C.Structure):
    """Mirror of `yl_lb_image` (40 bytes)."""

    _fields_ = [
        ("src", C.c_void_p),
        ("sh", C.c_int32),
        ("sw", C.c_int32),
        ("pitch", C.c_int32),
        ("new_w", C.c_int32),
        ("new_h", C.c_int32),
        ("left", C.c_int32),
        ("top", C.c_int32),
        ("_pad", C.c_int32),
    ]


class ConvArgs(C.Structure):
    _fields_ = [
        ("x", Tensor),
        ("y", Tensor),
        ("res", Tensor),
        ("y_up", Tensor),
        ("w", C.c_void_p),
        ("bias", C.c_void_p),
        ("k", C.c_int32),
        ("stride", C.c_int32),
        ("ci_pad", C.c_int32),
        ("co_pad", C.c_int32),
        ("act", C.c_int32),
        ("upsample2x", C.c_int32),
        ("impl", C.c_int32),
        ("_pad", C.c_int32),
        ("det", DetEpilogue),
    ]


class ConvTcPlan(C.Structure):
    """Mirror of `yl_conv_tc_plan` (how the tcgen05 path would run a conv; yl_conv_tc_info)."""

    _fields_ = [(k, C.c_int32) for k in ("flat", "patch", "wres", "tile_w", "tile_h", "tile_n", "m_tiles", "n_tiles",
                                         "co_tile", "kblk", "stages", "grid", "smem_bytes", "tmem_cols", "cw",
                                         "stg_sub", "epi_kind")]


class ConvChain(C.Structure):
    """Mirror of `yl_conv_chain` (a built chain of conv layers: yl_conv_chain_build / yl_conv_chain_run)."""

    _fields_ = [("desc", C.c_void_p)] + [(k, C.c_int32) for k in ("n_layers", "batch", "cluster", "smem_bytes",
                                                                   "tmem_cols", "reserved")]


class TtaCanvas(C.Structure):
    """Mirror of `yl_tta_canvas` (32 bytes)."""

    _fields_ = [("y", C.c_void_p)] + [(k, C.c_int32) for k in ("H", "W", "h", "w", "flip", "_pad")]


class TtaPass(C.Structure):
    """Mirror of `yl_tta_pass` (32 bytes)."""

    _fields_ = [("pred", C.c_void_p), ("A", C.c_int32), ("a0", C.c_int32), ("n", C.c_int32), ("flip", C.c_int32),
                ("scale", C.c_float), ("_pad", C.c_int32)]


class EmbedTap(C.Structure):
    """Mirror of `yl_embed_tap` (48 bytes)."""

    _fields_ = [("x", Tensor), ("col", C.c_int32), ("_pad", C.c_int32)]


class CocoevalSet(C.Structure):
    """Mirror of `yl_cocoeval_set`."""

    _fields_ = [(k, C.c_int32) for k in ("n_pairs", "n_cats", "n_slots", "max_gt", "max_dt")] + [
        (k, C.c_void_p) for k in ("pair_cat", "gt_off", "gt_bbox", "gt_area", "gt_iscrowd", "gt_id", "slot_off", "dt_bbox",
                                  "dt_score", "dt_area", "dt_id")]


class CocoevalParams(C.Structure):
    """Mirror of `yl_cocoeval_params`."""

    _fields_ = [(k, C.c_void_p) for k in ("iou_thrs", "rec_thrs", "area_rng", "max_dets")] + [
        (k, C.c_int32) for k in ("T", "R", "A", "M")]


class CocoevalSlots(C.Structure):
    """Mirror of `yl_cocoeval_slots`."""

    _fields_ = [(k, C.c_void_p) for k in ("key", "rank", "flags", "npig")]


_PROTOTYPES = {
    "yl_version": (C.c_int, []),
    "yl_last_error_string": (C.c_char_p, []),
    "yl_init": (C.c_int, [C.c_int]),
    "yl_set_pdl": (C.c_int, [C.c_int]),
    "yl_debug_timeline": (C.c_int, [C.c_void_p, C.c_int]),
    "yl_fold_bn_pack": (C.c_int, [C.c_void_p] * 6 + [C.c_float] + [C.c_int] * 6 + [C.c_void_p, C.c_void_p, C.c_void_p]),
    "yl_nchw_to_nhwc": (C.c_int, [C.c_void_p, C.POINTER(Tensor), C.c_void_p]),
    "yl_nhwc_to_nchw": (C.c_int, [C.POINTER(Tensor), C.c_void_p, C.c_void_p]),
    "yl_copy_slice": (C.c_int, [C.POINTER(Tensor), C.POINTER(Tensor), C.c_void_p]),
    "yl_upsample2x": (C.c_int, [C.POINTER(Tensor), C.POINTER(Tensor), C.c_void_p]),
    "yl_conv_bn_act": (C.c_int, [C.POINTER(ConvArgs), C.c_void_p]),
    "yl_conv_tc_supported": (C.c_int, [C.POINTER(ConvArgs)]),
    "yl_conv_b2b_det_supported": (C.c_int, [C.POINTER(ConvArgs), C.POINTER(ConvArgs)]),
    "yl_conv_b2b_det": (C.c_int, [C.POINTER(ConvArgs), C.POINTER(ConvArgs), C.c_void_p]),
    "yl_conv_tc_info": (C.c_int, [C.POINTER(ConvArgs), C.POINTER(ConvTcPlan)]),
    "yl_conv_chain_desc_bytes": (C.c_size_t, [C.c_int]),
    "yl_conv_chain_supported": (C.c_int, [C.POINTER(ConvArgs)]),
    "yl_conv_chain_build": (C.c_int, [C.POINTER(ConvArgs), C.c_int, C.c_void_p, C.c_size_t, C.POINTER(ConvChain),
                                      C.c_void_p]),
    "yl_conv_chain_run": (C.c_int, [C.POINTER(ConvChain), C.c_void_p]),
    "yl_conv_chain_debug": (C.c_int, [C.c_void_p]),
    "yl_stem_conv": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                               C.POINTER(Tensor), C.c_int, C.c_void_p]),
    "yl_dwconv3x3": (C.c_int, [C.POINTER(Tensor), C.POINTER(Tensor), C.c_void_p, C.c_void_p, C.c_int,
                               C.POINTER(Tensor), C.c_void_p]),
    "yl_dw_pw_supported": (C.c_int, [C.POINTER(ConvArgs)]),
    "yl_dw_pw_conv": (C.c_int, [C.POINTER(ConvArgs), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "yl_dw_pw_det_supported": (C.c_int, [C.POINTER(ConvArgs), C.POINTER(ConvArgs)]),
    "yl_dw_pw_det": (C.c_int, [C.POINTER(ConvArgs), C.c_void_p, C.c_void_p, C.c_int, C.POINTER(ConvArgs), C.c_void_p]),
    "yl_sppf_pool": (C.c_int, [C.POINTER(Tensor)] * 4 + [C.c_int, C.c_void_p]),
    "yl_psa_attention": (C.c_int, [C.POINTER(Tensor), C.POINTER(Tensor), C.c_int, C.c_int, C.c_int, C.c_float,
                                   C.c_void_p]),
    "yl_detect_decode": (C.c_int, [C.POINTER(Tensor), C.c_int, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p,
                                   C.c_void_p]),
    "yl_detect_decode_into": (C.c_int, [C.POINTER(Tensor), C.c_int, C.POINTER(C.c_float), C.c_int, C.c_int, C.c_void_p,
                                        C.c_int, C.c_int, C.c_void_p]),
    "yl_dfl": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "yl_nms_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "yl_nms_batched": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_double, C.c_void_p, C.c_int,
                                 C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_size_t, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "yl_nms_priors_workspace_bytes": (C.c_size_t, [C.c_int] * 5),
    "yl_nms_batched_priors": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_float, C.c_double, C.c_void_p,
                                        C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "yl_nms_begin": (C.c_int, [C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "yl_debug_nms_phases": (C.c_int, [C.c_void_p]),
    "yl_nms_select": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_float,
                                C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p]),
    "yl_nms_boxes_workspace_bytes": (C.c_size_t, [C.c_int]),
    "yl_nms_boxes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p,
                               C.c_void_p, C.c_void_p]),
    "yl_xywh2xyxy_inplace": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "yl_scale_boxes": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "yl_to_f32": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p]),
    "yl_stem_fused_supported": (C.c_int, [C.c_int, C.c_int, C.c_int]),
    "yl_stem_fused": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.POINTER(Tensor), C.c_void_p]),
    "yl_c3k2_tail_supported": (C.c_int, [C.c_int, C.c_int]),
    "yl_c3k2_tail": (C.c_int, [C.POINTER(Tensor), C.POINTER(Tensor), C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "yl_c3k2_tail_tc": (C.c_int, [C.POINTER(Tensor), C.POINTER(Tensor), C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "yl_match_predictions": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                       C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "yl_confusion_matrix": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_int, C.c_int, C.c_float, C.c_float, C.c_void_p, C.c_void_p]),
    "yl_letterbox_u8": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "yl_tta_scale_img": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(TtaCanvas),
                                   C.c_void_p]),
    "yl_tta_merge": (C.c_int, [C.POINTER(TtaPass), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "yl_embed_pool": (C.c_int, [C.POINTER(EmbedTap), C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                C.POINTER(C.c_size_t), C.c_void_p]),
    "yl_cocoeval_evaluate": (C.c_int, [C.POINTER(CocoevalSet), C.POINTER(CocoevalParams), C.POINTER(CocoevalSlots),
                                       C.c_void_p]),
    "yl_cocoeval_accumulate": (C.c_int, [C.POINTER(CocoevalParams), C.c_int, C.c_int] + [C.c_void_p] * 9),
}

EXPORTS = tuple(_PROTOTYPES)


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """dlopen libyl11.so and attach prototypes (no GPU needed)."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise YLError(
                f"{_LIB_PATH} is missing: build it with `python yolo-lite_b200/csrc/build.py` "
                "(yololite has no CPU or library fallback)"
            )
        lib = C.CDLL(str(_LIB_PATH))
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def available() -> bool:
    return _LIB_PATH.exists() and torch.cuda.is_available()


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load().yl_last_error_string().decode("utf-8", "replace")
        raise YLError(f"{what or 'libyl11'} failed ({rc}): {msg}")


def init(device: int | torch.device | None = None):
    """Bind the library to a CUDA device (idempotent per device). Raises when there is no B200."""
    lib = load()
    if not torch.cuda.is_available():
        raise YLError("CUDA is not available: yololite runs on sm_100 GPUs only (no CPU fallback)")
    if device is None:
        device = torch.cuda.current_device()
    if isinstance(device, torch.device):
        device = device.index if device.index is not None else torch.cuda.current_device()
    device = int(device)
    if device not in _inited_devices:
        torch.cuda.init()
        with torch.cuda.device(device):
            check(lib.yl_init(device), "yl_init")
        _inited_devices.add(device)
    return lib


def stream_ptr(stream: torch.cuda.Stream | None = None) -> int:
    s = stream if stream is not None else torch.cuda.current_stream()
    return int(s.cuda_stream)


def view(buf: torch.Tensor, n: int, h: int, w: int, c: int, coff: int = 0) -> Tensor:
    """Describe channels [coff, coff+c) of an NHWC buffer `buf` of shape (n, h, w, cstride)."""
    assert buf.is_cuda and buf.is_contiguous() and buf.dim() == 4, "expected a contiguous NHWC CUDA buffer"
    assert buf.shape[0] == n and buf.shape[1] == h and buf.shape[2] == w, (tuple(buf.shape), n, h, w)
    if buf.dtype == torch.bfloat16:
        dt = YL_BF16
    elif buf.dtype == torch.float32:
        dt = YL_F32
    else:
        raise TypeError(f"unsupported buffer dtype {buf.dtype}")
    assert coff + c <= buf.shape[3]
    return Tensor(buf.data_ptr(), n, h, w, c, buf.shape[3], coff, dt, 0)


def null_tensor() -> Tensor:
    return Tensor(None, 0, 0, 0, 0, 0, 0, 0, 0)
