"""Inference configuration: the keys of the reference's cfg/default.yaml that the predict/val path reads,
with the same names, defaults and override semantics (`get_cfg(overrides=...)`, reference cfg/__init__.py:125-179).
Unknown keys raise (the reference raises SyntaxError with suggestions, cfg/__init__.py:219-249); training keys
are accepted and ignored so dictionaries written for the reference keep working.
"""
from __future__ import annotations

from difflib import get_close_matches
from pathlib import Path
from types import SimpleNamespace

CFG_DIR = Path(__file__).resolve().parent

# key: default  (reference cfg/default.yaml; only inference-relevant keys are acted upon)
DEFAULT_CFG_DICT = {
    "task": "detect", "mode": "predict", "model": None, "data": None, "imgsz": 640, "batch": 16, "device": None,
    "verbose": True, "half": False, "dnn": False, "rect": False, "project": None, "name": None, "exist_ok": False,
    "conf": None, "iou": 0.7, "max_det": 300, "classes": None, "agnostic_nms": False, "augment": False,
    "visualize": False, "embed": None, "source": None, "vid_stride": 1, "stream_buffer": False,
    "save": False, "save_txt": False, "save_conf": False, "save_crop": False, "save_json": False,
    "save_hybrid": False, "show": False, "show_labels": True, "show_conf": True, "show_boxes": True,
    "line_width": None, "plots": False, "single_cls": False, "split": "val", "workers": 0, "retina_masks": False,
}
# accepted-but-ignored (training) keys of the reference's default.yaml
_IGNORED = {
    "epochs", "time", "patience", "cache", "pretrained", "optimizer", "seed", "deterministic", "cos_lr",
    "close_mosaic", "resume", "amp", "fraction", "profile", "freeze", "multi_scale", "overlap_mask", "mask_ratio",
    "dropout", "val", "lr0", "lrf", "momentum", "weight_decay", "warmup_epochs", "warmup_momentum", "warmup_bias_lr",
    "box", "cls", "dfl", "pose", "kobj", "label_smoothing", "nbs", "hsv_h", "hsv_s", "hsv_v", "degrees", "translate",
    "scale", "shear", "perspective", "flipud", "fliplr", "bgr", "mosaic", "mixup", "copy_paste", "copy_paste_mode",
    "auto_augment", "erasing", "crop_fraction", "cfg", "tracker", "save_period", "save_frames", "save_dir",
    "format", "keras", "optimize", "int8", "dynamic", "simplify", "opset", "workspace", "nms",
}
DEFAULT_CFG_KEYS = tuple(DEFAULT_CFG_DICT)
DEFAULT_CFG = SimpleNamespace(**DEFAULT_CFG_DICT)

_FRACTION = {"conf", "iou"}
_INT = {"max_det", "vid_stride", "workers", "batch"}
_BOOL = {"half", "dnn", "rect", "agnostic_nms", "augment", "visualize", "save", "save_txt", "save_conf", "save_crop",
         "save_json", "save_hybrid", "show", "verbose", "plots", "single_cls", "stream_buffer"}


def get_save_dir(args) -> Path:
    """Output directory of a run (reference cfg/__init__.py get_save_dir): `<project or runs/<task>>/<name or mode>`,
    numbered `val2`, `val3`, ... when it exists, unless `exist_ok`.  Not created here."""
    path = Path(args.project or Path("runs") / args.task) / (args.name or f"{args.mode}")
    if path.exists() and not args.exist_ok:
        for n in range(2, 9999):
            p = Path(f"{path}{n}")
            if not p.exists():
                break
        path = p
    return path


def get_cfg(cfg=DEFAULT_CFG, overrides=None) -> SimpleNamespace:
    """Merge `overrides` into the defaults with the reference's type/range checks."""
    base = dict(vars(cfg)) if isinstance(cfg, SimpleNamespace) else dict(cfg or DEFAULT_CFG_DICT)
    for k, v in (overrides or {}).items():
        if k in _IGNORED:
            continue
        if k not in DEFAULT_CFG_DICT:
            hint = get_close_matches(k, list(DEFAULT_CFG_DICT) + sorted(_IGNORED), n=3)
            raise SyntaxError(f"'{k}' is not a valid yololite argument." + (f" Similar arguments: {hint}" if hint else ""))
        base[k] = v
    for k, v in base.items():
        if v is None:
            continue
        if k in _FRACTION:
            if not isinstance(v, (int, float)):
                raise TypeError(f"'{k}={v}' must be a float in [0, 1]")
            if not 0.0 <= v <= 1.0:
                raise ValueError(f"'{k}={v}' is out of range, must be in [0.0, 1.0]")
        elif k in _INT and (not isinstance(v, int) or isinstance(v, bool)):
            raise TypeError(f"'{k}={v}' must be an int")
        elif k in _BOOL and not isinstance(v, bool):
            raise TypeError(f"'{k}={v}' must be a bool")
    return SimpleNamespace(**base)
