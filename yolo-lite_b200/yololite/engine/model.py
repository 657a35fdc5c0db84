"""YOLOLite facade (reference yololite/engine/model.py:17-146): `YOLOLite("yolo11n.pt" | "yolo11n.yaml" | [a.pt, b.pt])`
(a list of checkpoints is a model ensemble), `model(source)`, `.predict(source, stream=False, **kwargs)`,
`.val(**kwargs)`.  Training is out of scope."""
from __future__ import annotations

from pathlib import Path
from typing import Union

import torch.nn as nn

from ..nn.tasks import _ENSEMBLE_NO_EMBED, DetectionModel, Ensemble, attempt_load_one_weight, attempt_load_weights, \
    yaml_model_load
from .predictor import DetectionPredictor


class YOLOLite(nn.Module):
    def __init__(self, model: Union[str, Path] = "yolo11n.pt", task: str = None, verbose: bool = False) -> None:
        super().__init__()
        self.callbacks = None
        self.predictor = None
        self.model = None
        self.trainer = None
        self.ckpt = None
        self.cfg = None
        self.ckpt_path = None
        self.overrides = {}
        self.metrics = None
        self.task = task
        if isinstance(model, (list, tuple)) and len(model) > 1:
            self._load_ensemble([str(w).strip() for w in model])
            return
        model = str(model[0] if isinstance(model, (list, tuple)) else model).strip()
        if Path(model).suffix in {".yaml", ".yml"}:
            self._new(model, task=task, verbose=verbose)
        else:
            self._load(model)

    def __call__(self, source=None, stream: bool = False, **kwargs) -> list:
        return self.predict(source, stream, **kwargs)

    def _new(self, cfg: str, task=None, verbose=False) -> None:
        cfg_dict = yaml_model_load(cfg)
        self.cfg = cfg
        self.task = task or "detect"
        self.model = DetectionModel(cfg_dict, verbose=verbose)
        self.overrides["model"] = self.cfg
        self.overrides["task"] = self.task
        self.model.args = {**self.overrides}
        self.model.task = self.task
        self.model_name = cfg

    def _load(self, weights: str) -> None:
        self.model, self.ckpt = attempt_load_one_weight(weights)
        self.task = self.model.args.get("task", "detect")
        self.overrides = self.model.args = {k: v for k, v in self.model.args.items()
                                            if k in {"imgsz", "data", "task", "single_cls"}}
        self.ckpt_path = self.model.pt_path
        self.overrides["model"] = weights
        self.overrides["task"] = self.task
        self.model_name = weights

    def _load_ensemble(self, weights: list) -> None:
        """Checkpoints loaded as one Ensemble (attempt_load_weights); overrides and ckpt_path come from member 0."""
        self.model = attempt_load_weights(weights)
        first = self.model[0]
        self.task = first.args.get("task", "detect")
        self.overrides = self.model.args = {k: v for k, v in first.args.items() if k in {"imgsz", "data", "task", "single_cls"}}
        self.ckpt_path = first.pt_path
        self.overrides["model"] = weights
        self.overrides["task"] = self.task
        self.model_name = weights

    def predict(self, source=None, stream: bool = False, **kwargs):
        """Same defaults as the reference (conf=0.25, batch=1, mode=predict); `save` defaults to False here
        because writing annotated images is outside the scope (the reference injects save=True, model.py:95)."""
        custom = {"conf": 0.25, "batch": 1, "mode": "predict"}
        args = {**self.overrides, **custom, **kwargs}
        if self.predictor is None or kwargs.get("_new_predictor", True):
            args.pop("_new_predictor", None)
            predictor = DetectionPredictor(overrides=args)
            if self.predictor is not None and self.predictor.model is not None:
                predictor.model, predictor.device = self.predictor.model, self.predictor.device   # keep plans warm
            else:
                predictor.setup_model(model=self.model, verbose=False)
                self.model = predictor.model.model
            self.predictor = predictor
        return self.predictor(source=source, stream=stream)

    def embed(self, source=None, stream: bool = False, **kwargs):
        """Image feature vectors (reference Model.embed): `predict` with `embed` defaulting to the last layer before the
        head (22 for YOLO11; 256 values per image for yolo11n).  Yields / returns one 1-D fp32 tensor per image.
        TypeError for a model ensemble (its members share no feature space)."""
        if isinstance(self.model, Ensemble):
            raise TypeError(_ENSEMBLE_NO_EMBED)
        if not kwargs.get("embed"):
            kwargs["embed"] = [len(self.model.model) - 2]
        return self.predict(source, stream, **kwargs)

    def val(self, dataloader=None, **kwargs):
        """Validate on labelled batches (reference engine/model.py:101-107).  `dataloader`: iterable of batch dicts in
        the reference's collate layout; or `data=<dataset yaml | image dir>`: the split is loaded with the minimal rect
        loader (`yololite.data.RectValLoader`, the reference's `YOLODataset(rect=True)` batches)."""
        from .validator import DetectionValidator

        custom = {"rect": True}
        args = {**self.overrides, **custom, **kwargs, "mode": "val"}
        if dataloader is None and kwargs.get("data"):
            from ..data import build_val_loader

            stride = int(self.model.stride.max()) if hasattr(self.model, "stride") else 32
            imgsz = args.get("imgsz") or 640
            dataloader, names = build_val_loader(kwargs["data"], imgsz=int(imgsz if isinstance(imgsz, int) else imgsz[0]),
                                                 batch_size=int(args.get("batch") or 16), stride=max(stride, 32),
                                                 split=args.get("split") or "val")
            if names and len(names) == len(self.model.names):
                self.model.names = dict(names) if isinstance(names, dict) else dict(enumerate(names))
        validator = DetectionValidator(dataloader=dataloader, args=args)
        validator(model=self.model)
        self.metrics = validator.metrics
        return validator.metrics

    def train(self, **kwargs):
        raise NotImplementedError("training is outside yololite's scope (YOLO11 *inference* hot path only)")
