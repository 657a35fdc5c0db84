"""DetectionValidator (reference yololite/engine/validator.py:21-470): runs the hot path over labelled batches and
accumulates detection metrics.  What is kept: the stage names (`preprocess / postprocess / init_metrics /
update_metrics / get_stats / finalize_metrics`), the batch dict layout of the reference's collate function
(`img, cls, bboxes (normalised xywh), batch_idx, ori_shape, ratio_pad, im_file`), the val defaults (conf 0.001,
iou 0.7, max_det 300, multi_label NMS) and the `stats` / `DetMetrics` outputs.  What changed: prediction rescale,
label preparation and `box_iou + match_predictions` (a per-image torch/numpy loop in the reference, :313-360) run
batched on the GPU (`yl_scale_boxes`, `yl_match_predictions`); one host read per batch.

Two switches of the reference are kept: `save_hybrid=True` passes each image's ground-truth labels to NMS as priors
(hybrid metrics, inflated by construction), `plots=True` accumulates a `ConfusionMatrix` (`yl_confusion_matrix`, one
launch per batch), exposed as `validator.confusion_matrix` and `metrics.confusion_matrix`.  Neither launches or
allocates anything while it is off.

Dataset construction (data/build.py, data/dataset.py, augmentations, caching) is training-side I/O and out of scope:
pass `dataloader=` (any iterable of batch dicts) instead of a dataset yaml."""
from __future__ import annotations

import numpy as np
import torch

from .. import _C
from ..cfg import DEFAULT_CFG, get_cfg
from ..utils import LOGGER, ops
from ..utils.metrics import ConfusionMatrix, DetMetrics, match_predictions_batched
from ..utils.torch_utils import select_device, smart_inference_mode


class DetectionValidator:
    def __init__(self, dataloader=None, save_dir=None, pbar=None, args=None, _callbacks=None):
        self.args = get_cfg(DEFAULT_CFG, args)
        self.dataloader = dataloader
        if self.args.conf is None:
            self.args.conf = 0.001                      # reference validator.py:60
        self.args.task = "detect"
        self.device = None
        self.names, self.nc, self.seen = None, None, 0
        self.iouv = torch.linspace(0.5, 0.95, 10)       # mAP@0.5:0.95
        self.niou = self.iouv.numel()
        self.metrics = DetMetrics()
        self.stats = None
        self.speed = {"preprocess": 0.0, "inference": 0.0, "loss": 0.0, "postprocess": 0.0}
        self.confusion_matrix = None
        self.lb = None              # save_hybrid priors of the current batch (packed for ops.nms_padded)
        self._layout = None         # (label order, offsets) of the current batch
        if self.args.save_hybrid:   # reference DetectionValidator.__init__
            LOGGER.warning("WARNING 'save_hybrid=True' will append ground truth to predictions for autolabelling.\n"
                           "WARNING 'save_hybrid=True' will cause incorrect mAP.\n")

    # ------------------------------------------------------------------ stages
    def preprocess(self, batch):
        """uint8 / float image batch -> float [0, 1] on the device (reference :262-266 divides by 255).  With
        save_hybrid, the priors: each image's labels in their original order, boxes `bboxes * (w, h, w, h)` of the
        network input, built where the loader left them (on the host for a CPU loader, so no device read)."""
        self._layout = None
        if self.args.save_hybrid:
            h, w = batch["img"].shape[2:]
            order, offsets = self._label_layout(batch)
            bboxes = batch["bboxes"].view(-1, 4)[order].float()
            self.lb = (bboxes * torch.tensor((w, h, w, h), device=bboxes.device), batch["cls"].view(-1)[order], offsets)
        img = batch["img"].to(self.device, non_blocking=True)
        batch["img"] = img.float() / 255 if img.dtype == torch.uint8 else img.float()
        for k in ("batch_idx", "cls", "bboxes"):
            batch[k] = batch[k].to(self.device)
        return batch

    def postprocess(self, preds):
        """Batched NMS with the validator's settings (multi_label, reference :280-290); device-resident."""
        a = self.args
        return ops.nms_padded(preds, a.conf, a.iou, None, a.single_cls or a.agnostic_nms, True, a.max_det,
                              labels=self.lb if a.save_hybrid else None)

    def init_metrics(self, model):
        self.names = model.names
        self.nc = len(model.names)
        self.metrics = DetMetrics(names=self.names)
        self.seen = 0
        self.stats = dict(tp=[], conf=[], pred_cls=[], target_cls=[], target_img=[])
        self.confusion_matrix = ConfusionMatrix(nc=self.nc, conf=self.args.conf) if self.args.plots else None

    def _label_layout(self, batch):
        """Stable image-major order of the batch's labels and the B + 1 per-image offsets, once per batch."""
        if self._layout is None:
            bi = batch["batch_idx"].long().view(-1)
            counts = torch.bincount(bi, minlength=batch["img"].shape[0])
            self._layout = (torch.argsort(bi, stable=True), [0] + torch.cumsum(counts, 0).tolist())
        return self._layout

    def _labels_native(self, batch):
        """Labels of the whole batch in original-image pixels (reference _prepare_batch :234-246), image-major."""
        B = batch["img"].shape[0]
        h, w = batch["img"].shape[2:]
        order, offsets = self._label_layout(batch)
        order = order.to(self.device)
        cls = batch["cls"].view(-1)[order].float()
        box = ops.xywh2xyxy(batch["bboxes"].view(-1, 4)[order].float()) * torch.tensor([w, h, w, h], device=self.device)
        for si in range(B):                               # labels are few: the reference's own helper, per image
            s, e = offsets[si], offsets[si + 1]
            if e > s:
                ops.scale_boxes((h, w), box[s:e], batch["ori_shape"][si], ratio_pad=batch["ratio_pad"][si])
        return box, cls, offsets

    def update_metrics(self, preds, batch):
        dets, counts = preds
        B, max_det, _ = dets.shape
        h, w = batch["img"].shape[2:]
        # predictions -> original-image space, all images in one launch (reference _prepare_pred :248-254)
        params = np.empty((B, 5), np.float32)
        for i in range(B):
            s0 = batch["ori_shape"][i]
            gain, pad = ops.letterbox_params((h, w), s0, batch["ratio_pad"][i])
            params[i] = (gain, pad[0], pad[1], s0[1], s0[0])
        predn = dets.clone()
        if self.args.single_cls:
            predn[..., 5] = 0
        pd = torch.from_numpy(params).to(self.device)
        _C.check(_C.load().yl_scale_boxes(predn.data_ptr(), counts.data_ptr(), B, max_det, pd.data_ptr(), _C.stream_ptr()),
                 "yl_scale_boxes")
        gt_box, gt_cls, offsets = self._labels_native(batch)
        tp = match_predictions_batched(predn, counts, gt_box, gt_cls, offsets, self.iouv)
        if self.confusion_matrix is not None:
            self.confusion_matrix.process_batched(predn, counts, gt_box, gt_cls, offsets)
        n = counts.tolist()                               # the one host read of the batch
        for si in range(B):
            self.seen += 1
            s, e = offsets[si], offsets[si + 1]
            cls = gt_cls[s:e]
            if n[si] == 0 and e == s:
                continue
            self.stats["tp"].append(tp[si, : n[si]])
            self.stats["conf"].append(predn[si, : n[si], 4])
            self.stats["pred_cls"].append(predn[si, : n[si], 5])
            self.stats["target_cls"].append(cls)
            self.stats["target_img"].append(cls.unique())

    def get_stats(self):
        stats = {k: (torch.cat(v, 0).cpu().numpy() if v else np.zeros((0, self.niou) if k == "tp" else (0,)))
                 for k, v in self.stats.items()}
        self.nt_per_class = np.bincount(stats["target_cls"].astype(int), minlength=self.nc)
        self.nt_per_image = np.bincount(stats["target_img"].astype(int), minlength=self.nc)
        stats.pop("target_img", None)
        if len(stats) and stats["tp"].any():
            self.metrics.process(**stats)
        return self.metrics.results_dict

    def finalize_metrics(self):
        self.metrics.speed = self.speed
        if self.confusion_matrix is not None:
            self.confusion_matrix.matrix   # the one host read of the accumulated counts
        self.metrics.confusion_matrix = self.confusion_matrix

    def print_results(self):
        pf = "%22s" + "%11i" * 2 + "%11.3g" * len(self.metrics.keys)
        LOGGER.info(pf % ("all", self.seen, self.nt_per_class.sum(), *self.metrics.mean_results()))

    # ------------------------------------------------------------------ driver
    @smart_inference_mode()
    def __call__(self, trainer=None, model=None):
        if trainer is not None:
            raise NotImplementedError("validation inside a training loop is out of scope (inference path only)")
        if self.dataloader is None:
            raise NotImplementedError(
                "dataset loading from a data yaml (data/build.py, data/dataset.py) is outside yololite's scope: "
                "construct DetectionValidator(dataloader=<iterable of batch dicts>, args=...)")
        self.device = select_device(self.args.device)
        model = model.to(self.device).eval()
        self.init_metrics(model)
        for batch in self.dataloader:
            batch = self.preprocess(batch)
            y, _ = model.infer(batch["img"], augment=self.args.augment)
            preds = self.postprocess(y)
            self.update_metrics(preds, batch)
        stats = self.get_stats()
        self.finalize_metrics()
        if self.args.verbose:
            self.print_results()
        return stats
