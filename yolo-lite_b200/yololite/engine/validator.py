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

`save_json=True` follows upstream `pred_to_json` / `eval_json`: every image's rescaled detections become COCO result
rows (one extra device read of the batch's detections), written to `<save_dir>/predictions.json` at the end of the run.
When the data yaml names COCO val2017 and `<path>/annotations/instances_val2017.json` exists, the file is scored with
`utils.cocoeval.COCOeval` (pycocotools' bbox evaluation, on the GPU) and `metrics/mAP50-95(B)` / `metrics/mAP50(B)` of
the returned stats become its `stats[0]` / `stats[1]`; the evaluator stays on `validator.coco_eval`.

Dataset construction (data/build.py, data/dataset.py, augmentations, caching) is training-side I/O and out of scope:
pass `dataloader=` (any iterable of batch dicts) instead of a dataset yaml."""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np
import torch

from .. import _C
from ..cfg import DEFAULT_CFG, get_cfg, get_save_dir
from ..utils import LOGGER, ops
from ..utils.metrics import ConfusionMatrix, DetMetrics, match_predictions_batched
from ..utils.torch_utils import select_device, smart_inference_mode


class DetectionValidator:
    def __init__(self, dataloader=None, save_dir=None, pbar=None, args=None, _callbacks=None):
        self.args = get_cfg(DEFAULT_CFG, args)
        self.dataloader = dataloader
        self.save_dir = Path(save_dir) if save_dir else None
        if self.args.conf is None:
            self.args.conf = 0.001                      # reference validator.py:60
        self.args.task = "detect"
        self.args.mode = "val"
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
        self.jdict, self.json_files = [], []   # save_json: COCO result rows, files of the evaluated images
        self.is_coco, self.class_map, self.coco_eval = False, None, None
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
        self.jdict, self.json_files = [], []
        if self.args.save_json:
            self.is_coco = self._coco_annotations() is not None
            self.class_map = ops.coco80_to_coco91_class() if self.is_coco else list(range(1, self.nc + 1))

    def _coco_annotations(self):
        """`<path>/annotations/instances_val2017.json` when the data yaml's split is COCO val2017 (`val2017.txt` or a
        `val2017` image directory) and the file exists, else None."""
        data = self.args.data
        if not data or Path(str(data)).suffix not in {".yaml", ".yml"}:
            return None
        from ..data.dataset import load_data_yaml

        d = load_data_yaml(data)
        split = str(d.get(self.args.split) or "").rstrip("/")
        anno = d["path"] / "annotations" / "instances_val2017.json"
        return anno if (split.endswith("val2017.txt") or Path(split).name == "val2017") and anno.is_file() else None

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
        if self.args.save_json:
            predn_host = predn.cpu()                      # save_json's one extra read of the batch
            for si in range(B):
                self.json_files.append(batch["im_file"][si])
                if n[si]:
                    self.pred_to_json(predn_host[si, : n[si]], batch["im_file"][si])
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

    def pred_to_json(self, predn, filename):
        """Append one image's COCO result rows (upstream pred_to_json): predn (n, 6) host fp32 [x1, y1, x2, y2, conf,
        cls] in original-image pixels -> top-left xywh in fp32, each value through Python's round()."""
        stem = Path(filename).stem
        image_id = int(stem) if stem.isnumeric() else stem
        box = ops.xyxy2xywh(predn[:, :4])
        box[:, :2] -= box[:, 2:] / 2
        for p, b in zip(predn.tolist(), box.tolist()):
            self.jdict.append({"image_id": image_id, "category_id": self.class_map[int(p[5])],
                               "bbox": [round(x, 3) for x in b], "score": round(p[4], 5)})

    def eval_json(self, stats):
        """Score predictions.json with COCOeval on the GPU (COCO val2017 layouts only, upstream eval_json)."""
        anno_json = self._coco_annotations() if self.is_coco else None
        if anno_json is not None and len(self.jdict):
            from ..utils.cocoeval import COCO, COCOeval

            pred_json = self.save_dir / "predictions.json"
            LOGGER.info(f"\nEvaluating pycocotools mAP using {pred_json} and {anno_json}...")
            try:
                for x in pred_json, anno_json:
                    assert x.is_file(), f"{x} file not found"
                anno = COCO(str(anno_json))
                pred = anno.loadRes(str(pred_json))
                val = COCOeval(anno, pred, "bbox")
                val.params.imgIds = [int(Path(x).stem) for x in self.json_files]
                val.evaluate()
                val.accumulate()
                val.summarize()
                self.coco_eval = val
                stats[self.metrics.keys[-1]], stats[self.metrics.keys[-2]] = val.stats[:2]
            except Exception as e:
                LOGGER.warning(f"pycocotools unable to run: {e}")
        return stats

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
        if self.args.save_json and self.jdict:
            self.save_dir = self.save_dir or get_save_dir(self.args)
            self.save_dir.mkdir(parents=True, exist_ok=True)
            with open(str(self.save_dir / "predictions.json"), "w") as f:
                LOGGER.info(f"Saving {f.name}...")
                json.dump(self.jdict, f)
            stats = self.eval_json(stats)
        return stats
