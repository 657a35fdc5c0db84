"""Detection metrics of the validator (reference yololite/utils/metrics.py: box_iou :51-70, ConfusionMatrix,
compute_ap :445-474, ap_per_class :477-564, Metric :567-736, DetMetrics :739-840; engine/validator.py
match_predictions :195-233).

`box_iou` + `match_predictions` — the per-image torch/numpy loop of the reference's `update_metrics` — run as ONE
CUDA kernel over the whole batch (`match_predictions_batched`, csrc/metrics.cu) on the padded NMS output;
`ap_per_class` stays numpy on the host (it runs once per validation, on a few thousand rows).  The validator's
`ConfusionMatrix` (plots=True) is a metric too: its per-image `process_batch` runs as one CUDA kernel per batch
(`yl_confusion_matrix`) into a device-resident integer matrix that the host reads once.  Drawing plots and JSON
export are visualisation / I-O and out of scope."""
from __future__ import annotations

import numpy as np
import torch

__all__ = ("box_iou", "match_predictions_batched", "ConfusionMatrix", "compute_ap", "ap_per_class", "Metric",
           "DetMetrics", "smooth")


def box_iou(box1: torch.Tensor, box2: torch.Tensor, eps: float = 1e-7) -> torch.Tensor:
    """Pairwise IoU of (N, 4) and (M, 4) xyxy boxes -> (N, M), fp32."""
    a1, a2 = box1.float()[:, None, :2], box1.float()[:, None, 2:]
    b1, b2 = box2.float()[None, :, :2], box2.float()[None, :, 2:]
    inter = (torch.min(a2, b2) - torch.max(a1, b1)).clamp_(0).prod(2)
    return inter / ((a2 - a1).prod(2) + (b2 - b1).prod(2) - inter + eps)


def match_predictions_batched(dets: torch.Tensor, counts: torch.Tensor, gt_boxes: torch.Tensor, gt_cls: torch.Tensor,
                              gt_offsets, iouv: torch.Tensor) -> torch.Tensor:
    """True-positive matrix of a whole batch on the GPU.

    dets (B, max_det, 6) fp32 + counts (B,) int32: padded NMS output, boxes already in the labels' space;
    gt_boxes (L, 4) xyxy, gt_cls (L,): labels of all images back to back; gt_offsets: B + 1 ints;
    iouv: (n,) thresholds.  Returns (B, max_det, n) bool; rows >= counts[b] are False."""
    from .. import _C

    if not dets.is_cuda:
        raise RuntimeError("match_predictions_batched runs on CUDA (sm_100) only; there is no CPU fallback")
    lib = _C.init(dets.device)
    B, max_det, _ = dets.shape
    dev = dets.device
    offs = torch.as_tensor(list(gt_offsets), dtype=torch.int32)
    assert offs.numel() == B + 1
    max_l = int((offs[1:] - offs[:-1]).max()) if B else 0
    offs = offs.to(dev)
    gtb = gt_boxes.to(dev, torch.float32).contiguous().view(-1, 4)
    gtc = gt_cls.to(dev, torch.float32).contiguous().view(-1)
    thr = iouv.to(dev, torch.float32).contiguous()
    tp = torch.empty((B, max_det, thr.numel()), dtype=torch.uint8, device=dev)
    d = dets if (dets.dtype == torch.float32 and dets.is_contiguous()) else dets.float().contiguous()
    c = counts.to(dev, torch.int32).contiguous()
    _C.check(lib.yl_match_predictions(d.data_ptr(), c.data_ptr(), B, max_det, gtb.data_ptr() if gtb.numel() else None,
                                      gtc.data_ptr() if gtc.numel() else None, offs.data_ptr(), max_l, thr.data_ptr(),
                                      thr.numel(), tp.data_ptr(), _C.stream_ptr()), "yl_match_predictions")
    return tp.bool()


class ConfusionMatrix:
    """Detection confusion matrix (reference utils/metrics.py ConfusionMatrix, task "detect").

    `matrix` is (nc+1, nc+1) float64 indexed [predicted, true]; index nc is background.  Detections count when
    conf > `conf` (0.25 when given None or the validator's default 0.001), pairs when IoU > `iou_thres`.  Counts
    accumulate on the GPU (`process_batch` per image, `process_batched` per validator batch) and are folded into
    `matrix` on the first read after them."""

    def __init__(self, nc, conf=0.25, iou_thres=0.45, task="detect"):
        if task != "detect":
            raise NotImplementedError(f"ConfusionMatrix task {task!r}: only detection is on the GPU path")
        self.task = task
        self.nc = nc
        self.conf = 0.25 if conf in {None, 0.001} else conf
        self.iou_thres = iou_thres
        self._matrix = np.zeros((nc + 1, nc + 1))
        self._counts = None   # device int64[(nc+1)^2 + 1] accumulator; the last element counts out-of-range classes

    @property
    def matrix(self) -> np.ndarray:
        if self._counts is not None:   # the one host read of the accumulated batches
            c = self._counts.cpu().numpy()
            self._counts = None
            if c[-1]:
                raise ValueError(f"ConfusionMatrix: {int(c[-1])} class ids outside [0, {self.nc}]")
            self._matrix += c[:-1].reshape(self.nc + 1, self.nc + 1)
        return self._matrix

    @matrix.setter
    def matrix(self, value):
        self._counts = None
        self._matrix = np.asarray(value, dtype=np.float64)

    def process_batched(self, dets, counts, gt_boxes, gt_cls, gt_offsets):
        """A whole batch in one launch, the layout of `match_predictions_batched`: dets (B, max_det, 6) + counts (B,)
        on the GPU (boxes in the labels' space), gt_boxes (L, 4) xyxy, gt_cls (L,), gt_offsets B + 1 host ints."""
        from .. import _C

        if not dets.is_cuda:
            raise RuntimeError("ConfusionMatrix runs on CUDA (sm_100) only; there is no CPU fallback")
        lib = _C.init(dets.device)
        dev = dets.device
        B, max_det, _ = dets.shape
        offs = [int(o) for o in gt_offsets]
        assert len(offs) == B + 1
        max_l = max(e - s for s, e in zip(offs[:-1], offs[1:]))
        offs_t = torch.as_tensor(offs, dtype=torch.int32).to(dev)
        gtb = gt_boxes.to(dev, torch.float32).contiguous().view(-1, 4)
        gtc = gt_cls.to(dev, torch.float32).contiguous().view(-1)
        d = dets if (dets.dtype == torch.float32 and dets.is_contiguous()) else dets.float().contiguous()
        c = counts.to(dev, torch.int32).contiguous()
        if self._counts is None:
            self._counts = torch.zeros((self.nc + 1) ** 2 + 1, dtype=torch.int64, device=dev)
        _C.check(lib.yl_confusion_matrix(d.data_ptr(), c.data_ptr(), B, max_det, gtb.data_ptr() if gtb.numel() else None,
                                         gtc.data_ptr() if gtc.numel() else None, offs_t.data_ptr(), max_l, self.nc,
                                         float(self.conf), float(self.iou_thres), self._counts.data_ptr(),
                                         _C.stream_ptr()), "yl_confusion_matrix")

    def process_batch(self, detections, gt_bboxes, gt_cls):
        """One image, the reference's signature: detections (N, 6) [x1, y1, x2, y2, conf, cls] or None, gt_bboxes
        (M, 4) xyxy, gt_cls (M,)."""
        dev = gt_bboxes.device if detections is None else detections.device
        n = 0 if detections is None else detections.shape[0]
        dets = torch.zeros((1, max(n, 1), 6), dtype=torch.float32, device=dev)
        if n:
            dets[0, :n] = detections[:, :6].float()
        counts = torch.tensor([n], dtype=torch.int32).to(dev)
        self.process_batched(dets, counts, gt_bboxes, gt_cls, [0, gt_cls.shape[0]])

    def tp_fp(self):
        """True and false positives per class (background excluded)."""
        tp = self.matrix.diagonal()
        fp = self.matrix.sum(1) - tp
        return tp[:-1], fp[:-1]

    def plot(self, normalize=True, save_dir="", names=(), on_plot=None):
        from . import LOGGER

        LOGGER.info("ConfusionMatrix.plot: drawing plots is outside yololite's scope; read `.matrix` instead")


def smooth(y, f=0.05):
    """Box filter of fraction f (reference metrics.py:387-393)."""
    nf = round(len(y) * f * 2) // 2 + 1
    p = np.ones(nf // 2)
    yp = np.concatenate((p * y[0], y, p * y[-1]), 0)
    return np.convolve(yp, np.ones(nf) / nf, mode="valid")


def compute_ap(recall, precision):
    """101-point interpolated AP (COCO) of one PR curve; returns (ap, precision envelope, recall with sentinels)."""
    mrec = np.concatenate(([0.0], recall, [1.0]))
    mpre = np.concatenate(([1.0], precision, [0.0]))
    mpre = np.flip(np.maximum.accumulate(np.flip(mpre)))
    x = np.linspace(0, 1, 101)
    trapz = getattr(np, "trapezoid", None) or np.trapz
    ap = trapz(np.interp(x, mrec, mpre), x)
    return ap, mpre, mrec


def ap_per_class(tp, conf, pred_cls, target_cls, eps=1e-16):
    """Per-class AP at every IoU threshold + P/R/F1 at the max-F1 confidence (reference metrics.py:477-564)."""
    order = np.argsort(-conf)
    tp, conf, pred_cls = tp[order], conf[order], pred_cls[order]
    unique_classes, nt = np.unique(target_cls, return_counts=True)
    nc = unique_classes.shape[0]
    x, prec_values = np.linspace(0, 1, 1000), []
    ap, p_curve, r_curve = np.zeros((nc, tp.shape[1])), np.zeros((nc, 1000)), np.zeros((nc, 1000))
    for ci, c in enumerate(unique_classes):
        sel = pred_cls == c
        n_l, n_p = nt[ci], sel.sum()
        if n_p == 0 or n_l == 0:
            continue
        fpc = (1 - tp[sel]).cumsum(0)
        tpc = tp[sel].cumsum(0)
        recall = tpc / (n_l + eps)
        r_curve[ci] = np.interp(-x, -conf[sel], recall[:, 0], left=0)
        precision = tpc / (tpc + fpc)
        p_curve[ci] = np.interp(-x, -conf[sel], precision[:, 0], left=1)
        for j in range(tp.shape[1]):
            ap[ci, j], mpre, mrec = compute_ap(recall[:, j], precision[:, j])
            if j == 0:
                prec_values.append(np.interp(x, mrec, mpre))
    prec_values = np.array(prec_values)
    f1_curve = 2 * p_curve * r_curve / (p_curve + r_curve + eps)
    i = smooth(f1_curve.mean(0), 0.1).argmax()
    p, r, f1 = p_curve[:, i], r_curve[:, i], f1_curve[:, i]
    tp_n = (r * nt).round()
    fp_n = (tp_n / (p + eps) - tp_n).round()
    return tp_n, fp_n, p, r, f1, ap, unique_classes.astype(int), p_curve, r_curve, f1_curve, x, prec_values


class Metric:
    """P / R / F1 / AP container with the reference's accessors (metrics.py:567-736)."""

    def __init__(self) -> None:
        self.p, self.r, self.f1, self.all_ap, self.ap_class_index, self.nc = [], [], [], [], [], 0

    @property
    def ap50(self):
        return self.all_ap[:, 0] if len(self.all_ap) else []

    @property
    def ap(self):
        return self.all_ap.mean(1) if len(self.all_ap) else []

    @property
    def mp(self):
        return self.p.mean() if len(self.p) else 0.0

    @property
    def mr(self):
        return self.r.mean() if len(self.r) else 0.0

    @property
    def map50(self):
        return self.all_ap[:, 0].mean() if len(self.all_ap) else 0.0

    @property
    def map75(self):
        return self.all_ap[:, 5].mean() if len(self.all_ap) else 0.0

    @property
    def map(self):
        return self.all_ap.mean() if len(self.all_ap) else 0.0

    def mean_results(self):
        return [self.mp, self.mr, self.map50, self.map]

    def class_result(self, i):
        return self.p[i], self.r[i], self.ap50[i], self.ap[i]

    @property
    def maps(self):
        maps = np.zeros(self.nc) + self.map
        for i, c in enumerate(self.ap_class_index):
            maps[c] = self.ap[i]
        return maps

    def fitness(self):
        w = [0.0, 0.0, 0.1, 0.9]
        return (np.array(self.mean_results()) * w).sum()

    def update(self, results):
        (self.p, self.r, self.f1, self.all_ap, self.ap_class_index, self.p_curve, self.r_curve, self.f1_curve, self.px,
         self.prec_values) = results


class DetMetrics:
    """Detection metrics front-end (metrics.py:739-840, without plots)."""

    def __init__(self, save_dir=None, plot=False, on_plot=None, names=None) -> None:
        self.names = names or {}
        self.box = Metric()
        self.speed = {"preprocess": 0.0, "inference": 0.0, "loss": 0.0, "postprocess": 0.0}
        self.task = "detect"
        self.confusion_matrix = None   # the validator's ConfusionMatrix when it ran with plots=True

    def process(self, tp, conf, pred_cls, target_cls):
        results = ap_per_class(tp, conf, pred_cls, target_cls)[2:]
        self.box.nc = len(self.names)
        self.box.update(results)

    @property
    def keys(self):
        return ["metrics/precision(B)", "metrics/recall(B)", "metrics/mAP50(B)", "metrics/mAP50-95(B)"]

    def mean_results(self):
        return self.box.mean_results()

    def class_result(self, i):
        return self.box.class_result(i)

    @property
    def maps(self):
        return self.box.maps

    @property
    def fitness(self):
        return self.box.fitness()

    @property
    def ap_class_index(self):
        return self.box.ap_class_index

    @property
    def results_dict(self):
        return dict(zip(self.keys + ["fitness"], self.mean_results() + [self.fitness]))
