"""oracle/val_extras_ref.py — TEST INFRASTRUCTURE, not product code.

numpy restatements of the two validator switches, in the upstream Ultralytics code the reference copies:

  non_max_suppression(labels=...)  utils/ops.py:138-273 with the autolabel priors of :225-230 (the validator's
                                   `save_hybrid`): per image, after the confidence mask, one row per label (box
                                   xywh2xyxy(lb[:, 1:5]), score 1.0 at its class) is appended after the anchor rows,
                                   and the "no rows left" exit comes after that append.  Everything else is
                                   oracle/nms_ref.py's restatement, same deliberate differences (stable max_nms sort,
                                   no wall-clock exit, caller's array not mutated).
  ConfusionMatrix                  utils/metrics.py ConfusionMatrix.__init__ / process_batch / tp_fp (task "detect");
                                   upstream's IoU ties are ordered by np.argsort (unspecified), here by stable sorts:
                                   lower label index, then lower detection index.
"""
from __future__ import annotations

import numpy as np

from .metrics_ref import box_iou
from .nms_ref import nms, xywh2xyxy


def non_max_suppression(prediction: np.ndarray, conf_thres=0.25, iou_thres=0.45, classes=None, agnostic=False,
                        multi_label=False, labels=(), max_det=300, nc=0, max_nms=30000, max_wh=7680):
    """prediction (B, 4+nc, A) fp32; labels: () or B arrays (n_i, 5) [cls, cx, cy, w, h] in the prediction's pixel
    frame.  Returns a list of (n_i, 6) fp32 arrays [x1, y1, x2, y2, conf, cls], descending confidence."""
    assert 0 <= conf_thres <= 1 and 0 <= iou_thres <= 1                     # ops.py:186-187
    p = np.asarray(prediction, dtype=np.float32)
    bs = p.shape[0]
    nc = nc or (p.shape[1] - 4)                                             # ops.py:200
    assert p.shape[1] == 4 + nc, "mask channels are out of scope"
    conf32 = np.float32(conf_thres)
    xc = p[:, 4:].max(axis=1) > conf32                                      # ops.py:203 (strict >)
    multi_label = bool(multi_label) and nc > 1                              # ops.py:208
    p = p.transpose(0, 2, 1)                                                # ops.py:210 -> (B, A, 4+nc)
    out = [np.zeros((0, 6), np.float32) for _ in range(bs)]                 # ops.py:218
    for xi in range(bs):                                                    # ops.py:219
        x = p[xi][xc[xi]]                                                   # ops.py:222 (anchor order)
        box = xywh2xyxy(x[:, :4])                                           # ops.py:213
        cls = x[:, 4:]
        if len(labels) and len(labels[xi]):                                 # ops.py:225-230
            lb = np.asarray(labels[xi], dtype=np.float32).reshape(-1, 5)
            v = np.zeros((len(lb), nc), np.float32)
            v[np.arange(len(lb)), lb[:, 0].astype(np.int64)] = 1.0
            box = np.concatenate([box, xywh2xyxy(lb[:, 1:5])], 0)
            cls = np.concatenate([cls, v], 0)
        if not box.shape[0]:                                                # ops.py:233
            continue
        if multi_label:                                                     # ops.py:239-241 (row-major i, j)
            i, j = np.nonzero(cls > conf32)
            x = np.concatenate([box[i], cls[i, j][:, None], j[:, None].astype(np.float32)], 1)
        else:                                                               # ops.py:242-244 (first max wins)
            j = cls.argmax(1)
            conf = cls[np.arange(cls.shape[0]), j]
            x = np.concatenate([box, conf[:, None], j[:, None].astype(np.float32)], 1)[conf > conf32]
        if classes is not None:                                             # ops.py:247-248
            x = x[np.isin(x[:, 5], np.asarray(classes, dtype=np.float32))]
        n = x.shape[0]
        if not n:
            continue
        if n > max_nms:                                                     # ops.py:254-255
            x = x[np.argsort(-x[:, 4], kind="stable")[:max_nms]]
        c = x[:, 5:6] * np.float32(0 if agnostic else max_wh)               # ops.py:258
        boxes = (x[:, :4] + c).astype(np.float32)                           # ops.py:264 (fp32 add)
        keep = nms(boxes, x[:, 4], iou_thres, max_keep=max_det)             # ops.py:265-266
        out[xi] = np.ascontiguousarray(x[keep[:max_det]], dtype=np.float32)  # ops.py:268
    return out


class ConfusionMatrix:
    """(nc+1, nc+1) float64, [predicted, true], index nc = background."""

    def __init__(self, nc, conf=0.25, iou_thres=0.45):
        self.nc = nc
        self.matrix = np.zeros((nc + 1, nc + 1))
        self.conf = 0.25 if conf in {None, 0.001} else conf
        self.iou_thres = iou_thres

    def process_batch(self, detections, gt_bboxes, gt_cls):
        """detections (N, 6) [x1, y1, x2, y2, conf, cls] or None, gt_bboxes (M, 4) xyxy, gt_cls (M,)."""
        if gt_cls.shape[0] == 0:
            if detections is not None:
                detections = detections[detections[:, 4] > np.float32(self.conf)]
                for dc in detections[:, 5].astype(int):
                    self.matrix[dc, self.nc] += 1                       # false positives
            return
        if detections is None:
            for gc in gt_cls.astype(int):
                self.matrix[self.nc, gc] += 1                           # background FN
            return
        detections = detections[detections[:, 4] > np.float32(self.conf)]
        gt_classes = gt_cls.astype(int)
        detection_classes = detections[:, 5].astype(int)
        iou = box_iou(gt_bboxes, detections[:, :4])
        x = np.nonzero(iou > np.float32(self.iou_thres))
        if x[0].shape[0]:
            matches = np.concatenate((np.stack(x, 1), iou[x[0], x[1]][:, None]), 1)
            if x[0].shape[0] > 1:
                # upstream: argsort()[::-1] + np.unique(return_index); stable descending sorts pin the tie order
                matches = matches[np.argsort(-matches[:, 2], kind="stable")]
                matches = matches[np.unique(matches[:, 1], return_index=True)[1]]
                matches = matches[np.argsort(-matches[:, 2], kind="stable")]
                matches = matches[np.unique(matches[:, 0], return_index=True)[1]]
        else:
            matches = np.zeros((0, 3))
        n = matches.shape[0] > 0
        m0, m1, _ = matches.transpose().astype(int)
        for i, gc in enumerate(gt_classes):
            j = m0 == i
            if n and sum(j) == 1:
                self.matrix[detection_classes[m1[j]], gc] += 1          # correct
            else:
                self.matrix[self.nc, gc] += 1                           # true background
        for i, dc in enumerate(detection_classes):
            if not any(m1 == i):
                self.matrix[dc, self.nc] += 1                           # predicted background

    def tp_fp(self):
        tp = self.matrix.diagonal()
        fp = self.matrix.sum(1) - tp
        return tp[:-1], fp[:-1]


def batch_confusion(cm, dets, counts, gt_boxes, gt_cls, offsets):
    """The validator's per-image calls over one padded batch (detections=None for an image without any)."""
    for b in range(dets.shape[0]):
        n, s, e = int(counts[b]), int(offsets[b]), int(offsets[b + 1])
        if n == 0 and e == s:
            continue
        cm.process_batch(dets[b, :n] if n else None, gt_boxes[s:e], gt_cls[s:e])
    return cm
