"""Post-processing ops with the reference's signatures (yololite/utils/ops.py): `non_max_suppression`
(:138-273), `xywh2xyxy` (:372-389), `scale_boxes` (:66-98), `clip_boxes` (:276-295), `Profile` (:18-63).

`non_max_suppression` keeps the reference's argument list and its `list[Tensor(n, 6)]` return layout, but the
per-image Python loop, boolean-index compaction (host syncs) and torchvision.ops.nms are replaced by two
batched CUDA kernels (csrc/nms.cu) that are bit-exact against the reference's CPU arithmetic; the only host
synchronisation is one read of the (B,) counts at the end.  There is no wall-clock early exit
(`max_time_img` is accepted and ignored: the reference silently drops images when it fires, ops.py:269-271).
Ground-truth priors (`labels=`, ops.py:225-230) join each image's candidates after its anchors inside the same
two kernels (`yl_nms_batched_priors`).
"""
from __future__ import annotations

import contextlib
import time

import numpy as np
import torch

from .. import _ops

__all__ = ("non_max_suppression", "nms_padded", "xywh2xyxy", "xyxy2xywh", "scale_boxes", "clip_boxes", "Profile",
           "make_divisible", "convert_torch2numpy_batch")


class Profile(contextlib.ContextDecorator):
    """`with Profile(device=...) as dt:` accumulating wall time; synchronises CUDA on both edges."""

    def __init__(self, t=0.0, device: torch.device | None = None):
        self.t = t
        self.device = device
        self.cuda = bool(device and str(device).startswith("cuda"))

    def __enter__(self):
        self.start = self.time()
        return self

    def __exit__(self, *exc):
        self.dt = self.time() - self.start
        self.t += self.dt

    def __str__(self):
        return f"Elapsed time is {self.t} s"

    def time(self):
        if self.cuda:
            torch.cuda.synchronize(self.device)
        return time.time()


def make_divisible(x, divisor):
    import math

    if isinstance(divisor, torch.Tensor):
        divisor = int(divisor.max())
    return math.ceil(x / divisor) * divisor


def xywh2xyxy(x):
    """(cx, cy, w, h) -> (x1, y1, x2, y2) on the last dim; torch tensor or numpy array."""
    assert x.shape[-1] == 4, f"input shape last dimension expected 4 but input shape is {x.shape}"
    y = torch.empty_like(x) if isinstance(x, torch.Tensor) else np.empty_like(x)
    half = x[..., 2:] / 2
    y[..., :2] = x[..., :2] - half
    y[..., 2:] = x[..., :2] + half
    return y


def xyxy2xywh(x):
    assert x.shape[-1] == 4
    y = torch.empty_like(x) if isinstance(x, torch.Tensor) else np.empty_like(x)
    y[..., 0] = (x[..., 0] + x[..., 2]) / 2
    y[..., 1] = (x[..., 1] + x[..., 3]) / 2
    y[..., 2] = x[..., 2] - x[..., 0]
    y[..., 3] = x[..., 3] - x[..., 1]
    return y


def coco80_to_coco91_class():
    """COCO 80-class index -> category id of the 91-id COCO annotation files (reference data/converter.py)."""
    return [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 27, 28, 31, 32, 33,
            34, 35, 36, 37, 38, 39, 40, 41, 42, 43, 44, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 59, 60, 61,
            62, 63, 64, 65, 67, 70, 72, 73, 74, 75, 76, 77, 78, 79, 80, 81, 82, 84, 85, 86, 87, 88, 89, 90]


def clip_boxes(boxes, shape):
    """Clamp xyxy boxes to an image of `shape` = (h, w), in place."""
    if isinstance(boxes, torch.Tensor):
        boxes[..., 0].clamp_(0, shape[1])
        boxes[..., 1].clamp_(0, shape[0])
        boxes[..., 2].clamp_(0, shape[1])
        boxes[..., 3].clamp_(0, shape[0])
    else:
        boxes[..., [0, 2]] = boxes[..., [0, 2]].clip(0, shape[1])
        boxes[..., [1, 3]] = boxes[..., [1, 3]].clip(0, shape[0])
    return boxes


def letterbox_params(img1_shape, img0_shape, ratio_pad=None):
    """gain and (padx, pady) that map img0 (original) into img1 (network input), reference ops.py:83-91."""
    if ratio_pad is None:
        gain = min(img1_shape[0] / img0_shape[0], img1_shape[1] / img0_shape[1])
        pad = (round((img1_shape[1] - img0_shape[1] * gain) / 2 - 0.1),
               round((img1_shape[0] - img0_shape[0] * gain) / 2 - 0.1))
    else:
        gain = ratio_pad[0][0]
        pad = ratio_pad[1]
    return gain, pad


def scale_boxes(img1_shape, boxes, img0_shape, ratio_pad=None, padding=True, xywh=False):
    """Rescale xyxy boxes from the network input shape to the original image shape, in place."""
    gain, pad = letterbox_params(img1_shape, img0_shape, ratio_pad)
    if padding:
        boxes[..., 0] -= pad[0]
        boxes[..., 1] -= pad[1]
        if not xywh:
            boxes[..., 2] -= pad[0]
            boxes[..., 3] -= pad[1]
    boxes[..., :4] /= gain
    return clip_boxes(boxes, img0_shape)


def convert_torch2numpy_batch(batch: torch.Tensor) -> np.ndarray:
    return (batch.permute(0, 2, 3, 1).contiguous() * 255).clamp(0, 255).to(torch.uint8).cpu().numpy()


def pack_priors(labels, device=None):
    """The reference's `labels` argument (B tensors (n_i, 5): cls, cx, cy, w, h) -> the packed priors of
    `nms_padded`: (xywh (L, 4), cls (L,), offsets: B + 1 ints), on the labels' own device unless `device` is given."""
    offsets = [0]
    for lb in labels:
        offsets.append(offsets[-1] + len(lb))
    rows = [lb.reshape(-1, 5) for lb in labels]
    lb = torch.cat([r.to(device) if device is not None else r for r in rows], 0) if rows else torch.zeros((0, 5))
    return lb[:, 1:5], lb[:, 0], offsets


def _check_priors(labels, nc):
    """Validate packed priors; returns them as (xywh, int64 cls, offsets).  The range test runs where the class ids
    are: free on the host, one read for device tensors."""
    xywh, cls, offsets = labels
    offsets = [int(o) for o in offsets]
    if xywh.shape != (offsets[-1], 4) or cls.reshape(-1).shape != (offsets[-1],):
        raise ValueError(f"labels: {tuple(xywh.shape)} boxes and {tuple(cls.shape)} classes for {offsets[-1]} priors")
    cls = cls.reshape(-1).long()   # lb[:, 0].long() of the reference
    if cls.numel() and bool(((cls < 0) | (cls >= nc)).any()):
        bad = cls[(cls < 0) | (cls >= nc)][0].item()
        raise ValueError(f"labels: class id {bad} is outside [0, {nc})")
    return xywh, cls, offsets


def nms_padded(prediction, conf_thres=0.25, iou_thres=0.45, classes=None, agnostic=False, multi_label=False,
               max_det=300, nc=0, max_nms=30000, max_wh=7680, out=None, counts=None, labels=None):
    """Device-resident NMS: (B, 4+nc, A) -> (dets (B, max_det, 6) fp32, counts (B,) int32), fully async.

    `labels`: None or ground-truth priors packed as `pack_priors` returns them (boxes in the prediction's pixel frame;
    CPU or CUDA); a class id outside [0, nc) raises ValueError.
    This is what the engine uses; `non_max_suppression` below turns it into the reference's list layout."""
    if isinstance(prediction, (list, tuple)):
        prediction = prediction[0]
    nc = nc or (prediction.shape[1] - 4)
    if labels is not None:
        labels = _check_priors(labels, nc)
    if not prediction.is_cuda:
        raise RuntimeError("yololite NMS runs on CUDA (sm_100) only; there is no CPU fallback")
    if prediction.shape[1] != 4 + nc:
        raise NotImplementedError("mask coefficients (nm > 0) are outside the detection path")
    pred = prediction if (prediction.dtype == torch.float32 and prediction.is_contiguous()) else \
        prediction.float().contiguous()
    if labels is not None:
        xywh, cls, offsets = labels
        labels = (xywh.to(pred.device, torch.float32), cls.to(pred.device, torch.int32), offsets)
    return _ops.nms_batched(pred, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, max_nms, max_wh,
                            out=out, counts=counts, labels=labels)


def non_max_suppression(
    prediction,
    conf_thres=0.25,
    iou_thres=0.45,
    classes=None,
    agnostic=False,
    multi_label=False,
    labels=(),
    max_det=300,
    nc=0,
    max_time_img=0.05,
    max_nms=30000,
    max_wh=7680,
    in_place=True,
    rotated=False,
):
    """Drop-in for the reference's non_max_suppression: returns a list (one per image) of (n, 6) tensors
    [x1, y1, x2, y2, confidence, class] sorted by descending confidence.  `labels`: the reference's autolabel priors,
    one (n_i, 5) tensor [cls, cx, cy, w, h] per image (CPU or CUDA), appended to the image's candidates with score
    1.0; a class id outside [0, nc) raises ValueError (the reference fails with an IndexError there)."""
    assert 0 <= conf_thres <= 1, f"Invalid Confidence threshold {conf_thres}, valid values are between 0.0 and 1.0"
    assert 0 <= iou_thres <= 1, f"Invalid IoU {iou_thres}, valid values are between 0.0 and 1.0"
    if isinstance(prediction, (list, tuple)):
        prediction = prediction[0]
    if rotated:
        raise NotImplementedError("rotated boxes (OBB) are outside the detection path")
    if prediction.shape[-1] == 6:  # end2end layout (B, N, 6): plain confidence filter, as in the reference
        output = [p[p[:, 4] > conf_thres][:max_det] for p in prediction]
        if classes is not None:
            cl = torch.tensor(classes, device=prediction.device)
            output = [p[(p[:, 5:6] == cl).any(1)] for p in output]
        return output
    priors = None
    if labels is not None and len(labels):
        if len(labels) != prediction.shape[0]:
            raise ValueError(f"labels: {len(labels)} entries for a batch of {prediction.shape[0]} images")
        priors = pack_priors(labels)
    dets, counts = nms_padded(prediction, conf_thres, iou_thres, classes, agnostic, multi_label, max_det, nc,
                              max_nms, max_wh, labels=priors)
    if in_place and prediction.dtype == torch.float32 and prediction.is_contiguous():
        # observable side effect of the reference (ops.py:213): caller's boxes become xyxy
        from .. import _C

        B, C4, A = prediction.shape
        _C.check(_C.load().yl_xywh2xyxy_inplace(prediction.data_ptr(), B, C4, A, _C.stream_ptr()),
                 "yl_xywh2xyxy_inplace")
    n = counts.tolist()  # the single host sync of the path
    return [dets[i, : n[i]] for i in range(len(n))]
