"""oracle/tta_ref.py — TEST INFRASTRUCTURE, not product code.

fp32 CPU restatement of the reference's test-time augmentation over oracle/yolo11_ref.forward: `scale_img`
(utils/torch_utils.py) and `DetectionModel._predict_augment / _descale_pred / _clip_augmented` (nn/tasks.py), written
as the reference writes them.  tests/test_tta*.py compare yololite's `augment=True` path against it.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from . import yolo11_ref

SCALES = (1, 0.83, 0.67)   # _predict_augment
FLIPS = (None, 3, None)    # 3 = left-right


def scale_img(img, ratio=1.0, same_shape=False, gs=32):
    """utils/torch_utils.py scale_img: bilinear resize by `ratio`, pad to a multiple of gs with 0.447."""
    if ratio == 1.0:
        return img
    h, w = img.shape[2:]
    s = (int(h * ratio), int(w * ratio))
    img = F.interpolate(img, size=s, mode="bilinear", align_corners=False)
    if not same_shape:
        h, w = (math.ceil(x * ratio / gs) * gs for x in (h, w))
    return F.pad(img, [0, w - s[1], 0, h - s[0]], value=0.447)


def descale_pred(p, flips, scale, img_size, dim=1):
    """DetectionModel._descale_pred: undo the scale and flip of one pass's (B, 4+nc, A) prediction."""
    p[:, :4] /= scale
    x, y, wh, cls = p.split((1, 1, 2, p.shape[dim] - 4), dim)
    if flips == 2:
        y = img_size[0] - y
    elif flips == 3:
        x = img_size[1] - x
    return torch.cat((x, y, wh, cls), dim)


def clip_augmented(y, nl=3):
    """DetectionModel._clip_augmented: drop the largest-stride level of the first pass and the smallest of the last."""
    g = sum(4 ** x for x in range(nl))
    e = 1
    i = (y[0].shape[-1] // g) * sum(4 ** x for x in range(e))
    y[0] = y[0][..., :-i]
    i = (y[-1].shape[-1] // g) * sum(4 ** (nl - 1 - x) for x in range(e))
    y[-1] = y[-1][..., i:]
    return y


@torch.no_grad()
def predict_augment(sd, x, gs=32):
    """DetectionModel._predict_augment over yolo11_ref.forward: x (B, 3, h, w) fp32 in [0, 1] -> (B, 4+nc, A_tta)."""
    x = x.float()
    img_size = x.shape[-2:]
    y = []
    for si, fi in zip(SCALES, FLIPS):
        xi = scale_img(x.flip(fi) if fi else x, si, gs=gs)
        yi = yolo11_ref.forward(sd, xi)[0]
        y.append(descale_pred(yi, fi, si, img_size))
    return torch.cat(clip_augmented(y), -1)
