"""oracle/embed_ref.py — TEST INFRASTRUCTURE, not product code.

fp32 CPU restatement of the reference's feature embeddings: `BaseModel._predict_once(x, embed=idx)` (nn/tasks.py:118-145)
appends `adaptive_avg_pool2d(x, (1, 1)).squeeze(-1).squeeze(-1)` after every layer whose index is in `idx` (layer order,
a repeated index once) and, at layer max(idx), returns `torch.unbind(torch.cat(embeddings, 1), 0)`.  An empty `idx` is
falsy: the reference then predicts normally (here: None).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from . import yolo11_ref


def pool(x: torch.Tensor) -> torch.Tensor:
    """adaptive_avg_pool2d(x, (1, 1)).squeeze(-1).squeeze(-1): (B, C, H, W) -> (B, C)."""
    return F.adaptive_avg_pool2d(x, (1, 1)).squeeze(-1).squeeze(-1)


def from_features(ys, idx):
    """(B, D) embeddings from the per-layer outputs `ys` of yolo11_ref.forward(..., return_features=True), or None for an
    empty `idx`."""
    if not idx:
        return None
    return torch.cat([pool(y) for i, y in enumerate(ys) if i in idx], 1)


@torch.no_grad()
def embed(sd, x, idx):
    """(B, D) fp32 embeddings of `x` for the layer indices `idx` (the stack of the reference's per-image tuple), or None
    for an empty `idx`."""
    if not idx:
        return None
    return from_features(yolo11_ref.forward(sd, x, return_features=True)[2], idx)
