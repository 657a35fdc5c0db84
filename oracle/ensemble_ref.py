"""oracle/ensemble_ref.py — TEST INFRASTRUCTURE, not product code.

fp32 CPU restatement of the reference's model ensemble: `Ensemble.forward` (nn/tasks.py) runs every member on the same
batch, in list order, and returns `(torch.cat([m(x)[0] for m in self], 2), None)`: the members' (B, 4+nc, A_k)
predictions side by side along the anchor axis.  Members are state_dicts run through yolo11_ref.forward.
"""
from __future__ import annotations

import torch

from . import yolo11_ref


@torch.no_grad()
def forward(sds, x):
    """(y (B, 4+nc, sum of A_k) fp32, None) of the ensemble of the members `sds` on `x`."""
    return torch.cat([yolo11_ref.forward(sd, x)[0] for sd in sds], 2), None
