"""AutoBackend (reference yololite/nn/autobackend.py:20-165): wraps a DetectionModel or an Ensemble (in-memory module,
a *.pt path, or a list of *.pt paths, which loads as an ensemble) for the predictor: device move, `.forward(im)` ->
[y, raw_list], `.warmup()`, attrs `stride, names, fp16, pt, device, nn_module`.  There is exactly one backend (the sm_100a kernels); `fp16`
is accepted for API compatibility — the compute type is always bf16 with fp32 accumulation."""
from __future__ import annotations

import torch
import torch.nn as nn

from ..utils import LOGGER


class AutoBackend(nn.Module):
    @torch.no_grad()
    def __init__(self, weights="yolo11n.pt", device=None, dnn=False, data=None, fp16=False, batch=1, fuse=True,
                 verbose=True):
        super().__init__()
        device = device if isinstance(device, torch.device) else torch.device(device or "cuda")
        if device.type != "cuda":
            raise RuntimeError("yololite runs on sm_100 GPUs only (no CPU fallback)")
        self.nn_module = isinstance(weights, nn.Module)
        if self.nn_module:
            model = weights.to(device)
        else:
            ws = [str(w) for w in (weights if isinstance(weights, list) else [weights])]
            for w in ws:
                if not w.endswith(".pt"):
                    raise NotImplementedError(f"'{w}': only PyTorch *.pt checkpoints or nn.Module objects are supported")
            from .tasks import attempt_load_weights

            # a list of two or more checkpoints loads as one Ensemble (reference autobackend.py: attempt_load_weights)
            model = attempt_load_weights(ws if len(ws) > 1 else ws[0], device=device, inplace=True, fuse=fuse)
        model = model.float().eval()
        for p in model.parameters():
            p.requires_grad = False
        self.model = model
        self.pt = True
        self.triton = False
        self.jit = False
        self.fp16 = False          # compute is bf16/fp32-accumulate regardless of `half`
        if fp16 and verbose:
            LOGGER.info("half=True ignored: the B200 path always computes in bf16 with fp32 accumulation")
        self.device = device
        self.stride = max(int(model.stride.max()), 32)
        self.names = model.module.names if hasattr(model, "module") else model.names
        self.task = getattr(model, "task", "detect")
        self.batch = batch

    def forward(self, im, augment=False, visualize=False, embed=None):
        """[y, raw maps]; with `augment=True` [merged test-time-augmentation prediction, None].  With `embed=[layer
        indices]` and no `augment` (which wins, as in the reference) the per-image feature vectors of
        `model.infer_embed`: a list of B 1-D tensors, or the tensor itself when B == 1 (TypeError for an Ensemble)."""
        if visualize:
            raise NotImplementedError("visualize is not part of the inference hot path")
        if embed and not augment:
            y = torch.unbind(self.model.infer_embed(im, embed), 0)
            return y[0] if len(y) == 1 else list(y)
        y, raws = self.model.infer(im, augment=augment)
        return [y, None] if augment else [y, raws]

    def warmup(self, imgsz=(1, 3, 640, 640)):
        """Build (and graph-capture) the plan for `imgsz` ahead of the first real batch."""
        im = torch.zeros(*imgsz, dtype=torch.float32, device=self.device)
        self.forward(im)
