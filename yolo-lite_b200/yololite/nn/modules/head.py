"""Detect head of YOLO11 (reference yololite/nn/modules/head.py:16-168, non-end2end path).

Same constructor, attributes (`nc, nl, reg_max, no, stride, cv2, cv3, dfl`), class attributes and state_dict
keys as the reference.  Per level the box branch (Conv3x3, Conv3x3, Conv2d1x1) and the class branch
(DW3x3+Conv1x1, DW3x3+Conv1x1, Conv2d1x1; `legacy` = three dense convs) write their last 1x1 conv in fp32
into the two channel slices of one (B, H, W, 4*reg_max + nc) raw map — the reference's per-level `torch.cat`
(head.py:64-65) — and a single decode kernel turns the three raw maps into the (B, 4+nc, A) prediction
(`_inference`, head.py:95-126).
"""
from __future__ import annotations

import copy
import math

import torch
import torch.nn as nn

from ._emit import YLModule, emit_any
from .block import DFL
from .conv import Conv, DWConv

__all__ = ("Detect",)


class Detect(YLModule):
    dynamic = False
    export = False
    format = None
    end2end = False
    max_det = 300
    shape = None
    anchors = torch.empty(0)
    strides = torch.empty(0)
    legacy = False
    #: decode (DFL / anchors / sigmoid) inside the epilogue of the last head convs instead of a separate kernel
    fuse_decode = True
    #: put the per-level box / class chains on parallel graph branches
    parallel_branches = True
    #: engine path (plan ends with single-label NMS): run the confidence filter + best-class selection of
    #: non_max_suppression inside the class convs' epilogue instead of writing and re-reading (B, nc, A) scores
    fuse_filter = True

    def __init__(self, nc=80, ch=()):
        super().__init__()
        self.nc = nc
        self.nl = len(ch)
        self.reg_max = 16
        self.no = nc + self.reg_max * 4
        self.stride = torch.zeros(self.nl)
        c2, c3 = max((16, ch[0] // 4, self.reg_max * 4)), max(ch[0], min(self.nc, 100))
        self.cv2 = nn.ModuleList(
            nn.Sequential(Conv(x, c2, 3), Conv(c2, c2, 3), nn.Conv2d(c2, 4 * self.reg_max, 1)) for x in ch
        )
        if self.legacy:
            self.cv3 = nn.ModuleList(
                nn.Sequential(Conv(x, c3, 3), Conv(c3, c3, 3), nn.Conv2d(c3, self.nc, 1)) for x in ch
            )
        else:
            self.cv3 = nn.ModuleList(
                nn.Sequential(
                    nn.Sequential(DWConv(x, x, 3), Conv(x, c3, 1)),
                    nn.Sequential(DWConv(c3, c3, 3), Conv(c3, c3, 1)),
                    nn.Conv2d(c3, self.nc, 1),
                )
                for x in ch
            )
        self.dfl = DFL(self.reg_max) if self.reg_max > 1 else nn.Identity()
        if self.end2end:
            raise NotImplementedError("end2end (YOLOv10-style) heads are not part of the YOLO11 path")

    # ------------------------------------------------------------------ plan
    def _fuses_decode(self) -> bool:
        """Whether the decode runs in the epilogue of the last head convs: what the tcgen05 path needs (otherwise the
        decode kernel runs after them)."""
        c2, c3 = self.cv2[0][-1].in_channels, self.cv3[0][-1].in_channels
        return (self.fuse_decode and self.reg_max == 16 and self.nc <= 256 and self.nc % 8 == 0
                and c2 % 8 == 0 and c3 % 8 == 0)

    def _fuses_filter(self, g, A: int) -> bool:
        """Whether the class convs run the NMS class filter in their epilogue for a prediction of A anchors."""
        import os

        return (self._fuses_decode() and self.fuse_filter and getattr(g, "nms_fuse_conf", None) is not None
                and not getattr(g, "want_raw", True) and A * self.nc < (1 << 32)
                and os.environ.get("YL_FUSE_FILTER", "1") != "0")

    def _emit(self, g, feats, out=None):
        """feats: list of nl NHWC views. Returns (y tensor (B, 4+nc, A) fp32, [raw NHWC f32 views]).

        `out`: None, or (y, anchor base) to write anchors [base, base + A) of a wider (B, 4+nc, A_total) prediction y
        (one member of a model ensemble).  The head then runs the class filter exactly when the caller has already begun
        the NMS workspace of the whole prediction (`g.cand_ws`), and returns that y."""
        assert len(feats) == self.nl
        if float(self.stride.sum()) == 0.0:
            raise RuntimeError("Detect.stride is unset (it is filled in by DetectionModel)")
        nbox = 4 * self.reg_max
        want_raw = getattr(g, "want_raw", True)
        raws = []
        if not self._fuses_decode():
            for i, x in enumerate(feats):
                raw = g.alloc(x.n, x.h, x.w, self.no, dtype=torch.float32)
                emit_any(g, self.cv2[i], x, out=raw.slice(0, nbox), out_dtype=torch.float32)
                emit_any(g, self.cv3[i][-1], self._emit_branch(g, self.cv3[i][:-1], x), out=raw.slice(nbox, self.nc),
                         out_dtype=torch.float32)
                raws.append(raw)
            y = g.detect_decode(raws, [float(s) for s in self.stride], self.reg_max, self.nc, into=out)
            return y, raws
        # fused: the last 1x1 conv of each branch decodes its logits straight into the prediction (DFL + anchors
        # + stride / sigmoid in the conv epilogue); the raw (B, H, W, no) maps are written only on request
        from ... import _C, _ops
        from ._emit import packed

        feats = [g.mat(x) for x in feats]
        n = feats[0].n
        A = sum(x.h * x.w for x in feats)
        import os

        conf = getattr(g, "nms_fuse_conf", None)
        if out is None:
            y, a0 = torch.empty((n, 4 + self.nc, A), dtype=torch.float32, device=g.device), 0
            g.buffers.append(y)
            filt = self._fuses_filter(g, A)
            cand_ws = g.nms_begin(n, A, self.nc) if filt else None
        else:
            y, a0 = out
            assert tuple(y.shape[:2]) == (n, 4 + self.nc) and 0 <= a0 and a0 + A <= y.shape[2], (tuple(y.shape), a0, A)
            cand_ws = getattr(g, "cand_ws", None)
            filt = cand_ws is not None
        for i, x in enumerate(feats):
            raw = g.alloc(x.n, x.h, x.w, self.no, dtype=torch.float32) if want_raw else None
            for j, (branch, mode, lo, cnt) in enumerate(((self.cv2[i], _C.DET_BOX, 0, nbox),
                                                          (self.cv3[i], _C.DET_CLS, nbox, self.nc))):
                # every (level, branch) chain depends only on its pyramid feature: side lanes let the graph run
                # them next to the rest of the neck (the last level's box branch stays on the main lane)
                lanes_on = self.parallel_branches and os.environ.get("YL_DET_LANES", "1") != "0"
                lane = 0 if (i == self.nl - 1 and j == 0) or not lanes_on else 1 + 2 * i + j
                with g.lane(lane):
                    last = branch[-1]
                    if filt and mode == _C.DET_CLS:
                        det = _ops.DetEpilogue(y, _C.DET_CLS_FILTER, self.reg_max, self.nc, a0, float(self.stride[i]),
                                               conf=conf, cand_ws=cand_ws)
                    else:
                        det = _ops.DetEpilogue(y, mode, self.reg_max, self.nc, a0, float(self.stride[i]))
                    # engine path, class branch: its last stage (DWConv + Conv) and the final conv + Detect epilogue run as
                    # one back-to-back launch when the kernel takes the shape
                    if mode == _C.DET_CLS and not want_raw and self._emit_cls_tail(g, branch, x, det):
                        continue
                    if mode == _C.DET_BOX and not want_raw and self._emit_box_tail(g, branch, x, det):
                        continue
                    t = self._emit_branch(g, branch[:-1], x)
                    g.conv(t, packed(last, None, last), 1, act=False, out=raw.slice(lo, cnt) if want_raw else None,
                           out_dtype=torch.float32, det=det, store=want_raw)
            if want_raw:
                raws.append(raw)
            a0 += x.h * x.w
        return y, raws

    @staticmethod
    def _emit_branch(g, mods, x):
        """The convs of one head branch in front of its last 1x1.  A class-branch stage `Sequential(DWConv 3x3, Conv 1x1)`
        (head.py:46-47) runs as ONE launch when the fused kernel takes the shape (yl_dw_pw_conv)."""
        from ._emit import act_flag, packed

        for sub in mods:
            y = None
            if (isinstance(sub, nn.Sequential) and len(sub) == 2 and isinstance(sub[0], DWConv) and type(sub[1]) is Conv
                    and sub[0].conv.kernel_size == (3, 3) and sub[0].conv.stride == (1, 1)
                    and sub[1].conv.kernel_size == (1, 1) and sub[1].conv.stride == (1, 1) and sub[1].conv.groups == 1):
                dw, pw = sub[0], sub[1]
                y = g.dwpw(g.mat(x), packed(dw.conv, dw.bn, dw), act_flag(dw.act), packed(pw.conv, pw.bn, pw),
                           act_flag(pw.act))
            x = y if y is not None else emit_any(g, sub, x)
        return x

    @classmethod
    def _emit_box_tail(cls, g, branch, x, det) -> bool:
        """[..., Conv k3, Conv2d 1x1 + box decode] with the last two as ONE launch (yl_conv_b2b_det).  Emits the earlier
        convs and returns True, or emits nothing and returns False."""
        from ._emit import act_flag, packed

        if len(branch) < 2 or not isinstance(branch[-1], nn.Conv2d) or type(branch[-2]) is not Conv:
            return False
        cv, last = branch[-2], branch[-1]
        if not (cv.conv.stride == (1, 1) and cv.conv.groups == 1 and last.kernel_size == (1, 1) and last.stride == (1, 1)
                and last.groups == 1 and g.conv_det_enabled):
            return False
        t = cls._emit_branch(g, branch[:-2], x)
        if g.conv_det(g.mat(t), packed(cv.conv, cv.bn, cv), act_flag(cv.act), packed(last, None, last), det):
            return True
        # the back-to-back kernel does not take the shape: finish the branch the plain way
        t = cls._emit_branch(g, branch[-2:-1], t)
        g.conv(t, packed(last, None, last), 1, act=False, out=None, out_dtype=torch.float32, det=det, store=False)
        return True

    @classmethod
    def _emit_cls_tail(cls, g, branch, x, det) -> bool:
        """[..., Sequential(DWConv 3x3, Conv 1x1), Conv2d 1x1 + Detect epilogue] with the last two as ONE launch
        (yl_dw_pw_det).  Emits the earlier stages and returns True, or emits nothing and returns False."""
        from ._emit import act_flag, packed

        if len(branch) < 2 or not isinstance(branch[-1], nn.Conv2d):
            return False
        sub, last = branch[-2], branch[-1]
        if not (isinstance(sub, nn.Sequential) and len(sub) == 2 and isinstance(sub[0], DWConv) and type(sub[1]) is Conv
                and sub[0].conv.kernel_size == (3, 3) and sub[0].conv.stride == (1, 1)
                and sub[1].conv.kernel_size == (1, 1) and sub[1].conv.stride == (1, 1) and sub[1].conv.groups == 1
                and last.kernel_size == (1, 1) and last.stride == (1, 1) and last.groups == 1):
            return False
        t = cls._emit_branch(g, branch[:-2], x)
        dw, pw = sub[0], sub[1]
        if g.dwpw_det(g.mat(t), packed(dw.conv, dw.bn, dw), act_flag(dw.act), packed(pw.conv, pw.bn, pw), act_flag(pw.act),
                      packed(last, None, last), det):
            return True
        # the back-to-back kernel does not take the shape: finish the branch the plain way
        t = cls._emit_branch(g, branch[-2:-1], t)
        g.conv(t, packed(last, None, last), 1, act=False, out=None, out_dtype=torch.float32, det=det, store=False)
        return True

    def _yl_export(self, g, res):
        y, raws = res
        return y, [g.to_nchw(r) for r in raws]

    def forward(self, x):
        """list of nl NCHW feature maps -> (y, [raw maps (B, no, H, W)]) like the reference in eval mode."""
        if self.training:
            raise NotImplementedError("yololite is inference-only: call .eval() (training is out of scope)")
        return super().forward(list(x))

    def bias_init(self):
        """Reference head.py:128-139: box bias 1.0, class bias log(5 / nc / (640 / s)^2)."""
        for a, b, s in zip(self.cv2, self.cv3, self.stride):
            a[-1].bias.data[:] = 1.0
            b[-1].bias.data[: self.nc] = math.log(5 / self.nc / (640 / float(s)) ** 2)
        self._yl_invalidate()
