"""Functional layer over the C-ABI: NHWC channel-slice views and one Python call per kernel launch.

Everything here enqueues work on the current torch CUDA stream and returns immediately; nothing allocates
except the explicit `new_buffer` / `pack_conv` helpers that plans call once at build time.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import _C


@dataclass
class View:
    """Channels [coff, coff + c) of an NHWC buffer (n, h, w, cstride)."""

    buf: torch.Tensor
    coff: int
    c: int

    @property
    def n(self):
        return self.buf.shape[0]

    @property
    def h(self):
        return self.buf.shape[1]

    @property
    def w(self):
        return self.buf.shape[2]

    def ct(self) -> _C.Tensor:
        return _C.view(self.buf, self.n, self.h, self.w, self.c, self.coff)

    def slice(self, off: int, c: int) -> "View":
        assert 0 <= off and off + c <= self.c
        return View(self.buf, self.coff + off, c)

    def torch_nhwc(self) -> torch.Tensor:
        return self.buf[..., self.coff:self.coff + self.c]


def new_buffer(n, h, w, c, dtype=torch.bfloat16, device=None) -> View:
    buf = torch.empty((n, h, w, c), dtype=dtype, device=device or torch.device("cuda", torch.cuda.current_device()))
    return View(buf, 0, c)


def round_up(v: int, m: int) -> int:
    return (v + m - 1) // m * m


@dataclass
class PackedConv:
    w: torch.Tensor      # bf16: dense [co_pad, k*k*ci_pad], depthwise [k*k, co_pad]
    bias: torch.Tensor   # f32 [co_pad]
    k: int
    ci: int
    co: int
    ci_pad: int
    co_pad: int
    depthwise: bool


def _f32(t, dev):
    return None if t is None else t.detach().to(device=dev, dtype=torch.float32).contiguous()


def _ptr(t):
    return None if t is None else t.data_ptr()


def pack_conv(weight: torch.Tensor, bn=None, conv_bias=None, device=None) -> PackedConv:
    """Fold BN (gamma, beta, mean, var, eps) into an OIHW conv weight and pack it for the kernels.

    Depthwise is detected as weight.shape[1] == 1 and co > 1 with k > 1 (DWConv, conv.py:100-105)."""
    lib = _C.init(device)
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    co, cig, k, k2 = weight.shape
    assert k == k2
    depthwise = cig == 1 and co > 1 and k > 1
    w = _f32(weight, dev)
    if bn is not None:
        gamma, beta, mean, var, eps = bn
        gamma, beta, mean, var = (_f32(t, dev) for t in (gamma, beta, mean, var))
    else:
        gamma = beta = mean = var = None
        eps = 0.0
    cb = _f32(conv_bias, dev)
    co_pad = round_up(co, 8) if depthwise else round_up(co, 16)   # yl_dwconv3x3 takes w as [9][c], c % 8 == 0
    ci_pad = 1 if depthwise else round_up(cig, 8)
    if depthwise:
        wp = torch.empty((k * k, co_pad), dtype=torch.bfloat16, device=dev)
    else:
        wp = torch.empty((co_pad, k * k * ci_pad), dtype=torch.bfloat16, device=dev)
    bias = torch.empty((co_pad,), dtype=torch.float32, device=dev)
    _C.check(lib.yl_fold_bn_pack(_ptr(w), _ptr(gamma), _ptr(beta), _ptr(mean), _ptr(var), _ptr(cb), float(eps), co,
                                 cig, k, co_pad, ci_pad, int(depthwise), wp.data_ptr(), bias.data_ptr(),
                                 _C.stream_ptr()), "yl_fold_bn_pack")
    # the fp32 sources must outlive the async kernel: synchronise once (build time, not hot path)
    torch.cuda.current_stream().synchronize()
    return PackedConv(wp, bias, k, cig, co, ci_pad, co_pad, depthwise)


@dataclass
class DetEpilogue:
    """Fused Detect decode of a head conv (see yl_det_epilogue): `pred` is the (B, 4+nc, A) fp32 prediction."""

    pred: torch.Tensor
    mode: int            # _C.DET_BOX | _C.DET_CLS | _C.DET_CLS_FILTER
    reg_max: int
    nc: int
    anchor0: int
    stride: float
    conf: float = 0.0                      # DET_CLS_FILTER: confidence threshold of the NMS that follows
    cand_ws: torch.Tensor | None = None    # DET_CLS_FILTER: NMS workspace the candidates are appended to


class NoOutput:
    """Shape-only destination for a conv whose result is consumed by a fused epilogue (no NHWC store)."""

    def __init__(self, n, h, w, c, dtype=torch.float32):
        self.n, self.h, self.w, self.c, self.dtype = n, h, w, c, dtype

    def ct(self) -> _C.Tensor:
        return _C.Tensor(None, self.n, self.h, self.w, self.c, self.c, 0,
                         _C.YL_F32 if self.dtype is torch.float32 else _C.YL_BF16, 0)


def conv_args(x: View, y, pc: PackedConv, stride=1, act=True, res: View | None = None, upsample=False,
              impl=_C.IMPL_AUTO, y_up: View | None = None, det: DetEpilogue | None = None) -> _C.ConvArgs:
    a = _C.ConvArgs()
    a.x, a.y = x.ct(), y.ct()
    if det is not None:
        assert det.pred.is_cuda and det.pred.dtype == torch.float32 and det.pred.is_contiguous() and det.pred.dim() == 3
        a.det.pred = det.pred.data_ptr()
        a.det.mode, a.det.reg_max, a.det.nc = det.mode, det.reg_max, det.nc
        a.det.A, a.det.anchor0, a.det.stride = det.pred.shape[2], det.anchor0, float(det.stride)
        if det.mode == _C.DET_CLS_FILTER:
            a.det.conf, a.det.cand_ws = float(det.conf), det.cand_ws.data_ptr()
    a.res = res.ct() if res is not None else _C.null_tensor()
    a.y_up = y_up.ct() if y_up is not None else _C.null_tensor()
    a.w, a.bias = pc.w.data_ptr(), pc.bias.data_ptr()
    a.k, a.stride, a.ci_pad, a.co_pad = pc.k, stride, pc.ci_pad, pc.co_pad
    a.act = _C.ACT_SILU if act else _C.ACT_NONE
    a.upsample2x = int(bool(upsample))
    a.impl = impl
    return a


def conv(x: View, y, pc: PackedConv, stride=1, act=True, res=None, upsample=False, impl=_C.IMPL_AUTO,
         y_up=None, det=None):
    lib = _C.load()
    if pc.depthwise:
        assert stride == 1 and pc.k == 3 and not upsample, "depthwise path is 3x3 stride 1"
        addp = C.byref(res.ct()) if res is not None else None
        _C.check(lib.yl_dwconv3x3(C.byref(x.ct()), C.byref(y.ct()), pc.w.data_ptr(), pc.bias.data_ptr(), int(act),
                                  addp, _C.stream_ptr()), "yl_dwconv3x3")
        return
    a = conv_args(x, y, pc, stride, act, res, upsample, impl, y_up, det)
    _C.check(lib.yl_conv_bn_act(C.byref(a), _C.stream_ptr()), "yl_conv_bn_act")


def stem_conv(x_nchw: torch.Tensor, y: View, pc: PackedConv, act=True):
    """Fused ingest + first layer: NCHW fp32 CUDA batch (<= 4 channels) -> 3x3 s2 conv + folded BN + SiLU -> NHWC bf16."""
    assert x_nchw.is_cuda and x_nchw.dtype == torch.float32 and x_nchw.is_contiguous() and x_nchw.dim() == 4
    n, c, h, w = x_nchw.shape
    yt = y.ct()
    _C.check(_C.load().yl_stem_conv(x_nchw.data_ptr(), n, c, h, w, pc.w.data_ptr(), pc.ci_pad, pc.bias.data_ptr(),
                                    C.byref(yt), int(act), _C.stream_ptr()), "yl_stem_conv")


def sppf_pool(x: View, y1: View, y2: View, y3: View, k=5):
    _C.check(_C.load().yl_sppf_pool(C.byref(x.ct()), C.byref(y1.ct()), C.byref(y2.ct()), C.byref(y3.ct()), k,
                                    _C.stream_ptr()), "yl_sppf_pool")


def upsample2x(x: View, y: View):
    _C.check(_C.load().yl_upsample2x(C.byref(x.ct()), C.byref(y.ct()), _C.stream_ptr()), "yl_upsample2x")


def copy_slice(x: View, y: View):
    _C.check(_C.load().yl_copy_slice(C.byref(x.ct()), C.byref(y.ct()), _C.stream_ptr()), "yl_copy_slice")


def attention(qkv: View, out: View, heads: int, key_dim: int, head_dim: int, scale: float):
    _C.check(_C.load().yl_psa_attention(C.byref(qkv.ct()), C.byref(out.ct()), heads, key_dim, head_dim, float(scale),
                                        _C.stream_ptr()), "yl_psa_attention")


def nchw_to_nhwc(x: torch.Tensor, y: View):
    assert x.is_cuda and x.dtype == torch.float32 and x.is_contiguous() and x.dim() == 4
    assert tuple(x.shape) == (y.n, y.c, y.h, y.w), (tuple(x.shape), (y.n, y.c, y.h, y.w))
    _C.check(_C.load().yl_nchw_to_nhwc(x.data_ptr(), C.byref(y.ct()), _C.stream_ptr()), "yl_nchw_to_nhwc")


def nhwc_to_nchw(x: View, out: torch.Tensor | None = None) -> torch.Tensor:
    if out is None:
        out = torch.empty((x.n, x.c, x.h, x.w), dtype=torch.float32, device=x.buf.device)
    _C.check(_C.load().yl_nhwc_to_nchw(C.byref(x.ct()), out.data_ptr(), _C.stream_ptr()), "yl_nhwc_to_nchw")
    return out


def detect_decode(levels: list[View], strides, reg_max: int, nc: int, y: torch.Tensor, anchor_base: int | None = None):
    """Decode the raw head maps `levels` into y (B, 4+nc, A) (yl_detect_decode), or, with `anchor_base`, into anchors
    [anchor_base, anchor_base + A) of a wider y (yl_detect_decode_into)."""
    arr = (_C.Tensor * len(levels))(*[v.ct() for v in levels])
    st = (C.c_float * len(levels))(*[float(s) for s in strides])
    if anchor_base is None:
        _C.check(_C.load().yl_detect_decode(arr, len(levels), st, reg_max, nc, y.data_ptr(), _C.stream_ptr()),
                 "yl_detect_decode")
    else:
        _C.check(_C.load().yl_detect_decode_into(arr, len(levels), st, reg_max, nc, y.data_ptr(), y.shape[2],
                                                 int(anchor_base), _C.stream_ptr()), "yl_detect_decode_into")


def dfl_expectation(x: torch.Tensor, reg_max: int) -> torch.Tensor:
    lib = _C.init(x.device)
    b, c, a = x.shape
    assert c == 4 * reg_max
    x = x.contiguous().float()
    y = torch.empty((b, 4, a), dtype=torch.float32, device=x.device)
    _C.check(lib.yl_dfl(x.data_ptr(), y.data_ptr(), b, reg_max, a, _C.stream_ptr()), "yl_dfl")
    return y


class NmsWorkspace:
    """Grow-only device scratch for yl_nms_batched, cached per (device, stream): two batches in flight on two
    streams must not share candidate lists."""

    _cache: dict = {}

    @classmethod
    def get(cls, nbytes: int, device) -> torch.Tensor:
        key = (device.type, device.index, int(torch.cuda.current_stream(device).cuda_stream))
        t = cls._cache.get(key)
        if t is None or t.numel() < nbytes:
            t = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
            cls._cache[key] = t
        return t


def nms_batched(pred: torch.Tensor, conf: float, iou: float, classes=None, agnostic=False, multi_label=False,
                max_det=300, max_nms=30000, max_wh=7680.0, out=None, counts=None, labels=None):
    """pred (B, 4+nc, A) fp32 contiguous CUDA -> (dets (B, max_det, 6) fp32, counts (B,) int32), all async.
    `classes`: None, a sequence of class ids, or a contiguous int32 tensor of them on pred's device.
    `labels`: None or ground-truth priors packed as (xywh (L, 4) fp32, cls (L,) int32, both on pred's device, and the
    B + 1 host ints `offsets`: image b owns rows [offsets[b], offsets[b+1])); class ids must already be in [0, nc)."""
    lib = _C.init(pred.device)
    assert pred.is_cuda and pred.dtype == torch.float32 and pred.is_contiguous() and pred.dim() == 3
    B, C4, A = pred.shape
    nc = C4 - 4
    lab_xywh = lab_cls = lab_off = None
    max_l = 0
    if labels is not None:
        lab_xywh, lab_cls, offsets = labels
        offsets = [int(o) for o in offsets]
        assert len(offsets) == B + 1 and offsets[0] == 0, "labels: offsets must be B + 1 ints starting at 0"
        max_l = max(e - s for s, e in zip(offsets[:-1], offsets[1:]))
        assert max_l >= 0 and lab_xywh.shape == (offsets[-1], 4) and lab_cls.shape == (offsets[-1],)
        assert lab_xywh.dtype == torch.float32 and lab_cls.dtype == torch.int32
        assert lab_xywh.device == pred.device and lab_cls.device == pred.device
        lab_xywh, lab_cls = lab_xywh.contiguous(), lab_cls.contiguous()
        lab_off = torch.as_tensor(offsets, dtype=torch.int32).to(pred.device)
    ws_bytes = lib.yl_nms_priors_workspace_bytes(B, A, nc, int(multi_label), max_l)
    ws = NmsWorkspace.get(ws_bytes, pred.device)
    if out is None:
        out = torch.empty((B, max_det, 6), dtype=torch.float32, device=pred.device)
    if counts is None:
        counts = torch.empty((B,), dtype=torch.int32, device=pred.device)
    cls_t = None
    if isinstance(classes, torch.Tensor):   # already a device int32 list: no host->device copy (and no sync) per call
        cls_t = classes
    elif classes is not None:
        cls_t = torch.as_tensor(list(classes), dtype=torch.int32).to(pred.device)
    _C.check(lib.yl_nms_batched_priors(pred.data_ptr(), B, nc, A, float(conf), float(iou), _ptr(cls_t),
                                       0 if cls_t is None else cls_t.numel(), int(agnostic), int(multi_label),
                                       int(max_det), int(max_nms), float(max_wh), _ptr(lab_xywh), _ptr(lab_cls),
                                       _ptr(lab_off), max_l, ws.data_ptr(), ws.numel(), out.data_ptr(),
                                       counts.data_ptr(), _C.stream_ptr()), "yl_nms_batched_priors")
    return out, counts


def nms_boxes(boxes: torch.Tensor, scores: torch.Tensor, iou: float) -> torch.Tensor:
    """torchvision.ops.nms drop-in on CUDA tensors (returns int64 keep indices, descending score)."""
    lib = _C.init(boxes.device)
    n = boxes.shape[0]
    boxes = boxes.contiguous().float()
    scores = scores.contiguous().float()
    keep = torch.empty((max(n, 1),), dtype=torch.int64, device=boxes.device)
    count = torch.zeros((1,), dtype=torch.int32, device=boxes.device)
    ws = NmsWorkspace.get(lib.yl_nms_boxes_workspace_bytes(n), boxes.device)
    _C.check(lib.yl_nms_boxes(boxes.data_ptr(), scores.data_ptr(), n, float(iou), ws.data_ptr(), ws.numel(),
                              keep.data_ptr(), count.data_ptr(), _C.stream_ptr()), "yl_nms_boxes")
    return keep[: int(count.item())]


def tta_scale_img(x: torch.Tensor, canvases):
    """scale_img of test-time augmentation passes 1 and 2 in one launch (yl_tta_scale_img).  x: contiguous (n, c, h, w)
    CUDA batch, fp32 / fp16 / uint8 image bytes; canvases: two (y (n, c, H, W) fp32, (h_content, w_content), flip)."""
    n, c, h, w = x.shape
    arr = (_C.TtaCanvas * 2)(*[_C.TtaCanvas(y.data_ptr(), y.shape[2], y.shape[3], ch, cw, int(bool(flip)), 0)
                               for y, (ch, cw), flip in canvases])
    _C.check(_C.load().yl_tta_scale_img(x.data_ptr(), _C.INGEST_DTYPES[x.dtype], n, c, h, w, arr, _C.stream_ptr()),
             "yl_tta_scale_img")


def tta_merge(passes, img_w: int, out: torch.Tensor) -> torch.Tensor:
    """_descale_pred + _clip_augmented + cat of the three passes (yl_tta_merge).  passes: three (pred (B, 4+nc, A) fp32,
    first kept anchor, kept count, scale, flip); out: (B, 4+nc, sum of kept counts) fp32."""
    B, C4, _ = out.shape
    arr = (_C.TtaPass * 3)(*[_C.TtaPass(p.data_ptr(), p.shape[2], a0, n, int(bool(flip)), float(s), 0)
                             for p, a0, n, s, flip in passes])
    _C.check(_C.load().yl_tta_merge(arr, B, C4 - 4, int(img_w), out.data_ptr(), _C.stream_ptr()), "yl_tta_merge")
    return out


def embed_pool_taps(views):
    """yl_embed_tap array of NHWC bf16 channel slices whose pooled means fill consecutive output columns, and the total
    width D."""
    arr = (_C.EmbedTap * len(views))()
    col = 0
    for k, v in enumerate(views):
        arr[k] = _C.EmbedTap(v.ct(), col, 0)
        col += v.c
    return arr, col


def embed_pool_workspace(taps, B: int, D: int, device) -> torch.Tensor:
    """Zeroed workspace of yl_embed_pool for these taps (at least 16 bytes)."""
    need = C.c_size_t(0)
    _C.check(_C.load().yl_embed_pool(taps, len(taps), B, D, None, None, C.byref(need), None), "yl_embed_pool")
    return torch.zeros(max(int(need.value), 16), dtype=torch.uint8, device=device)


def embed_pool(views, out: torch.Tensor, workspace: torch.Tensor | None = None) -> torch.Tensor:
    """Per-channel spatial mean of every view (adaptive_avg_pool2d to 1x1), side by side in out (B, sum of c) fp32, in one
    launch (yl_embed_pool).  `workspace`: from embed_pool_workspace for the same views (allocated here when None)."""
    taps, D = embed_pool_taps(views)
    B = views[0].n
    assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and tuple(out.shape) == (B, D)
    if workspace is None:
        workspace = embed_pool_workspace(taps, B, D, out.device)
    cap = C.c_size_t(workspace.numel())
    _C.check(_C.load().yl_embed_pool(taps, len(taps), B, D, out.data_ptr(), workspace.data_ptr(), C.byref(cap),
                                     _C.stream_ptr()), "yl_embed_pool")
    return out
