"""Static launch plans: the host-side "graph executor" of the B200 path.

A `Builder` records, for one fixed input shape, the exact sequence of C-ABI kernel launches a module tree
performs, with every activation buffer pre-allocated (NHWC bf16) and channel concatenation expressed as
aliasing (producers write straight into channel slices of the consumer's buffer).  `Plan.run()` replays the
pre-marshalled ctypes calls on the current stream; `Plan.capture()` wraps that replay in a CUDA graph so a
forward is one `cudaGraphLaunch` (the reference issues ~300 ATen kernels per forward, nn/tasks.py:118-145).

The Builder also records which buffer slices every launch reads and writes.  Emitters may put independent
sub-chains (the Detect branches of each pyramid level) on side "lanes" (`with g.lane(k):`); at capture time a
lane becomes a forked stream whose launches wait only on their true producers, so the CUDA graph has parallel
branches and the launch-latency-bound tail of small layers overlaps the big head convolutions.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os
from typing import Callable

import torch

from . import _C, _ops
from ._ops import PackedConv, View


class Dest:
    """Deferred output placement: resolves to a View once the producer knows its output shape."""

    def __init__(self, resolve: Callable[[int, int, int, int], View]):
        self._resolve = resolve

    def __call__(self, n, h, w, c) -> View:
        v = self._resolve(n, h, w, c)
        assert (v.n, v.h, v.w, v.c) == (n, h, w, c), f"destination {(v.n, v.h, v.w, v.c)} != {(n, h, w, c)}"
        return v


class DualDest:
    """Two placements for one conv result: `primary` (None | View | Dest) at conv resolution and `up`
    (None | View | Dest) receiving the nearest-2x replicated copy (nn.Upsample fused into the producer's TMA
    store).  After emission `up_view` holds the upsampled View."""

    def __init__(self, primary, up):
        self.primary, self.up = primary, up
        self.up_view: View | None = None


class NchwInput:
    """The caller's NCHW fp32 batch, not yet converted.  A stem conv consumes it directly (fused ingest);
    anything else forces the NHWC bf16 materialisation."""

    def __init__(self, static: torch.Tensor):
        self.static = static
        self.n, self.c, self.h, self.w = static.shape
        self.view: View | None = None


class Builder:
    def __init__(self, device: torch.device):
        self.device = device
        self.lib = _C.init(device)
        self.calls: list[tuple] = []      # (fn, args tuple without stream, keepalive)
        self.lanes: list[int] = []        # lane (forked stream) of every call; 0 = the main stream
        self.deps: list[tuple] = []       # per call: indices of earlier calls whose results it reads / overwrites
        self._cur_lane = 0
        self.lane_base = 0                # lane ids of `lane(k)` are offset by this (the members of an ensemble plan)
        self._access: dict = {}           # buffer data_ptr -> [(c0, c1, call index, is_write)]
        self.buffers: list[torch.Tensor] = []
        self.bytes = 0
        self.meta: list[dict] = []
        self.ingest: NchwInput | None = None
        self.model_start = 0               # index of the first launch of the model being recorded (its image ingest)
        self.n_ingest = 1                  # leading launches that read the caller's batch and stay outside the graph
        self.want_raw = True               # Detect: also write the raw head maps (module-level API)
        # single-label NMS arguments (conf, ...) of the step this plan ends with, when the Detect head may run the class
        # filter in its conv epilogues (set by BaseModel._get_plan); the head then fills `cand_ws`
        self.nms_fuse_conf: float | None = None
        self.cand_ws: torch.Tensor | None = None
        self.layer: int | None = None      # model layer being emitted (recorded in `meta`; set by BaseModel._emit)
        # conv chains (csrc/conv_chain.cu): runs of small-map convs as ONE launch, one 4-CTA cluster per image.  Opt-in
        # (YL_CHAIN=1): parity-exact, but measured 3-5 % slower than the per-layer launches at every batch size — those
        # layers are bound by L2 -> SM operand traffic and the per-MMA A-operand read, not by launch overhead
        # (profiles/r02_conv_chain.md)
        self.chain_enabled = os.environ.get("YL_CHAIN", "0") == "1"
        self.chain_min_batch = int(os.environ.get("YL_CHAIN_MIN_BATCH", "1"))
        self.chain_max_hw = int(os.environ.get("YL_CHAIN_MAX_HW", "1600"))
        # DWConv 3x3 + Conv 1x1 pairs (Detect class branch) as one launch (csrc/dwpw_tc.cu)
        self.dwpw_enabled = os.environ.get("YL_DWPW", "1") != "0"
        self.dwpw_det_enabled = os.environ.get("YL_DWPW_DET", "1") != "0"
        # tail of the Detect box branch (Conv 3x3 + final 1x1 + box decode) as one back-to-back launch: opt-in.  Bit-identical
        # and 12 us less kernel time per step, but the step got 1.3 % SLOWER (40.5 k vs 41.0 k images/s): the longer kernels
        # overlap worse with the class-branch kernels on the other graph lanes (profiles/r02_SUMMARY.md)
        self.conv_det_enabled = os.environ.get("YL_CONV_DET", "0") == "1"

    # ------------------------------------------------------------------ memory
    def alloc(self, n, h, w, c, dtype=torch.bfloat16) -> View:
        buf = torch.empty((n, h, w, c), dtype=dtype, device=self.device)
        self.buffers.append(buf)
        self.bytes += buf.numel() * buf.element_size()
        return View(buf, 0, c)

    def _out(self, out, n, h, w, c, dtype=torch.bfloat16) -> View:
        if out is None:
            return self.alloc(n, h, w, c, dtype)
        if isinstance(out, Dest):
            return out(n, h, w, c)
        assert (out.n, out.h, out.w, out.c) == (n, h, w, c), ((out.n, out.h, out.w, out.c), (n, h, w, c))
        return out

    @contextlib.contextmanager
    def lane(self, k: int):
        """Launches emitted inside run on side lane `k` (a forked stream at graph capture)."""
        prev, self._cur_lane = self._cur_lane, self.lane_base + int(k)
        try:
            yield
        finally:
            self._cur_lane = prev

    @contextlib.contextmanager
    def model(self, lane_base: int = 0):
        """Record one model of a multi-model plan (an ensemble member): its first launch is its own image ingest, and
        `lane(k)` inside it means lane `lane_base + k` (its main lane is `lane_base`)."""
        self.model_start = len(self.calls)
        self.lane_base = self._cur_lane = int(lane_base)
        try:
            yield
        finally:
            self.lane_base = self._cur_lane = 0

    def _track(self, idx, reads, writes):
        """RAW / WAR / WAW dependencies of call `idx` from the channel-slice access history of each buffer."""
        deps = set()
        for views, is_write in ((reads, False), (writes, True)):
            for v in views:
                if v is None:
                    continue
                if isinstance(v, tuple):            # (tensor, lo, hi): an explicit sub-range of a plain tensor
                    key, c0, c1 = v[0].data_ptr(), int(v[1]), int(v[2])
                elif isinstance(v, torch.Tensor):
                    key, c0, c1 = v.data_ptr(), 0, 1 << 30
                else:
                    key, c0, c1 = v.buf.data_ptr(), v.coff, v.coff + v.c
                hist = self._access.setdefault(key, [])
                for (a0, a1, j, w) in hist:
                    if j != idx and a0 < c1 and c0 < a1 and (w or is_write):
                        deps.add(j)
                hist.append((c0, c1, idx, is_write))
        return tuple(sorted(deps))

    def _push(self, fn, *args, keep=(), kind="", bytes_=0, flops=0, desc="", reads=(), writes=()):
        idx = len(self.calls)
        self.calls.append((fn, args, keep))
        self.lanes.append(self._cur_lane)
        self.deps.append(self._track(idx, reads, writes))
        # algorithmic work of the launch (each operand touched once): the roofline numerators of DESIGN.md
        self.meta.append({"kind": kind or fn.__name__, "bytes": int(bytes_), "flops": int(flops), "desc": desc,
                          "layer": self.layer})

    # ------------------------------------------------------------------ ops
    def input_nchw(self, x_nchw_static: torch.Tensor) -> NchwInput:
        self.ingest = NchwInput(x_nchw_static)
        return self.ingest

    def mat(self, x):
        """NHWC bf16 view of `x` (materialises a pending NCHW input with the layout kernel)."""
        if isinstance(x, (list, tuple)):
            return [self.mat(v) for v in x]
        if not isinstance(x, NchwInput):
            return x
        if x.view is None:
            v = self.alloc(x.n, x.h, x.w, x.c)
            t = v.ct()
            self._push(self.lib.yl_nchw_to_nhwc, x.static.data_ptr(), C.byref(t), keep=(t, x.static),
                       kind="ingest_nchw_to_nhwc", bytes_=x.n * x.c * x.h * x.w * (4 + 2), writes=(v,))
            x.view = v
        return x.view

    def conv(self, x: View, pc: PackedConv, stride=1, act=True, out=None, res: View | None = None,
             upsample=False, out_dtype=torch.bfloat16, impl=_C.IMPL_AUTO, det=None, store=True) -> View:
        """`det`: _ops.DetEpilogue fusing the Detect decode into this conv; with `store=False` the conv result is
        consumed by that epilogue only and no NHWC tensor is written (returns None)."""
        k = pc.k
        dual = None
        if isinstance(out, DualDest):
            dual, out = out, out.primary
            assert not pc.depthwise and not upsample and not isinstance(x, NchwInput)
        if isinstance(x, NchwInput):
            if (x.view is None and len(self.calls) == self.model_start and k == 3 and stride == 2 and x.c <= 4
                    and not pc.depthwise and res is None and not upsample and out_dtype is torch.bfloat16
                    and pc.co in (16, 32, 48, 64, 96)):
                ho, wo = (x.h - 1) // 2 + 1, (x.w - 1) // 2 + 1
                y = self._out(out, x.n, ho, wo, pc.co)
                yt = y.ct()
                self._push(self.lib.yl_stem_conv, x.static.data_ptr(), x.n, x.c, x.h, x.w, pc.w.data_ptr(), pc.ci_pad,
                           pc.bias.data_ptr(), C.byref(yt), int(act), keep=(yt, pc, x.static), kind="stem_conv",
                           bytes_=x.n * x.c * x.h * x.w * 4 + x.n * ho * wo * pc.co * 2,
                           flops=2 * x.n * ho * wo * pc.co * x.c * 9, desc=f"{x.c}->{pc.co} k3s2 {x.h}x{x.w} nchw-f32 in",
                           writes=(y,))
                return y
            x = self.mat(x)
        ho = (x.h + 2 * (k // 2) - k) // stride + 1
        wo = (x.w + 2 * (k // 2) - k) // stride + 1
        u = 2 if upsample else 1
        if not store:
            assert det is not None and out is None and not pc.depthwise
            y = _ops.NoOutput(x.n, ho, wo, pc.co, out_dtype)
        else:
            y = self._out(out, x.n, ho * u, wo * u, pc.co, out_dtype)
        if pc.depthwise:
            assert stride == 1 and k == 3 and not upsample
            xt, yt = x.ct(), y.ct()
            rt = res.ct() if res is not None else None
            px = x.n * x.h * x.w
            self._push(self.lib.yl_dwconv3x3, C.byref(xt), C.byref(yt), pc.w.data_ptr(), pc.bias.data_ptr(), int(act),
                       C.byref(rt) if rt is not None else None, keep=(xt, yt, rt, pc), kind="dwconv3x3",
                       bytes_=px * x.c * 2 * (2 + (res is not None)) + 9 * x.c * 2, flops=2 * 9 * px * x.c,
                       reads=(x, res), writes=(y,))
            return y
        y_up = None
        if dual is not None:
            y_up = dual.up_view = self._out(dual.up, x.n, 2 * ho, 2 * wo, pc.co, out_dtype)
        a = _ops.conv_args(x, y, pc, stride, act, res, upsample, impl, y_up, det)
        opx = x.n * ho * wo
        esz = 4 if out_dtype is torch.float32 else 2
        tc = impl != _C.IMPL_DIRECT and bool(self.lib.yl_conv_tc_supported(C.byref(a)))
        if det is not None and not tc:
            raise RuntimeError(f"fused Detect decode rejected by the tcgen05 path: {x.c}->{pc.co} k{k}")
        out_bytes = opx * pc.co * esz * u * u if store else 0
        if det is not None:   # decoded rows of the prediction: 4 box values or nc scores per anchor, fp32
            out_bytes += opx * (4 if det.mode == _C.DET_BOX else (0 if det.mode == _C.DET_CLS_FILTER else det.nc)) * 4
        self._push(self.lib.yl_conv_bn_act, C.byref(a), keep=(a, pc, det), kind="conv_tc" if tc else "conv_direct",
                   bytes_=x.n * x.h * x.w * x.c * 2 + out_bytes + k * k * x.c * pc.co * 2
                   + (opx * pc.co * 2 if res is not None else 0) + (4 * opx * pc.co * esz if y_up is not None else 0),
                   flops=2 * opx * pc.co * x.c * k * k,
                   desc=f"{x.c}->{pc.co} k{k}s{stride} {x.h}x{x.w}" + (" +res" if res is not None else "")
                   + (" up2" if upsample else "") + (" +up2" if y_up is not None else "")
                   + (" f32" if esz == 4 and store else "")
                   + ("" if det is None else (" +filter" if det.mode == _C.DET_CLS_FILTER else " +decode")),
                   reads=(x, res),
                   # the fused decode writes its own block of the prediction: rows (box | class) x this level's anchors;
                   # blocks of different launches are disjoint, a reader of the whole tensor (NMS) depends on all of them
                   writes=(y if store else None, y_up,
                           None if det is None or det.mode == _C.DET_CLS_FILTER else
                           (det.pred, 2 * det.anchor0 + (det.mode == _C.DET_CLS), 2 * det.anchor0 + (det.mode == _C.DET_CLS) + 1),
                           # the class filter appends to the candidate lists: ordered after yl_nms_begin (which wrote the
                           # whole workspace), unordered among the levels (atomic appends), all before yl_nms_select
                           None if det is None or det.mode != _C.DET_CLS_FILTER else
                           (det.cand_ws, 1 + det.anchor0, 2 + det.anchor0)))
        return y if store else None

    def dwpw(self, x: View, pdw: PackedConv, act_dw: bool, ppw: PackedConv, act_pw: bool, out=None):
        """DWConv 3x3 (+BN+act) followed by Conv 1x1 (+BN+act) as one launch (yl_dw_pw_conv): the depthwise result feeds the
        1x1 GEMM through shared memory and is never written.  Returns None when the fused kernel does not take the shape
        (the caller then emits the two layers)."""
        x = self.mat(x)
        if not (self.dwpw_enabled and pdw.depthwise and pdw.k == 3 and ppw.k == 1 and not ppw.depthwise
                and pdw.co == x.c and pdw.co_pad == x.c and ppw.ci == x.c):
            return None
        y = self._out(out, x.n, x.h, x.w, ppw.co)
        a = _ops.conv_args(x, y, ppw, 1, act_pw, None, False, _C.IMPL_TCGEN05, None, None)
        if not self.lib.yl_dw_pw_supported(C.byref(a)):
            return None
        px = x.n * x.h * x.w
        self._push(self.lib.yl_dw_pw_conv, C.byref(a), pdw.w.data_ptr(), pdw.bias.data_ptr(), int(bool(act_dw)),
                   keep=(a, pdw, ppw), kind="dwpw_tc", bytes_=px * (x.c + ppw.co) * 2 + (9 * x.c + x.c * ppw.co) * 2,
                   flops=2 * px * (9 * x.c + x.c * ppw.co), desc=f"[dw3x3 {x.c}, {x.c}->{ppw.co} k1] {x.h}x{x.w}",
                   reads=(x,), writes=(y,))
        return y

    def conv_det(self, x: View, pc: PackedConv, act: bool, plast: PackedConv, det) -> bool:
        """Tail of a Detect box branch on the engine path: Conv k x k (+BN+act) + the final 1x1 conv with its Detect decode
        (no NHWC store) as ONE launch (yl_conv_b2b_det: back-to-back tcgen05 GEMMs, the tensor between them stays in shared
        memory).  False when the kernel does not take the shape."""
        x = self.mat(x)
        if not (self.conv_det_enabled and not pc.depthwise and not plast.depthwise and plast.k == 1 and plast.ci == pc.co):
            return False
        ho, wo = x.h, x.w                         # stride 1, 'same' padding
        mid = _ops.NoOutput(x.n, ho, wo, pc.co, torch.bfloat16)
        a1 = _ops.conv_args(x, mid, pc, 1, act, None, False, _C.IMPL_TCGEN05, None, None)
        a2 = _ops.conv_args(mid, _ops.NoOutput(x.n, ho, wo, plast.co, torch.float32), plast, 1, False, None, False,
                            _C.IMPL_TCGEN05, None, det)
        if not self.lib.yl_conv_b2b_det_supported(C.byref(a1), C.byref(a2)):
            return False
        px = x.n * ho * wo
        rows = 4 if det.mode == _C.DET_BOX else det.nc
        self._push(self.lib.yl_conv_b2b_det, C.byref(a1), C.byref(a2), keep=(a1, a2, pc, plast, det), kind="conv_tc",
                   bytes_=px * x.c * 2 + px * rows * 4 + (pc.k * pc.k * x.c * pc.co + pc.co * plast.co) * 2,
                   flops=2 * px * (pc.k * pc.k * x.c * pc.co + pc.co * plast.co),
                   desc=f"[{x.c}->{pc.co} k{pc.k}s1, {pc.co}->{plast.co} k1 +decode] {x.h}x{x.w}", reads=(x,),
                   writes=((det.pred, 2 * det.anchor0 + (det.mode == _C.DET_CLS), 2 * det.anchor0 + (det.mode == _C.DET_CLS) + 1),))
        return True

    def dwpw_det(self, x: View, pdw: PackedConv, act_dw: bool, ppw: PackedConv, act_pw: bool, plast: PackedConv, det) -> bool:
        """Last stage of a Detect class branch on the engine path: DWConv 3x3 + Conv 1x1 + the final 1x1 conv with its
        Detect epilogue (class decode / class filter, no NHWC store) as ONE launch (yl_dw_pw_det: two back-to-back tcgen05
        GEMMs, the c3-channel tensor between them stays in shared memory).  False when the kernel does not take the shape."""
        x = self.mat(x)
        if not (self.dwpw_enabled and self.dwpw_det_enabled and pdw.depthwise and pdw.k == 3 and ppw.k == 1 and plast.k == 1
                and not ppw.depthwise and not plast.depthwise and pdw.co == x.c and pdw.co_pad == x.c and ppw.ci == x.c
                and plast.ci == ppw.co):
            return False
        mid = _ops.NoOutput(x.n, x.h, x.w, ppw.co, torch.bfloat16)
        a1 = _ops.conv_args(x, mid, ppw, 1, act_pw, None, False, _C.IMPL_TCGEN05, None, None)
        a2 = _ops.conv_args(mid, _ops.NoOutput(x.n, x.h, x.w, plast.co, torch.float32), plast, 1, False, None, False,
                            _C.IMPL_TCGEN05, None, det)
        if not self.lib.yl_dw_pw_det_supported(C.byref(a1), C.byref(a2)):
            return False
        px = x.n * x.h * x.w
        filt = det.mode == _C.DET_CLS_FILTER
        self._push(self.lib.yl_dw_pw_det, C.byref(a1), pdw.w.data_ptr(), pdw.bias.data_ptr(), int(bool(act_dw)), C.byref(a2),
                   keep=(a1, a2, pdw, ppw, plast, det), kind="dwpw_tc",
                   bytes_=px * x.c * 2 + (0 if filt else px * det.nc * 4) + (9 * x.c + x.c * ppw.co + ppw.co * plast.co) * 2,
                   flops=2 * px * (9 * x.c + x.c * ppw.co + ppw.co * plast.co),
                   desc=f"[dw3x3 {x.c}, {x.c}->{ppw.co} k1, {ppw.co}->{plast.co} k1 {'+filter' if filt else '+decode'}] {x.h}x{x.w}",
                   reads=(x,),
                   writes=((det.cand_ws, 1 + det.anchor0, 2 + det.anchor0) if filt else
                           (det.pred, 2 * det.anchor0 + 1, 2 * det.anchor0 + 2),))
        return True

    def stem_fused(self, x: NchwInput, pc0: PackedConv, pc1: PackedConv, act0: bool, act1: bool, out=None) -> View:
        """Image ingest + the first two stride-2 3x3 convs in one launch (see yl_stem_fused)."""
        assert x.view is None and len(self.calls) == self.model_start, "the fused stem must be the model's first launch"
        h0, w0 = (x.h - 1) // 2 + 1, (x.w - 1) // 2 + 1
        h1, w1 = (h0 - 1) // 2 + 1, (w0 - 1) // 2 + 1
        y = self._out(out, x.n, h1, w1, pc1.co)
        yt = y.ct()
        self._push(self.lib.yl_stem_fused, x.static.data_ptr(), _C.YL_F32, x.n, x.c, x.h, x.w, pc0.w.data_ptr(), pc0.ci_pad,
                   pc0.bias.data_ptr(), int(act0), pc1.w.data_ptr(), pc1.ci_pad, pc1.bias.data_ptr(), int(act1),
                   C.byref(yt), keep=(yt, pc0, pc1, x.static), kind="stem_fused",
                   bytes_=x.n * x.c * x.h * x.w * 4 + x.n * h1 * w1 * pc1.co * 2,
                   flops=2 * x.n * (h0 * w0 * pc0.co * x.c * 9 + h1 * w1 * pc1.co * pc0.co * 9),
                   desc=f"[{x.c}->{pc0.co} k3s2, {pc0.co}->{pc1.co} k3s2] {x.h}x{x.w} nchw-f32 in", writes=(y,))
        return y

    def c3k2_tail(self, t: View, pa: PackedConv, pb: PackedConv, p2: PackedConv, shortcut: bool, out=None,
                  impl: str = "auto") -> View:
        """Fused [Bottleneck(3x3, 3x3) + C2f.cv2] on t = cv1(x) = [y0 | y1] (see yl_c3k2_tail); impl="tc" forces the
        tcgen05 version (yl_c3k2_tail_tc)."""
        y = self._out(out, t.n, t.h, t.w, p2.co)
        tt, yt = t.ct(), y.ct()
        c = t.c // 2
        px = t.n * t.h * t.w
        self._push(self.lib.yl_c3k2_tail_tc if impl == "tc" else self.lib.yl_c3k2_tail, C.byref(tt), C.byref(yt),
                   pa.w.data_ptr(), pa.bias.data_ptr(), pa.co_pad,
                   pa.ci_pad, pb.w.data_ptr(), pb.bias.data_ptr(), pb.ci_pad, p2.w.data_ptr(), p2.bias.data_ptr(),
                   p2.ci_pad, int(bool(shortcut)), keep=(tt, yt, pa, pb, p2), kind="c3k2_tail",
                   bytes_=px * (t.c + p2.co) * 2 + (pa.w.numel() + pb.w.numel() + p2.w.numel()) * 2,
                   flops=2 * px * (9 * c * (c // 2) * 2 + 3 * c * p2.co),
                   desc=f"[{c}->{c // 2} k3, {c // 2}->{c} k3{' +res' if shortcut else ''}, {3 * c}->{p2.co} k1] "
                        f"{t.h}x{t.w}", reads=(t,), writes=(y,))
        return y

    def sppf_pool(self, x: View, y1: View, y2: View, y3: View, k: int):
        ts = [v.ct() for v in (x, y1, y2, y3)]
        self._push(self.lib.yl_sppf_pool, *[C.byref(t) for t in ts], k, keep=tuple(ts), kind="sppf_pool",
                   bytes_=x.n * x.h * x.w * x.c * 2 * 4, reads=(x,), writes=(y1, y2, y3))

    def upsample2x(self, x: View, out=None) -> View:
        x = self.mat(x)
        y = self._out(out, x.n, 2 * x.h, 2 * x.w, x.c)
        xt, yt = x.ct(), y.ct()
        self._push(self.lib.yl_upsample2x, C.byref(xt), C.byref(yt), keep=(xt, yt), kind="upsample2x",
                   bytes_=x.n * x.h * x.w * x.c * 2 * 5, reads=(x,), writes=(y,))
        return y

    def copy(self, x: View, out=None) -> View:
        x = self.mat(x)
        y = self._out(out, x.n, x.h, x.w, x.c)
        xt, yt = x.ct(), y.ct()
        self._push(self.lib.yl_copy_slice, C.byref(xt), C.byref(yt), keep=(xt, yt), kind="copy_slice",
                   bytes_=x.n * x.h * x.w * x.c * 2 * 2, reads=(x,), writes=(y,))
        return y

    def attention(self, qkv: View, heads: int, key_dim: int, head_dim: int, scale: float, out=None) -> View:
        y = self._out(out, qkv.n, qkv.h, qkv.w, heads * head_dim)
        qt, yt = qkv.ct(), y.ct()
        ntok = qkv.h * qkv.w
        self._push(self.lib.yl_psa_attention, C.byref(qt), C.byref(yt), heads, key_dim, head_dim, float(scale),
                   keep=(qt, yt), kind="psa_attention", bytes_=qkv.n * ntok * (qkv.c + heads * head_dim) * 2,
                   flops=2 * qkv.n * heads * ntok * ntok * (key_dim + head_dim), reads=(qkv,), writes=(y,))
        return y

    def detect_decode(self, levels: list[View], strides, reg_max: int, nc: int, into=None) -> torch.Tensor:
        """`into`: None (a new (B, 4+nc, A) prediction) or (y, anchor base): write anchors [base, base + A) of the wider
        prediction y (yl_detect_decode_into; one member of an ensemble)."""
        n = levels[0].n
        a = sum(v.h * v.w for v in levels)
        arr = (_C.Tensor * len(levels))(*[v.ct() for v in levels])
        st = (C.c_float * len(levels))(*[float(s) for s in strides])
        bytes_ = n * a * ((4 * reg_max + nc) * 4 + (4 + nc) * 4)
        if into is None:
            y = torch.empty((n, 4 + nc, a), dtype=torch.float32, device=self.device)
            self.buffers.append(y)
            self._push(self.lib.yl_detect_decode, arr, len(levels), st, reg_max, nc, y.data_ptr(), keep=(arr, st),
                       kind="detect_decode", bytes_=bytes_, reads=tuple(levels), writes=(y,))
            return y
        y, base = into
        assert y.shape[0] == n and y.shape[1] == 4 + nc and 0 <= base and base + a <= y.shape[2], (tuple(y.shape), base, a)
        # written range in the anchor encoding of the fused decode epilogues (2 * anchor + box | class row)
        self._push(self.lib.yl_detect_decode_into, arr, len(levels), st, reg_max, nc, y.data_ptr(), y.shape[2], int(base),
                   keep=(arr, st), kind="detect_decode", bytes_=bytes_, desc=f"anchors [{base}, {base + a}) of {y.shape[2]}",
                   reads=tuple(levels), writes=((y, 2 * base, 2 * (base + a)),))
        return y

    def nms_begin(self, B: int, A: int, nc: int) -> torch.Tensor:
        """Workspace of a step whose class filter runs inside the Detect head convs (DET_CLS_FILTER): allocates it and
        records the launch that zeroes its candidate counters (the head convs that append candidates depend on it)."""
        ws = torch.empty(max(int(self.lib.yl_nms_workspace_bytes(B, A, nc, 0)), 16), dtype=torch.uint8, device=self.device)
        self.buffers.append(ws)
        self.cand_ws = ws
        self._push(self.lib.yl_nms_begin, ws.data_ptr(), ws.numel(), B, keep=(ws,), kind="nms_begin", bytes_=B * 4,
                   writes=(ws,))
        return ws

    def nms(self, pred: torch.Tensor, conf, iou, classes=None, agnostic=False, multi_label=False, max_det=300,
            max_nms=30000, max_wh=7680.0):
        """Batched NMS as the last launches of the plan (so a whole step is the ingest + ONE graph launch): the
        workspace, (B, max_det, 6) detections and (B,) counts are plan-owned static buffers."""
        B, C4, A = pred.shape
        nc = C4 - 4
        if self.cand_ws is not None:
            # the Detect head already filtered: candidates are in the workspace, only the per-image select remains
            assert not multi_label and classes is None and self.nms_fuse_conf == float(conf)
            ws = self.cand_ws
            out = torch.empty((B, max_det, 6), dtype=torch.float32, device=self.device)
            counts = torch.empty((B,), dtype=torch.int32, device=self.device)
            self.buffers += [out, counts]
            self._push(self.lib.yl_nms_select, pred.data_ptr(), B, nc, A, float(iou), int(agnostic), int(max_det),
                       int(max_nms), float(max_wh), ws.data_ptr(), ws.numel(), out.data_ptr(), counts.data_ptr(),
                       keep=(ws, out, counts, pred), kind="nms_select", bytes_=B * 4 * A * 4,
                       desc=f"iou {iou} max_det {max_det} (filter fused into the head)", reads=(pred, ws),
                       writes=(out, counts))
            return out, counts
        ws = torch.empty(max(int(self.lib.yl_nms_workspace_bytes(B, A, nc, int(multi_label))), 16), dtype=torch.uint8,
                         device=self.device)
        out = torch.empty((B, max_det, 6), dtype=torch.float32, device=self.device)
        counts = torch.empty((B,), dtype=torch.int32, device=self.device)
        cls_t = None if classes is None else torch.as_tensor(list(classes), dtype=torch.int32).to(self.device)
        self.buffers += [ws, out, counts]
        self._push(self.lib.yl_nms_batched, pred.data_ptr(), B, nc, A, float(conf), float(iou),
                   None if cls_t is None else cls_t.data_ptr(), 0 if cls_t is None else cls_t.numel(), int(agnostic),
                   int(multi_label), int(max_det), int(max_nms), float(max_wh), ws.data_ptr(), ws.numel(), out.data_ptr(),
                   counts.data_ptr(), keep=(ws, out, counts, cls_t, pred), kind="nms", bytes_=B * C4 * A * 4,
                   desc=f"conf {conf} iou {iou} max_det {max_det}", reads=(pred,), writes=(out, counts, ws))
        return out, counts

    def embed_pool(self, views: list[View]) -> torch.Tensor:
        """Per-channel spatial means of the tapped layer outputs `views`, side by side in a plan-owned (B, D) fp32 output
        (yl_embed_pool, one launch ordered after every producer of the taps)."""
        B = views[0].n
        taps, D = _ops.embed_pool_taps(views)
        out = torch.empty((B, D), dtype=torch.float32, device=self.device)
        ws = _ops.embed_pool_workspace(taps, B, D, self.device)
        self.buffers += [out, ws]
        cap = C.c_size_t(ws.numel())
        self._push(self.lib.yl_embed_pool, taps, len(views), B, D, out.data_ptr(), ws.data_ptr(), C.byref(cap),
                   keep=(taps, cap, ws, out), kind="embed_pool",
                   bytes_=sum(v.n * v.h * v.w * v.c * 2 for v in views) + B * D * 4,
                   desc=f"{len(views)} taps -> ({B}, {D}) f32", reads=tuple(views), writes=(out, ws))
        return out

    def to_nchw(self, x: View) -> torch.Tensor:
        x = self.mat(x)
        out = torch.empty((x.n, x.c, x.h, x.w), dtype=torch.float32, device=self.device)
        self.buffers.append(out)
        xt = x.ct()
        self._push(self.lib.yl_nhwc_to_nchw, C.byref(xt), out.data_ptr(), keep=(xt,), kind="export_nhwc_to_nchw",
                   bytes_=x.n * x.h * x.w * x.c * (x.buf.element_size() + 4), reads=(x,), writes=(out,))
        return out

    # ------------------------------------------------------------------ conv chains
    def _fuse_chains(self):
        """Merge runs of consecutive small-map conv launches of one lane into yl_conv_chain launches (one cluster per
        image walks the whole run; csrc/conv_chain.cu).  Members keep their order, so every dependency inside a run is
        satisfied by the chain's own layer barriers; the chain inherits the members' outside dependencies."""
        n = len(self.calls)
        lib = self.lib

        def member(i):
            fn, args, keep = self.calls[i]
            if fn is not lib.yl_conv_bn_act or self.meta[i]["kind"] != "conv_tc":
                return False
            a = keep[0]
            if a.x.n < self.chain_min_batch or a.y.h * a.y.w > self.chain_max_hw or a.x.h * a.x.w > self.chain_max_hw:
                return False
            return bool(lib.yl_conv_chain_supported(C.byref(a)))

        ok = [member(i) for i in range(n)]
        groups, i = [], 0
        while i < n:
            if not ok[i]:
                i += 1
                continue
            j = i
            while j + 1 < n and ok[j + 1] and self.lanes[j + 1] == self.lanes[i]:
                j += 1
            if j > i:
                groups.append((i, j))
            i = j + 1
        if not groups:
            return
        start = {g[0]: g for g in groups}
        new_index, calls, lanes, deps, meta = {}, [], [], [], []
        i = 0
        while i < n:
            if i in start:
                lo, hi = start[i]
                idx = len(calls)
                for m in range(lo, hi + 1):
                    new_index[m] = idx
                members = list(range(lo, hi + 1))
                arr = (_C.ConvArgs * len(members))(*[self.calls[m][2][0] for m in members])
                nbytes = int(lib.yl_conv_chain_desc_bytes(len(members)))
                desc = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
                chain = _C.ConvChain()
                _C.check(lib.yl_conv_chain_build(arr, len(members), desc.data_ptr(), nbytes, C.byref(chain),
                                                 _C.stream_ptr()), "yl_conv_chain_build")
                self.buffers.append(desc)
                calls.append((lib.yl_conv_chain_run, (C.byref(chain),),
                              (chain, desc, arr, [self.calls[m][2] for m in members])))
                lanes.append(self.lanes[lo])
                deps.append(tuple(sorted({new_index[d] for m in members for d in self.deps[m] if d < lo})))
                mm = [self.meta[m] for m in members]
                meta.append({"kind": "conv_chain", "bytes": sum(x["bytes"] for x in mm), "flops": sum(x["flops"] for x in mm),
                             "desc": f"{len(mm)} convs: " + " | ".join(x["desc"] for x in mm), "members": mm})
                i = hi + 1
            else:
                new_index[i] = len(calls)
                calls.append(self.calls[i])
                lanes.append(self.lanes[i])
                deps.append(tuple(sorted({new_index[d] for d in self.deps[i]})))
                meta.append(self.meta[i])
                i += 1
        self.calls, self.lanes, self.deps, self.meta = calls, lanes, deps, meta

    def hoist(self, first: list[int]):
        """Move calls `first` (in this order) in front of all others: the image ingests of an ensemble's members, which
        depend on no earlier launch, so that the plan starts with every launch that reads the caller's batch."""
        assert all(not self.deps[i] for i in first)
        chosen = set(first)
        order = list(first) + [i for i in range(len(self.calls)) if i not in chosen]
        new = {old: k for k, old in enumerate(order)}
        self.deps = [tuple(sorted(new[d] for d in self.deps[i])) for i in order]
        self.calls, self.lanes, self.meta = ([v[i] for i in order] for v in (self.calls, self.lanes, self.meta))
        self._access = {}                 # call indices changed: nothing may be recorded after this

    def finish(self) -> "Plan":
        if self.chain_enabled:
            self._fuse_chains()
        return Plan(self)


class Plan:
    """Replayable launch sequence (+ optional CUDA graph)."""

    def __init__(self, b: Builder):
        self.device = b.device
        self.calls = b.calls
        self.lanes = b.lanes
        self.deps = b.deps
        self.meta = b.meta
        self.buffers = b.buffers
        self.bytes = b.bytes
        self.graph: torch.cuda.CUDAGraph | None = None
        self._skip = 0
        self.n_launches = len(b.calls)
        self.n_ingest = b.n_ingest

    @property
    def native_ingest(self):
        """yl_dtypes that every ingest launch of the plan (its first `n_ingest` calls) reads directly from the caller's
        batch: the fused stem takes fp32, fp16 and uint8 images; the other ingests (stem_conv, nchw_to_nhwc) read fp32
        only."""
        if not self.calls:
            return ()
        out = (_C.YL_F32, _C.YL_F16, _C.YL_U8)
        for fn, _, _ in self.calls[: self.n_ingest]:
            name = fn.__name__
            if name != "yl_stem_fused":
                reads = (_C.YL_F32,) if name in ("yl_nchw_to_nhwc", "yl_stem_conv") else ()
                out = tuple(d for d in out if d in reads)
        return out

    def run(self, ingest_ptr: int | None = None, ingest_dtype: int = _C.YL_F32):
        """Replay.  `ingest_ptr`: device pointer of an NCHW batch (of `ingest_dtype`, one of `native_ingest`) to read
        instead of the static input (only the first `n_ingest` calls, the image ingests, consume it; they are never part
        of the CUDA graph)."""
        s = _C.stream_ptr()
        first = 0
        if self.graph is not None or ingest_ptr is not None:
            for fn, args, _ in self.calls[: self._skip if self.graph is not None else self.n_ingest]:
                a = args
                if ingest_ptr is not None and fn.__name__ in ("yl_nchw_to_nhwc", "yl_stem_conv", "yl_stem_fused"):
                    if fn.__name__ == "yl_stem_fused":
                        a = (ingest_ptr, int(ingest_dtype)) + tuple(args[2:])
                    else:
                        assert ingest_dtype == _C.YL_F32, "this plan's ingest kernel reads fp32 only"
                        a = (ingest_ptr,) + tuple(args[1:])
                _C.check(fn(*a, s), fn.__name__)
            first = self._skip if self.graph is not None else self.n_ingest
        if self.graph is not None:
            self.graph.replay()
            return
        self.run_eager(first)

    def run_eager(self, skip: int = 0):
        s = _C.stream_ptr()
        check = _C.check
        for fn, args, _ in self.calls[skip:]:
            rc = fn(*args, s)
            if rc != 0:
                check(rc, fn.__name__)

    def conv_dispatch(self):
        """[(meta desc, _C.ConvTcPlan)] for every tcgen05 conv launch of the plan: which host-side dispatch (image-stacked
        tiles, N split, halo patch, resident weights) each one takes at THIS batch size (yl_conv_tc_info)."""
        lib = _C.load()
        out = []
        for (fn, args, _), md in zip(self.calls, self.meta):
            if md["kind"] != "conv_tc":
                continue
            info = _C.ConvTcPlan()
            _C.check(lib.yl_conv_tc_info(args[0], C.byref(info)), "yl_conv_tc_info")
            out.append((md["desc"], info))
        return out

    def time_launches(self, reps: int = 3, inner: int = 4):
        """Per-launch device time (ms, median of `reps` eager passes in plan order) via CUDA events on the
        launching stream.  Every launch is issued `inner` times back to back between its two events and the
        elapsed time divided by `inner`: all launches are idempotent (outputs are pure functions of other buffers),
        so this measures the kernel's steady-state duration and keeps the ~5 us of event/launch latency out of a
        10 us kernel.  Cache state is the real one for the first of the `inner` launches (it runs right after its
        producers); tensors larger than L2 stream from HBM every time."""
        n = len(self.calls)
        s = _C.stream_ptr()
        times = []
        # the one exception to idempotence: head convs with the fused class filter APPEND candidates (atomic counters
        # zeroed by yl_nms_begin); they are issued once per pass so the select kernel sees each candidate once
        once = ["+filter" in md["desc"] for md in self.meta]
        for _ in range(reps):
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * n)]
            for i, (fn, args, _) in enumerate(self.calls):
                ev[2 * i].record()
                for _k in range(1 if once[i] else inner):
                    _C.check(fn(*args, s), fn.__name__)
                ev[2 * i + 1].record()
            torch.cuda.synchronize(self.device)
            times.append([ev[2 * i].elapsed_time(ev[2 * i + 1]) / (1 if once[i] else inner) for i in range(n)])
        t = torch.tensor(times).median(0).values.tolist()
        return t

    def capture(self, skip: int = 0):
        """Capture calls[skip:] into a CUDA graph (calls[:skip] stay eager, e.g. the image ingest)."""
        torch.cuda.synchronize(self.device)
        self.run_eager()  # warm-up outside capture (lazy module loading, first-touch)
        torch.cuda.synchronize(self.device)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            if any(self.lanes[skip:]):
                self._run_lanes(skip)
            else:
                self.run_eager(skip)
        self.graph = g
        self._skip = skip
        return self

    def _run_lanes(self, skip: int = 0):
        """Issue calls[skip:] with every lane on its own stream forked from the current one: a launch waits (via
        events) only for its cross-lane producers, same-lane order is stream order, and all lanes rejoin the
        current stream at the end.  Under stream capture this yields a graph with parallel branches."""
        main = torch.cuda.current_stream(self.device)
        streams = {0: main}
        n = len(self.calls)
        # fork every side lane from the capturing stream before any work is issued on it
        fork = torch.cuda.Event()
        fork.record(main)
        for lane in sorted(set(self.lanes[skip:])):
            if lane != 0:
                st = streams[lane] = torch.cuda.Stream(device=self.device)
                st.wait_event(fork)
        needed = set()                    # calls whose completion some other lane waits for
        for i in range(skip, n):
            for d in self.deps[i]:
                if d >= skip and self.lanes[d] != self.lanes[i]:
                    needed.add(d)
        events = {}
        check = _C.check
        lib = _C.load()
        for i in range(skip, n):
            fn, args, _ = self.calls[i]
            lane = self.lanes[i]
            st = streams[lane]
            cross = [d for d in self.deps[i] if d >= skip and self.lanes[d] != lane]
            for d in cross:
                st.wait_event(events[d])
            # a launch that follows an event wait keeps a plain (full) dependency: programmatic dependent launch
            # is only used between consecutive kernels of one lane
            if cross:
                lib.yl_set_pdl(0)
            rc = fn(*args, st.cuda_stream)
            if cross:
                lib.yl_set_pdl(1)
            if rc != 0:
                check(rc, fn.__name__)
            if i in needed:
                ev = events[i] = torch.cuda.Event()
                ev.record(st)
        for lane, st in streams.items():
            if lane != 0:
                ev = torch.cuda.Event()
                ev.record(st)
                main.wait_event(ev)
