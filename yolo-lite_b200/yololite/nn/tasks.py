"""Model graph of the YOLO11 detector: yaml -> module list -> static B200 launch plan.

Public surface follows reference yololite/nn/tasks.py: `DetectionModel(cfg, ch, nc, verbose)` with
`.model` (nn.Sequential, modules carry `.i .f .type .np`), `.save`, `.stride`, `.names`, `.yaml`, `.forward /
.predict`; `parse_model` (:525-664), `yaml_model_load` (:667-680), `guess_model_scale` (:683-698),
`attempt_load_one_weight / attempt_load_weights` (:461-522).  The layer loop of `_predict_once` (:118-145)
exists only at plan-build time: per input shape the whole forward is compiled into a fixed launch sequence
(optionally a CUDA graph), with skip connections and `Concat` resolved to buffer aliasing.
Test-time augmentation (`augment=True`, reference `DetectionModel._predict_augment`) runs the plans of its three input
shapes with two CUDA kernels around them (csrc/tta.cu).  Feature embeddings (`embed=[...]`) run a plan truncated after
the last tapped layer that ends in one pooling kernel (csrc/embed.cu).  A model ensemble (`Ensemble`, from
`attempt_load_weights([a.pt, b.pt, ...])`) runs all its members and one NMS in one plan.  Training-side members (loss,
criterion, profiling) are out of scope.
"""
from __future__ import annotations

import ast
import math
import re
from copy import deepcopy
from pathlib import Path
from typing import NamedTuple

import torch
import torch.nn as nn

from .. import _plan
from ..cfg import CFG_DIR, DEFAULT_CFG_DICT
from ..utils import LOGGER, yaml_load
from .modules import (C2PSA, C3, SPPF, Bottleneck, C2f, C3k, C3k2, Concat, Conv, Detect, DWConv)
from .modules._emit import YLModule, emit_any

_MODULES = {m.__name__: m for m in (Conv, DWConv, Bottleneck, SPPF, C2f, C3, C3k, C3k2, C2PSA, Concat, Detect)}
_REPEATABLE = {C2f, C3, C3k2, C2PSA}            # repeats become the module's own `n` argument
_CHANNEL_ARGS = {Conv, DWConv, Bottleneck, SPPF, C2f, C3, C3k2, C2PSA}


def make_divisible(x, divisor):
    """Smallest multiple of divisor >= x (reference utils/ops.py:101-114)."""
    if isinstance(divisor, torch.Tensor):
        divisor = int(divisor.max())
    return math.ceil(x / divisor) * divisor


def guess_model_scale(model_path) -> str:
    m = re.search(r"yolo[v]?\d+([nslmx])", Path(model_path).stem)
    return m.group(1) if m else ""


def yaml_model_load(path) -> dict:
    """'yolo11s.yaml' -> cfg/yolo11.yaml + scale 's' (reference tasks.py:667-680). Bare names resolve to the
    packaged cfg directory."""
    path = Path(path)
    unified = Path(re.sub(r"(\d+)([nslmx])(.+)?$", r"\1\3", str(path)))
    for cand in (unified, path, CFG_DIR / unified.name, CFG_DIR / path.name):
        if cand.exists():
            d = yaml_load(cand)
            break
    else:
        raise FileNotFoundError(f"model yaml '{path}' not found (also looked in {CFG_DIR})")
    d["scale"] = guess_model_scale(path)
    d["yaml_file"] = str(path)
    return d


def parse_model(d: dict, ch: int, verbose: bool = True):
    """Build the nn.Sequential of a model dict. Returns (model, sorted save list)."""
    nc, scales = d.get("nc"), d.get("scales")
    depth, width, max_channels = d.get("depth_multiple", 1.0), d.get("width_multiple", 1.0), float("inf")
    scale = d.get("scale")
    if scales:
        if not scale:
            scale = next(iter(scales))
            LOGGER.warning(f"WARNING: no model scale passed, assuming scale='{scale}'")
        depth, width, max_channels = scales[scale]
    if d.get("activation"):
        raise NotImplementedError("custom activations are not on the YOLO11 path (SiLU only)")
    legacy = True
    chs = [ch]
    layers, save = [], []
    for i, (f, n, name, args) in enumerate(d["backbone"] + d["head"]):
        args = list(args)
        if name.startswith("nn."):
            m = getattr(nn, name[3:])
        elif name in _MODULES:
            m = _MODULES[name]
        else:
            raise NotImplementedError(f"layer {i}: module '{name}' is outside the YOLO11 detection path")
        for j, a in enumerate(args):
            if isinstance(a, str):
                if a == "nc":
                    args[j] = nc
                else:
                    try:
                        args[j] = ast.literal_eval(a)
                    except (ValueError, SyntaxError):
                        pass
        n_ = n = max(round(n * depth), 1) if n > 1 else n
        if m in _CHANNEL_ARGS:
            c1, c2 = chs[f], args[0]
            if c2 != nc:
                c2 = make_divisible(min(c2, max_channels) * width, 8)
            args = [c1, c2, *args[1:]]
            if m in _REPEATABLE:
                args.insert(2, n)
                n = 1
            if m is C3k2:
                legacy = False
                if scale in "mlx":
                    args[3] = True
        elif m is Concat:
            c2 = sum(chs[x] for x in f)
        elif m is Detect:
            args.append([chs[x] for x in f])
            m.legacy = legacy
            c2 = None
        else:  # nn.Upsample, nn.Identity ...
            c2 = chs[f]
        m_ = nn.Sequential(*(m(*args) for _ in range(n))) if n > 1 else m(*args)
        m_.np = sum(p.numel() for p in m_.parameters())
        m_.i, m_.f, m_.type = i, f, f"{m.__module__}.{m.__name__}".replace("torch.nn.modules.", "torch.nn.")
        if verbose:
            LOGGER.info(f"{i:>3}{str(f):>20}{n_:>3}{m_.np:10.0f}  {m_.type:<45}{str(args):<30}")
        save.extend(x % i for x in ([f] if isinstance(f, int) else f) if x != -1)
        layers.append(m_)
        if i == 0:
            chs = []
        chs.append(c2)
    return nn.Sequential(*layers), sorted(save)


def initialize_weights(model: nn.Module):
    """Reference utils/torch_utils.py:242-252: BN eps 1e-3 / momentum 0.03, in-place activations."""
    for m in model.modules():
        if isinstance(m, nn.BatchNorm2d):
            m.eps = 1e-3
            m.momentum = 0.03
        elif isinstance(m, (nn.SiLU, nn.ReLU, nn.LeakyReLU, nn.Hardswish, nn.ReLU6)):
            m.inplace = True


#: scales and flips of DetectionModel._predict_augment (flip 3 = left-right); the reference hard-codes both
TTA_SCALES = (1, 0.83, 0.67)
TTA_FLIPS = (None, 3, None)


class TtaPass(NamedTuple):
    """Geometry of one pass of _predict_augment on an (h, w) input."""

    scale: float
    flip: int | None
    h: int            # resized content: (int(h * scale), int(w * scale)) as scale_img computes it
    w: int
    H: int            # canvas after scale_img's pad to a multiple of the largest stride
    W: int
    A: int            # anchors the model predicts on the canvas
    a0: int           # anchors [a0, a0 + n) survive _clip_augmented
    n: int


def tta_geometry(h: int, w: int, strides=(8, 16, 32)) -> list[TtaPass]:
    """The three passes of _predict_augment for an (h, w) input (a multiple of max(strides)): scale_img's content and
    canvas sizes (utils/torch_utils.py, Python double arithmetic as there) and the anchor ranges _clip_augmented keeps
    (the largest-stride level of the first pass and the smallest-stride level of the last pass are dropped)."""
    strides = [int(s) for s in strides]
    gs, nl = max(strides), len(strides)
    g = sum(4 ** x for x in range(nl))         # _clip_augmented: anchors per unit of the smallest level
    e = 1                                      # levels dropped at each end
    out = []
    for k, (si, fi) in enumerate(zip(TTA_SCALES, TTA_FLIPS)):
        if si == 1.0:                          # scale_img returns the image unchanged
            ch, cw, H, W = h, w, h, w
        else:
            ch, cw = int(h * si), int(w * si)
            H, W = (math.ceil(x * si / gs) * gs for x in (h, w))
        A = sum((H // s) * (W // s) for s in strides)
        a0, n = 0, A
        if k == 0:
            n = A - (A // g) * sum(4 ** x for x in range(e))
        elif k == len(TTA_SCALES) - 1:
            a0 = (A // g) * sum(4 ** (nl - 1 - x) for x in range(e))
            n = A - a0
        out.append(TtaPass(si, fi, ch, cw, H, W, A, a0, n))
    return out


def embed_indices(embed, n_layers: int) -> tuple[int, ...]:
    """The layer indices of `embed` as the plan key: sorted and de-duplicated (the reference's `m.i in embed` test pools
    in layer order and counts a repeated index once).  Unlike the reference, an index outside [0, n_layers - 2] raises
    ValueError: the last layer (Detect) returns a list the reference cannot pool, and the reference silently ignores a
    negative index and then returns detections."""
    if isinstance(embed, (str, bytes)) or not hasattr(embed, "__iter__"):
        raise TypeError(f"embed must be a list of layer indices, got {embed!r}")
    idx = set()
    for i in embed:
        if isinstance(i, bool) or not hasattr(i, "__index__"):
            raise TypeError(f"embed index {i!r} is not an int")
        i = i.__index__()
        if not 0 <= i <= n_layers - 2:
            raise ValueError(f"embed index {i} is outside [0, {n_layers - 2}] (layers 0..{n_layers - 2} precede the head)")
        idx.add(i)
    if not idx:
        raise ValueError("embed needs at least one layer index")
    return tuple(sorted(idx))


def fused_up_guard(layers):
    """Indices of layers whose output feeds an nn.Upsample (those producers need the dual-destination conv)."""
    out = set()
    for u, m in enumerate(layers):
        if isinstance(m, nn.Upsample):
            f = m.f if isinstance(m.f, int) else m.f[0]
            out.add(u - 1 if f == -1 else f)
    return out


def _lru(store: dict, key, limit, dev, build):
    """`store[key]`, made the most recently used entry (dicts keep insertion order); on a miss `build()` makes it, after
    the least recently used entry is evicted when `limit` entries are kept.  An evicted plan's buffers / graph may still
    be in flight on some stream, and the caching allocator would hand them to the new plan: the device is drained first
    (rare, build-time cost)."""
    entry = store.get(key)
    if entry is not None:
        store[key] = store.pop(key)
        return entry
    if len(store) >= max(int(limit), 1):
        torch.cuda.synchronize(dev)
        store.pop(next(iter(store)))
    entry = store[key] = build()
    return entry


def _nms_key(conf, iou, classes, agnostic, multi_label, max_det, max_nms, max_wh) -> tuple:
    """The NMS arguments of infer_nms as the hashable tuple of Builder.nms (part of the plan key)."""
    if classes is not None and not isinstance(classes, (list, tuple)):
        classes = [classes] if isinstance(classes, int) else list(classes)      # `classes=0` is legal in the reference
    return (float(conf), float(iou), None if classes is None else tuple(int(c) for c in classes), bool(agnostic),
            bool(multi_label), int(max_det), int(max_nms), float(max_wh))


class BaseModel(YLModule):
    """Layer-list model executed through a cached static plan (one per input shape and device)."""

    #: capture each plan into a CUDA graph (one launch per forward); set False to debug launch by launch
    use_cuda_graph = True
    #: plans kept per model (LRU): every (shape, slot, NMS arguments) owns activation buffers + a CUDA graph, so a
    #: stream of differently shaped rect batches or a conf/iou sweep must not grow GPU memory without bound
    max_plans = 16
    #: return fresh tensors from forward() like the reference; engine code uses infer() and skips the copy
    clone_outputs = True

    def forward(self, x, *args, **kwargs):
        if isinstance(x, dict):
            raise NotImplementedError("training/loss is out of scope: yololite is the inference path")
        return self.predict(x, *args, **kwargs)

    def predict(self, x, profile=False, visualize=False, augment=False, embed=None):
        """Module-level forward: (y (B, 4+nc, A), [raw (B, no, H, W)]) like the reference; with `augment=True` the
        merged test-time-augmentation prediction and None, like `_predict_augment`.  With `embed=[layer indices]` (and
        no `augment`, which wins as in the reference) the tuple of B per-image feature vectors of `_predict_once`: the
        per-channel spatial means of the tapped layers' outputs, concatenated in layer order (see `infer_embed`)."""
        if visualize or profile:
            raise NotImplementedError("visualize / profile are not part of the inference hot path")
        if augment and self._augment_supported():
            y, _ = self.infer(x, augment=True)
            return (y.clone() if self.clone_outputs else y), None
        if embed:
            e = self.infer_embed(x, embed)
            return torch.unbind(e.clone() if self.clone_outputs else e, 0)
        out = self.infer(x, want_raw=True)   # the module-level API returns the raw head maps like the reference
        if self.clone_outputs:
            y, raws = out
            return y.clone(), [r.clone() for r in raws]
        return out

    _predict_once = predict

    # ------------------------------------------------------------------ plan
    def _layer_scales(self):
        """Down-sampling factor of every layer output w.r.t. the image (replaces the 256x256 probe forward of
        the reference, tasks.py:258-268)."""
        sc = []
        for m in self.model:
            f = m.f
            src = (sc[f] if f != -1 else (sc[-1] if sc else 1.0)) if isinstance(f, int) else \
                [(sc[j] if j != -1 else sc[-1]) for j in f]
            if isinstance(m, Conv):
                s = src * m.conv.stride[0]
            elif isinstance(m, nn.Upsample):
                s = src / float(m.scale_factor)
            elif isinstance(m, Concat):
                s = src[0]
            elif isinstance(m, Detect):
                s = src
            else:
                s = src
            sc.append(s)
        return sc

    def _emit(self, g, x, out=None, embed=None):
        """Record the whole forward. Concat layers whose inputs each feed exactly one Concat become aliasing:
        the producers are handed a slice of the concat buffer as their destination.

        `embed`: sorted layer indices (embed_indices).  Only layers 0..max(embed) are recorded, and the return value is
        the list of the tapped layers' output Views (a buffer, a concat slice, a Concat's whole buffer or a fused
        upsample's replicated copy).

        `out`: None, or (y, anchor base): the Detect head writes its anchors into that window of a wider prediction y
        (Detect._emit; one member of an ensemble plan)."""
        from .._ops import View

        layers = list(self.model)
        n_layers = len(layers)
        # absolute source indices per layer
        srcs = []
        for i, m in enumerate(layers):
            f = [m.f] if isinstance(m.f, int) else list(m.f)
            srcs.append([(i - 1 if j == -1 else (j if j >= 0 else i + j)) for j in f])
        # placement: producer layer -> (concat layer, channel offset) when it feeds exactly one Concat
        n_cat_uses = [0] * n_layers
        for i, m in enumerate(layers):
            if isinstance(m, Concat):
                for j in srcs[i]:
                    if j >= 0:
                        n_cat_uses[j] += 1
        place, cat_buf = {}, {}
        for i, m in enumerate(layers):
            if isinstance(m, Concat) and all(j >= 0 and n_cat_uses[j] == 1 for j in srcs[i]) \
                    and len(set(srcs[i])) == len(srcs[i]):
                for j in srcs[i]:
                    place[j] = i
        ys: list = [None] * n_layers
        out_ch = {}

        def dest_for(j):
            ci = place.get(j)
            if ci is None:
                return None

            def resolve(n, h, w, c, j=j, ci=ci):
                if ci not in cat_buf:
                    # channel counts of all sources are known statically from the modules
                    chans = [self._out_channels(layers, k, out_ch) for k in srcs[ci]]
                    cat_buf[ci] = (g.alloc(n, h, w, sum(chans)), chans)
                buf, chans = cat_buf[ci]
                off = sum(chans[: srcs[ci].index(j)])
                return buf.slice(off, c)

            return _plan.Dest(resolve)

        # nn.Upsample fused into its producer: when layer j ends in a dense conv, that conv's TMA store also
        # writes the 2x2-replicated copy straight into the upsample's destination (usually a Concat slice)
        n_uses = [0] * n_layers
        for i in range(n_layers):
            for j in srcs[i]:
                if j >= 0:
                    n_uses[j] += 1
        fused_up = {}                    # producer layer j -> upsample layer u
        for u, m in enumerate(layers):
            if isinstance(m, nn.Upsample) and m.mode == "nearest" and float(m.scale_factor) == 2.0:
                j = srcs[u][0]
                if embed is not None and u > embed[-1]:
                    continue             # the upsample is never emitted: its producer writes only its plain output
                if j >= 0 and isinstance(layers[j], (Conv, C2f, C3, SPPF, C2PSA)) and j not in fused_up:
                    fused_up[j] = u
        done_up = {}

        # layers 0 + 1 as one launch (image ingest + two stride-2 3x3 convs) when layer 0 feeds only layer 1
        # (layer 0's output never leaves shared memory there, so a tap on it takes the unfused stem)
        fuse_stem = not (embed is not None and 0 in embed) and self._stem_fusable(g, x, layers, srcs, n_uses)
        cur = x
        for i, m in enumerate(layers):
            if embed is not None and i > embed[-1]:
                return [ys[k] for k in embed]
            g.layer = i
            if fuse_stem and i == 0:
                continue
            if fuse_stem and i == 1:
                from .modules._emit import act_flag, packed

                l0, l1 = layers[0], layers[1]
                cur = ys[1] = g.stem_fused(x, packed(l0.conv, l0.bn, l0), packed(l1.conv, l1.bn, l1), act_flag(l0.act),
                                           act_flag(l1.act), out=dest_for(1))
                continue
            inp = [ys[j] if j >= 0 else x for j in srcs[i]]
            if isinstance(m, Detect):
                return m._emit(g, inp, out=out)
            if isinstance(m, Concat):
                if i in cat_buf and all(place.get(j) == i for j in srcs[i]):
                    buf, chans = cat_buf[i]
                    cur = View(buf.buf, buf.coff, sum(chans))   # sources already live in the buffer
                else:
                    cur = m._emit(g, inp, out=dest_for(i))
            elif i in done_up:
                cur = done_up[i]
            elif i in fused_up:
                u = fused_up[i]
                dd = _plan.DualDest(dest_for(i), dest_for(u))
                cur = emit_any(g, m, inp[0], out=dd)
                assert dd.up_view is not None, f"layer {i}: producer did not honour the fused upsample"
                done_up[u] = dd.up_view
            else:
                cur = emit_any(g, m, inp[0], out=dest_for(i))
            ys[i] = cur
        return cur

    #: run layers 0 and 1 as one kernel when the shapes allow (YL_STEM_FUSE=0 disables)
    fuse_stem = True

    def _stem_fusable(self, g, x, layers, srcs, n_uses):
        import os

        from .. import _C

        if not self.fuse_stem or os.environ.get("YL_STEM_FUSE", "1") == "0" or len(layers) < 3:
            return False
        if not isinstance(x, _plan.NchwInput) or x.view is not None or len(g.calls) != g.model_start:
            return False
        l0, l1 = layers[0], layers[1]
        if type(l0) is not Conv or type(l1) is not Conv or srcs[1] != [0] or n_uses[0] != 1 or 1 in fused_up_guard(layers):
            return False
        for cv in (l0, l1):
            c = cv.conv
            if c.kernel_size != (3, 3) or c.stride != (2, 2) or c.groups != 1 or not hasattr(cv, "bn") or c.bias is not None:
                return False
        if l0.conv.in_channels != x.c:
            return False
        return bool(_C.load().yl_stem_fused_supported(x.c, l0.conv.out_channels, l1.conv.out_channels))

    @staticmethod
    def _out_channels(layers, k, memo):
        if k in memo:
            return memo[k]
        m = layers[k]
        if isinstance(m, Conv):
            c = m.conv.out_channels
        elif isinstance(m, (C2f, SPPF, C2PSA, C3)):
            c = m.cv2.conv.out_channels if not isinstance(m, C3) else m.cv3.conv.out_channels
        elif isinstance(m, Concat):
            f = [m.f] if isinstance(m.f, int) else list(m.f)
            c = sum(BaseModel._out_channels(layers, (k - 1 if j == -1 else j), memo) for j in f)
        elif isinstance(m, nn.Sequential):
            c = BaseModel._out_channels(list(m), len(m) - 1, {})
        else:  # Upsample / Identity: same as its input
            j = m.f if isinstance(m.f, int) else m.f[0]
            c = BaseModel._out_channels(layers, k - 1 if j == -1 else j, memo)
        memo[k] = c
        return c

    def _get_plan(self, shape, dev, want_raw=False, slot=0, nms=None, embed=None):
        """`nms`: None or the hashable argument tuple of Builder.nms: the plan then ends with the batched NMS and its
        entry carries (dets, counts) instead of the raw head maps.  `embed`: None or the index tuple of embed_indices:
        the plan stops after layer max(embed) and ends with the pooling launch; its entry carries the (B, D) fp32
        embeddings in place of `y` and no raw maps."""
        plans = self.__dict__.setdefault("_yl_plans", {})
        key = (tuple(shape), dev.index, bool(self.use_cuda_graph), bool(want_raw), int(slot), nms, embed)

        def build():
            with torch.cuda.device(dev):
                g = _plan.Builder(dev)
                g.want_raw = bool(want_raw)   # Detect writes its raw (B, H, W, no) maps only on request
                if nms is not None and not nms[4] and nms[2] is None:
                    g.nms_fuse_conf = float(nms[0])   # single-label, no class filter: the head may filter in its epilogue
                static_in = torch.zeros(tuple(shape), dtype=torch.float32, device=dev)
                xin = g.input_nchw(static_in)
                if embed is not None:
                    y, raws = g.embed_pool(self._emit(g, xin, embed=embed)), []
                else:
                    y, raws = self._emit(g, xin)
                post = g.nms(y, *nms) if nms is not None else None
                plan = g.finish()
                if self.use_cuda_graph:
                    plan.capture(skip=1)     # the image ingest stays eager so it can read the caller's tensor
                raw_views = [r.buf.permute(0, 3, 1, 2) for r in raws]   # (B, no, H, W) views, zero-copy
                return plan, static_in, y, raw_views if post is None else post

        return _lru(plans, key, self.max_plans, dev, build)

    @torch.no_grad()
    def infer(self, x: torch.Tensor, want_raw: bool = False, slot: int = 0, augment: bool = False):
        """Engine entry: NCHW float image batch on CUDA -> (y (B, 4+nc, A) fp32, [raw (B, no, H, W) views]).

        `augment=True`: test-time augmentation (reference `_predict_augment`) -> (merged (B, 4+nc, A_tta), []), boxes in
        the pixels of `x`; `merged` aliases a buffer of this (shape, device, slot) that the next such call overwrites.

        `slot` selects one of several independent plans (own activation buffers and CUDA graph) for the same
        shape, so a caller can keep two batches in flight on two streams: the launch-latency-bound small layers
        of one batch then overlap the bandwidth-bound large layers of the other.

        The raw head maps are only needed by callers of the module-level API (`forward`); the engine path
        (`want_raw=False`) gets an empty list and the plan never writes them.  The returned tensors alias the
        plan's static buffers and are overwritten by the next call with the same shape."""
        dev = self._engine_device(x)
        if augment and self._augment_supported():
            return self._infer_tta(x, dev, slot)["merged"], []
        plan, static_in, y, raws = self._get_plan(x.shape, dev, want_raw, slot)
        self._run_plan(plan, static_in, x, dev)
        return y, raws

    def _engine_device(self, x) -> torch.device:
        """The device of an engine-entry batch, after the checks every entry makes."""
        if not isinstance(x, torch.Tensor) or x.dim() != 4:
            raise TypeError("expected a (B, C, H, W) tensor")
        if not x.is_cuda:
            raise RuntimeError("yololite runs on CUDA (sm_100) only; move the input with .cuda() "
                               "(there is no CPU fallback)")
        dev = x.device
        p0 = next(self.parameters())
        if p0.device != dev:
            raise RuntimeError(f"model is on {p0.device} but input is on {dev}")
        s = int(self.stride.max()) if hasattr(self, "stride") else 32
        if x.shape[2] % s or x.shape[3] % s:
            raise ValueError(f"image size {tuple(x.shape[2:])} must be a multiple of the model stride {s}")
        return dev

    @torch.no_grad()
    def infer_embed(self, x: torch.Tensor, embed, slot: int = 0) -> torch.Tensor:
        """Engine entry for feature embeddings: NCHW image batch on CUDA (fp32, fp16 or uint8 bytes, read like `infer`)
        -> (B, D) fp32, row b the embedding of image b: for every layer index of `embed` in layer order (repeats count
        once) the per-channel spatial mean of that layer's output, D the sum of their channel counts.  That is the
        reference's `_predict_once(x, embed=...)`: the plan records layers 0..max(embed) only, then one yl_embed_pool
        launch.  Indices must lie in [0, len(model) - 2] (ValueError otherwise, see embed_indices).  The result
        aliases a buffer of this plan (shape, device, slot, indices) that the next such call overwrites."""
        dev = self._engine_device(x)
        idx = embed_indices(embed, len(self.model))
        plan, static_in, out, _ = self._get_plan(x.shape, dev, False, slot, embed=idx)
        self._run_plan(plan, static_in, x, dev)
        return out

    # ------------------------------------------------------------------ test-time augmentation
    def _augment_supported(self) -> bool:
        """Only a detection model has the TTA path; anything else predicts single-scale with the reference's warning."""
        if isinstance(self.model[-1], Detect) and not getattr(self, "end2end", False):
            return True
        LOGGER.warning("WARNING: Model does not support 'augment=True', reverting to single-scale prediction.")
        return False

    def _infer_tta(self, x, dev, slot):
        """_predict_augment on the engine path: pass 0 is the plain plan of `x` (same ingest, uint8 / fp16 read natively),
        yl_tta_scale_img writes the flipped / rescaled inputs of passes 1 and 2 straight into their plans' static inputs,
        the two plans replay, and yl_tta_merge builds the merged prediction in a buffer of the returned TTA state (keyed
        and bounded like the plans).  Asynchronous: nothing here waits for the device."""
        from .. import _C, _ops

        B, C, H, W = x.shape
        geo = tta_geometry(H, W, self.model[-1].stride.tolist())
        plans, shapes = [], []
        for k, p in enumerate(geo):
            shape = (B, C, p.H, p.W)
            # the three outputs must coexist until the merge: a canvas equal to an earlier pass's shape (small inputs,
            # where the rescaled canvas pads back to the same size) gets a plan slot of its own; callers use slots >= 0
            plans.append(self._get_plan(shape, dev, False, slot if shape not in shapes else -(3 * int(slot) + k)))
            shapes.append(shape)
        for (_, _, y, _), p in zip(plans, geo):
            assert y.shape[2] == p.A, (tuple(y.shape), p)
        st = self._tta_state(x.shape, dev, slot, plans[0][2].shape[1], sum(p.n for p in geo))
        plan0, in0, _, _ = plans[0]
        self._run_plan(plan0, in0, x, dev)
        xs = x if x.dtype in _C.INGEST_DTYPES else x.float()
        xs = xs if xs.is_contiguous() else xs.contiguous()
        with torch.cuda.device(dev):
            _ops.tta_scale_img(xs, [(plans[k][1], (geo[k].h, geo[k].w), geo[k].flip) for k in (1, 2)])
            plans[1][0].run()
            plans[2][0].run()
            _ops.tta_merge([(plans[k][2], p.a0, p.n, p.scale, p.flip) for k, p in enumerate(geo)], W, st["merged"])
        return st

    def _tta_state(self, shape, dev, slot, rows, anchors):
        """Output buffers of test-time augmentation for one (input shape, device, slot): the merged prediction and the
        NMS outputs per argument set.  LRU-bounded by `max_plans`, like the plans."""
        states = self.__dict__.setdefault("_yl_tta", {})
        key = (tuple(shape), dev.index, int(slot))
        st = states.get(key)
        if st is not None:
            states[key] = states.pop(key)
            return st
        if len(states) >= max(int(self.max_plans), 1):
            torch.cuda.synchronize(dev)          # the evicted buffers may still be in use on some stream
            states.pop(next(iter(states)))
        st = states[key] = {"merged": torch.empty((shape[0], rows, anchors), dtype=torch.float32, device=dev), "nms": {}}
        return st

    @staticmethod
    def _run_plan(plan, static_in, x, dev):
        """Feed `x` to the plan's ingest.  fp32 is read in place (zero-copy); fp16 is widened and uint8 is taken as
        image bytes (value / 255, the predictor's `/255`, predictor.py:84) — inside the fused stem when the plan has one,
        otherwise by one conversion launch into the plan's static fp32 input."""
        from .. import _C

        with torch.cuda.device(dev):
            yd = _C.INGEST_DTYPES.get(x.dtype)
            if yd is not None and x.is_contiguous() and yd in plan.native_ingest and x.data_ptr() % 16 == 0:
                plan.run(ingest_ptr=x.data_ptr(), ingest_dtype=yd)
            elif yd in (_C.YL_F16, _C.YL_U8) and x.is_contiguous() and x.data_ptr() % 16 == 0:
                _C.check(_C.load().yl_to_f32(x.data_ptr(), yd, static_in.data_ptr(), x.numel(), _C.stream_ptr()), "yl_to_f32")
                plan.run()
            else:
                if x.dtype == torch.uint8:
                    static_in.copy_(x.float() / 255, non_blocking=True)
                else:
                    static_in.copy_(x, non_blocking=True)
                plan.run()

    @torch.no_grad()
    def infer_nms(self, x: torch.Tensor, conf=0.25, iou=0.45, classes=None, agnostic=False, multi_label=False,
                  max_det=300, max_nms=30000, max_wh=7680.0, slot: int = 0, augment: bool = False):
        """Engine entry for a whole step: NCHW float batch on CUDA -> (dets (B, max_det, 6), counts (B,) int32), the
        padded output of `ops.nms_padded(self.infer(x)[0], ...)`, with the NMS kernels recorded in the same plan /
        CUDA graph as the model (ingest + one graph launch per step).  The returned tensors alias plan buffers and
        are overwritten by the next call with the same shape, arguments and slot.

        `augment=True`: the same NMS on the merged test-time-augmentation prediction of `infer(x, augment=True)`, into
        buffers of its TTA state (same aliasing rule)."""
        if not isinstance(x, torch.Tensor) or x.dim() != 4 or not x.is_cuda:
            raise RuntimeError("infer_nms expects a (B, C, H, W) CUDA tensor (yololite has no CPU fallback)")
        dev = x.device
        s = int(self.stride.max()) if hasattr(self, "stride") else 32
        if x.shape[2] % s or x.shape[3] % s:
            raise ValueError(f"image size {tuple(x.shape[2:])} must be a multiple of the model stride {s}")
        nms = _nms_key(conf, iou, classes, agnostic, multi_label, max_det, max_nms, max_wh)
        if augment and self._augment_supported():
            from .. import _ops

            st = self._infer_tta(x, dev, slot)
            out = st["nms"].pop(nms, None)
            if out is None:
                if len(st["nms"]) >= max(int(self.max_plans), 1):
                    torch.cuda.synchronize(dev)
                    st["nms"].pop(next(iter(st["nms"])))
                cls_t = None if nms[2] is None else torch.tensor(nms[2], dtype=torch.int32, device=dev)
                out = (torch.empty((x.shape[0], nms[5], 6), dtype=torch.float32, device=dev),
                       torch.empty((x.shape[0],), dtype=torch.int32, device=dev), cls_t)
            st["nms"][nms] = out                 # most recently used last
            with torch.cuda.device(dev):
                return _ops.nms_batched(st["merged"], conf, iou, out[2], agnostic, multi_label, max_det, max_nms, max_wh,
                                        out=out[0], counts=out[1])
        plan, static_in, _, post = self._get_plan(x.shape, dev, False, slot, nms)
        self._run_plan(plan, static_in, x, dev)
        return post

    def fuse(self, verbose=True):
        """Reference API (AutoBackend calls model.fuse(), autobackend.py:74; the reference deleted the method
        and crashes there).  BN is always folded at plan build, so this is a no-op returning self."""
        return self


class DetectionModel(BaseModel):
    """YOLO11 detection model built from a yaml dict or path."""

    def __init__(self, cfg="yolo11n.yaml", ch=3, nc=None, verbose=True):
        super().__init__()
        self.yaml = cfg if isinstance(cfg, dict) else yaml_model_load(cfg)
        ch = self.yaml["ch"] = self.yaml.get("ch", ch)
        if nc and nc != self.yaml["nc"]:
            LOGGER.info(f"Overriding model.yaml nc={self.yaml['nc']} with nc={nc}")
            self.yaml["nc"] = nc
        self.model, self.save = parse_model(deepcopy(self.yaml), ch=ch, verbose=verbose)
        self.names = {i: f"{i}" for i in range(self.yaml["nc"])}
        self.inplace = self.yaml.get("inplace", True)
        self.end2end = False
        m = self.model[-1]
        if isinstance(m, Detect):
            m.inplace = self.inplace
            m.stride = torch.tensor([float(s) for s in self._layer_scales()[-1]])
            self.stride = m.stride
            m.bias_init()
        else:
            self.stride = torch.Tensor([32])
        initialize_weights(self)


_ENSEMBLE_NO_EMBED = ("embed=[...] is not available for a model ensemble: its members have no common feature space "
                      "(the reference's Ensemble.forward takes no embed); embed with one member instead")


def _member_nc(m) -> int:
    """Class count of an ensemble member: its `nc` attribute, or its Detect head's for a checkpoint's model without one."""
    return int(m.nc) if hasattr(m, "nc") else int(m.model[-1].nc)


class Ensemble(nn.ModuleList):
    """Model ensemble (reference `Ensemble`, nn/tasks.py): every member runs on the same batch and their (B, 4+nc, A_k)
    predictions are concatenated along the anchor axis in member order (anchors member-major, then as in each member),
    so one NMS runs over the candidates of all members (the "NMS ensemble").

    `names`, `nc` and `yaml` are member 0's, `stride` is that of the member with the largest `stride.max()`; members
    must agree on the class count (AssertionError `Models differ in class counts [...]`) and the input channel count
    (ValueError).  A member without an `nc` attribute (a checkpoint's model) counts with its Detect head's `nc`.

    On the engine path one step is ONE plan: each member's image ingest (the launch it would get alone) reads the
    caller's batch, outside the CUDA graph; the rest of every member and the NMS are one graph replay.  The members'
    heads write straight into their anchor windows of one shared prediction, and with single-label NMS without a class
    filter they append their candidates to one workspace that a single select launch finishes (DESIGN.md §3.7)."""

    #: capture each plan into a CUDA graph; set False to debug launch by launch
    use_cuda_graph = True
    #: plans kept (LRU), as BaseModel.max_plans
    max_plans = 16
    #: return fresh tensors from forward() like the reference; engine code uses infer() and skips the copy
    clone_outputs = True
    #: lane ids of one member in the plan: each member's graph branches are independent of the other members'
    _member_lanes = 16

    def __init__(self, modules=None):
        super().__init__(modules)
        if not len(self):
            return
        ncs = [_member_nc(m) for m in self]
        assert all(ncs[0] == n for n in ncs), f"Models differ in class counts {ncs}"
        chs = [next(p for p in m.parameters() if p.dim() == 4).shape[1] for m in self]   # the first conv's input
        if any(c != chs[0] for c in chs):
            raise ValueError(f"ensemble members differ in input channel counts {chs}")
        self.names, self.nc, self.yaml = self[0].names, ncs[0], self[0].yaml
        self.stride = self[int(torch.argmax(torch.tensor([float(m.stride.max()) for m in self])))].stride

    _engine_device = BaseModel._engine_device

    def forward(self, x, augment=False, profile=False, visualize=False, embed=None):
        """(torch.cat([m(x)[0] for m in self], 2), None) like the reference.  `augment=True` logs a warning and predicts
        single-scale: the reference passes it into its members' `profile` slot and never runs TTA.  `embed` raises
        TypeError."""
        if embed:
            raise TypeError(_ENSEMBLE_NO_EMBED)
        if visualize or profile:
            raise NotImplementedError("visualize / profile are not part of the inference hot path")
        y, _ = self.infer(x, augment=augment)
        return (y.clone() if self.clone_outputs else y), None

    def predict(self, x, profile=False, visualize=False, augment=False, embed=None):
        """BaseModel.predict's signature over `forward`."""
        return self.forward(x, augment, profile, visualize, embed)

    @staticmethod
    def _single_scale(augment):
        if augment:
            LOGGER.warning("WARNING: test-time augmentation is not applied to model ensembles (the reference's "
                           "Ensemble.forward never runs it); predicting single-scale.")

    @torch.no_grad()
    def infer(self, x: torch.Tensor, want_raw: bool = False, slot: int = 0, augment: bool = False):
        """Engine entry, BaseModel.infer's signature: NCHW batch on CUDA (fp32, fp16 or uint8 image bytes) ->
        (y (B, 4+nc, sum of the members' anchors) fp32, []).  An ensemble has no raw head maps: `want_raw` returns
        none.  `augment=True` predicts single-scale (see forward).  y aliases a plan buffer that the next call with
        the same shape and slot overwrites."""
        dev = self._engine_device(x)
        self._single_scale(augment)
        plan, static_in, y, _ = self._get_plan(x.shape, dev, slot)
        BaseModel._run_plan(plan, static_in, x, dev)
        return y, []

    @torch.no_grad()
    def infer_nms(self, x: torch.Tensor, conf=0.25, iou=0.45, classes=None, agnostic=False, multi_label=False,
                  max_det=300, max_nms=30000, max_wh=7680.0, slot: int = 0, augment: bool = False):
        """Engine entry for a whole step, BaseModel.infer_nms's signature: the padded (dets (B, max_det, 6), counts (B,)
        int32) of `ops.nms_padded(self.infer(x)[0], ...)`, with the NMS in the same plan / CUDA graph as the members.
        The returned tensors alias plan buffers (same rule as BaseModel.infer_nms)."""
        dev = self._engine_device(x)
        self._single_scale(augment)
        nms = _nms_key(conf, iou, classes, agnostic, multi_label, max_det, max_nms, max_wh)
        plan, static_in, _, post = self._get_plan(x.shape, dev, slot, nms)
        BaseModel._run_plan(plan, static_in, x, dev)
        return post

    def infer_embed(self, x, embed, slot: int = 0):
        raise TypeError(_ENSEMBLE_NO_EMBED)

    def _get_plan(self, shape, dev, slot=0, nms=None):
        """(plan, static input, y, (dets, counts) or None) of one (shape, device, slot, NMS arguments), LRU-bounded by
        `max_plans`."""
        plans = self.__dict__.setdefault("_yl_plans", {})
        key = (tuple(shape), dev.index, bool(self.use_cuda_graph), int(slot), nms)
        return _lru(plans, key, self.max_plans, dev, lambda: self._build_plan(shape, dev, nms))

    def _build_plan(self, shape, dev, nms):
        B, _, H, W = shape
        heads = [m.model[-1] for m in self]
        if not all(isinstance(h, Detect) for h in heads):
            raise NotImplementedError("ensemble members must end in a Detect head")
        counts = [sum((H // int(s)) * (W // int(s)) for s in h.stride.tolist()) for h in heads]
        A = sum(counts)
        with torch.cuda.device(dev):
            g = _plan.Builder(dev)
            g.want_raw = False
            if nms is not None and not nms[4] and nms[2] is None:
                g.nms_fuse_conf = float(nms[0])
            static_in = torch.zeros(tuple(shape), dtype=torch.float32, device=dev)
            y = torch.empty((B, 4 + self.nc, A), dtype=torch.float32, device=dev)
            g.buffers.append(y)
            # the class filter runs in the heads only if every member can run it; the guards see the whole prediction
            if g.nms_fuse_conf is not None and all(h._fuses_filter(g, A) for h in heads):
                g.nms_begin(B, A, self.nc)
            ingest, base = [], 0
            for k, (m, n) in enumerate(zip(self, counts)):
                with g.model(lane_base=k * self._member_lanes):
                    ingest.append(g.model_start)
                    got, _ = m._emit(g, g.input_nchw(static_in), out=(y, base))
                assert got is y
                base += n
            post = g.nms(y, *nms) if nms is not None else None
            g.hoist(ingest)
            g.n_ingest = len(ingest)
            plan = g.finish()
            if self.use_cuda_graph:
                plan.capture(skip=plan.n_ingest)     # the ingests stay eager so they can read the caller's tensor
        return plan, static_in, y, post

    def fuse(self, verbose=True):
        """BN is folded at plan build (BaseModel.fuse): a no-op returning self."""
        return self


def torch_safe_load(weight):
    """torch.load of a reference/Ultralytics-format checkpoint: the pickled module classes resolve to this
    package's classes because the module paths are identical (`yololite.nn.tasks.DetectionModel`, ...)."""
    ckpt = torch.load(weight, map_location="cpu", weights_only=False)
    if not isinstance(ckpt, dict):
        ckpt = {"model": ckpt.model if hasattr(ckpt, "model") else ckpt}
    return ckpt, weight


def guess_model_task(model) -> str:
    return "detect"


def attempt_load_one_weight(weight, device=None, inplace=True, fuse=False):
    """Load a single checkpoint -> (model in eval mode, ckpt dict). Reference tasks.py:499-522."""
    ckpt, weight = torch_safe_load(weight)
    args = {**DEFAULT_CFG_DICT, **(ckpt.get("train_args") or {})}
    model = (ckpt.get("ema") or ckpt["model"]).to(device).float()
    model.args = {k: v for k, v in args.items() if k in DEFAULT_CFG_DICT}
    model.pt_path = weight
    model.task = guess_model_task(model)
    if not hasattr(model, "stride"):
        model.stride = torch.tensor([32.0])
    model = model.eval()
    for m in model.modules():
        if hasattr(m, "inplace"):
            m.inplace = inplace
    return model, ckpt


def attempt_load_weights(weights, device=None, inplace=True, fuse=False):
    """Reference tasks.py:461-496: every checkpoint of `weights` (a path or a list of paths) loaded as by
    attempt_load_one_weight.  One checkpoint returns its model itself; two or more return an `Ensemble` of them (see
    there: names / nc / yaml of member 0, the largest stride, class counts must agree; a member without an `nc`
    attribute counts with its Detect head's)."""
    ws = weights if isinstance(weights, list) else [weights]
    models = [attempt_load_one_weight(w, device, inplace, fuse)[0] for w in ws]
    if len(models) == 1:
        return models[0]
    LOGGER.info(f"Ensemble created with {weights}\n")
    return Ensemble(models)
