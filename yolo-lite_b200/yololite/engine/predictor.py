"""DetectionPredictor (reference yololite/engine/predictor.py:21-323): preprocess -> inference -> postprocess
per batch, yielding `Results`.  The three stages keep the reference's names and the `speed` dict; what changed:

  * inference is one CUDA-graph replay of the model plan (reference: ~300 ATen launches);
  * postprocess keeps detections on the device: batched NMS + box rescale/clip kernels, one host read of the
    counts, and no device->host copy of the input batch for tensor sources unless a caller asks for
    `orig_img` (the reference always converts the whole batch to uint8 numpy, ops.py:487-488);
  * a HOST tensor batch is ingested in chunks: chunk k+1's host->device copy runs on a copy stream while the
    model + NMS of chunk k run on the compute stream, so the PCIe transfer (the e2e bound for fp32 images:
    4.9 MB per 640x640 image) overlaps the whole GPU pipeline instead of preceding it;
  * `embed=[layer indices]` yields one feature vector (1-D fp32 tensor) per image instead of `Results`, as the
    reference's stream loop does; the model runs only up to the last tapped layer (`BaseModel.infer_embed`);
  * saving / plotting / video writing (predictor.py:248-323) are I/O features outside the hot path.
"""
from __future__ import annotations

import threading

import numpy as np
import torch

from .. import _C
from ..cfg import DEFAULT_CFG, get_cfg
from ..data import LetterBox, load_inference_source
from ..nn.autobackend import AutoBackend
from ..nn.tasks import _ENSEMBLE_NO_EMBED, Ensemble, embed_indices
from ..utils import LOGGER, ops
from ..utils.torch_utils import select_device, smart_inference_mode
from .results import BatchDetections, Results


class _LazyTensorImage:
    """orig_img stand-in for tensor sources: converts to HWC uint8 numpy only when somebody looks at it."""

    def __init__(self, batch: torch.Tensor, i: int):
        self._b, self._i = batch, i
        self.shape = (batch.shape[2], batch.shape[3], batch.shape[1])

    def __array__(self, dtype=None, copy=None):
        im = self._b[self._i].permute(1, 2, 0)
        a = (im if im.dtype == torch.uint8 else (im.float() * 255).clamp(0, 255).to(torch.uint8)).cpu().numpy()
        return a.astype(dtype) if dtype is not None else a


class DetectionPredictor:
    def __init__(self, cfg=DEFAULT_CFG, overrides=None):
        self.args = get_cfg(cfg, overrides)
        if self.args.conf is None:
            self.args.conf = 0.25
        if self.args.embed and self.args.augment:
            # the reference would yield the merged TTA prediction and then None in place of feature vectors
            raise ValueError("embed and augment=True cannot be combined: embeddings come from a single-scale pass")
        if self.args.save or self.args.save_txt or self.args.save_crop or self.args.show:
            if self.args.verbose:
                LOGGER.info("save/show requested: result files and plots are outside yololite's scope; ignored")
        self.done_warmup = False
        self.model = None
        self.data = self.args.data
        self.imgsz = None
        self.device = None
        self.dataset = None
        self.batch = None
        self.results = None
        self.seen = 0
        self.source_type = None
        self._lock = threading.Lock()

    # ------------------------------------------------------------------ stages
    def pre_transform(self, im):
        same_shapes = len({x.shape for x in im}) == 1
        letterbox = LetterBox(self.imgsz, auto=same_shapes and self.model.pt, stride=self.model.stride)
        return [letterbox(image=x) for x in im]

    def preprocess(self, im):
        """BCHW float tensor: `.to(device).float()`.  list of HWC BGR uint8 images: LetterBox, BGR->RGB, HWC->CHW,
        float, /255 as ONE CUDA kernel over the raw bytes (bit-exact against the reference's cv2 path): the upload
        is the uint8 pixels, 4x fewer PCIe bytes than the fp32 batch of the reference (predictor.py:67-85)."""
        if isinstance(im, torch.Tensor):
            im = im.to(self.device, non_blocking=True)
            # uint8 = image bytes: kept narrow, the model's ingest divides by 255 on the fly (yl_stem_fused / yl_to_f32)
            return im if im.dtype in (torch.uint8, torch.float16, torch.float32) else im.float()
        same_shapes = len({x.shape for x in im}) == 1
        if all(isinstance(x, np.ndarray) and x.dtype == np.uint8 and x.ndim == 3 and x.shape[2] == 3 for x in im):
            from ..data.augment import _Staging, letterbox_batch_cuda

            stg = self.model.__dict__.setdefault("_yl_lb_staging", _Staging())   # survives the per-call predictor
            return letterbox_batch_cuda(im, self.imgsz, auto=same_shapes and self.model.pt, stride=self.model.stride,
                                        device=self.device, staging=stg)
        arr = np.stack(self.pre_transform(im))
        arr = np.ascontiguousarray(arr[..., ::-1].transpose((0, 3, 1, 2)))
        t = torch.from_numpy(arr).to(self.device, non_blocking=True).float()
        t /= 255
        return t

    def inference(self, im, *args, **kwargs):
        return self.model(im)

    #: host batches are ingested in this many chunks (H2D of chunk k+1 overlaps compute of chunk k)
    pipeline_chunks = 4
    #: never split below this many images per chunk (tiny plans waste the 148 SMs) ...
    pipeline_min_chunk = 8
    #: ... nor below this many upload bytes per chunk: chunking exists to start computing before the whole batch has
    #: crossed PCIe; when a chunk's upload (~18 us per MB) is short next to its kernels (fp16 / uint8 batches), the
    #: smaller plans only cost GPU efficiency, and successive predict() calls already overlap upload and compute
    pipeline_min_chunk_bytes = 48 << 20
    #: chunks in flight on the GPU (1 or 2): consecutive chunks alternate between two streams / plan slots, so
    #: the launch-latency-bound small layers of one chunk overlap the bandwidth-bound layers of the other
    in_flight = 2
    #: staging states (device staging batches + output buffers) kept per backend, LRU over (shape, max_det, dtype)
    pipeline_states = 3

    def _chunking(self, im):
        """Number of ingest chunks for a host tensor batch: n > 1 = chunk-pipelined, -1 = asynchronous pipeline with the
        whole batch as one chunk, 1 = plain synchronous-order path (device tensors, lists of images)."""
        if not isinstance(im, torch.Tensor) or im.is_cuda or im.dim() != 4 \
                or im.dtype not in (torch.float32, torch.float16, torch.uint8) or not im.is_contiguous():
            return 1
        b = im.shape[0]
        nbytes = im.numel() * im.element_size()
        for n in range(int(self.pipeline_chunks), 1, -1):
            if b % n == 0 and b // n >= self.pipeline_min_chunk and nbytes // n >= self.pipeline_min_chunk_bytes:
                return n
        return -1          # asynchronous pipeline, whole batch as one chunk

    def _pipelined(self, im_host, n_chunks):
        """preprocess + inference + NMS of a host fp32 batch, chunk-pipelined.  Returns (device batch, dets,
        counts); the detections of chunk k land in rows [k*cb, (k+1)*cb) of the batch-level outputs.  With `embed`
        set: (device batch, (B, D) embeddings, None), chunk k's feature vectors in rows [k*cb, (k+1)*cb)."""
        a = self.args
        dev = self.device
        B = im_host.shape[0]
        cb = B // n_chunks
        model = self.model.model
        emb = embed_indices(a.embed, len(model.model)) if a.embed else None
        # fp16 / uint8 batches stay narrow all the way into the model's ingest kernel (2x / 4x fewer PCIe and HBM bytes);
        # uint8 means image bytes and is scaled by 1/255 there (reference predictor.py:83-84: `.float()`, `/= 255`)
        key = (tuple(im_host.shape), a.max_det, str(im_host.dtype), emb)
        # the staging state lives on the backend: YOLOLite.predict builds a fresh predictor per call, but the pinned
        # upload pipeline (two device staging batches, streams, events) must survive across calls.  The side streams
        # are shared by every state; buffers are kept per (shape, max_det, dtype) in a small LRU so that alternating
        # batch shapes (a full batch followed by the last partial one) neither reallocate nor free memory that
        # launches still in flight on the side streams are using.
        pipe = self.model.__dict__.get("_yl_pipe")
        if pipe is None:
            pipe = self.model.__dict__["_yl_pipe"] = {
                "copy": torch.cuda.Stream(device=dev), "lanes": [torch.cuda.Stream(device=dev) for _ in range(2)],
                "post": torch.cuda.Stream(device=dev), "states": {}, "snap": None}
        states = pipe["states"]
        st = states.get(key)
        if st is not None:
            states[key] = states.pop(key)                # most recently used last
        else:
            if len(states) >= self.pipeline_states:
                # the evicted buffers were only ever used on the side streams: drain those before the allocator may
                # hand the blocks to somebody else (the caller's stream never touched them)
                for side in (pipe["copy"], *pipe["lanes"], pipe["post"]):
                    side.synchronize()
                states.pop(next(iter(states)))
            st = {"key": key, "bufs": [torch.empty(im_host.shape, dtype=im_host.dtype, device=dev) for _ in range(2)],
                  "free": [None, None], "turn": 0,
                  "events": [torch.cuda.Event() for _ in range(n_chunks)]}
            if emb is None:
                st["dets"] = torch.empty((B, a.max_det, 6), dtype=torch.float32, device=dev)
                st["counts"] = torch.empty((B,), dtype=torch.int32, device=dev)
            else:
                D = sum(model._out_channels(list(model.model), k, {}) for k in emb)
                st["emb"] = torch.empty((B, D), dtype=torch.float32, device=dev)
            states[key] = st
        st["copy"], st["lanes"], st["post"] = pipe["copy"], pipe["lanes"], pipe["post"]
        self.model.__dict__["_yl_pipe_state"] = st       # the state the most recent call used
        j = st["turn"]
        st["turn"] ^= 1
        buf = st["bufs"][j]
        # Nothing of this pipeline runs on the caller's stream: upload on the copy stream, chunks alternate between
        # two lane streams, box rescale + result snapshot on the post stream.  The caller's stream is made to wait
        # for a batch only when somebody looks at its Results (BatchDetections.ready), so reading batch k-1 never
        # queues behind the upload / kernels of batch k.
        # The upload may start as soon as the kernels of the call that last read THIS staging batch are done (two
        # calls ago): it overlaps the previous call's kernels and the caller's host-side work.
        if st["free"][j] is not None:
            st["copy"].wait_event(st["free"][j])
        # order the pipeline after whatever the caller (or a plain-path predict on a device tensor, which shares the
        # plan slots) has already queued on the current stream; in the steady pattern that stream is idle here
        main = torch.cuda.current_stream(dev)
        for side in (st["copy"], *st["lanes"]):
            side.wait_stream(main)
        with torch.cuda.stream(st["copy"]):
            for k in range(n_chunks):
                buf[k * cb:(k + 1) * cb].copy_(im_host[k * cb:(k + 1) * cb], non_blocking=True)
                st["events"][k].record(st["copy"])
        fly = max(1, min(int(self.in_flight), 2))
        lanes = st["lanes"][:fly]
        lane0 = pipe.get("next_lane", 0)         # chunks (and single-chunk calls) keep alternating lanes across calls
        pipe["next_lane"] = (lane0 + n_chunks) % fly
        for k in range(n_chunks):
            li = (lane0 + k) % fly
            ln = lanes[li]
            with torch.cuda.stream(ln):
                ln.wait_event(st["events"][k])
                if emb is not None:
                    e = model.infer_embed(buf[k * cb:(k + 1) * cb], emb, slot=li)
                    if pipe["snap"] is not None:
                        ln.wait_event(pipe["snap"])
                    st["emb"][k * cb:(k + 1) * cb].copy_(e, non_blocking=True)
                    continue
                # model + NMS of the chunk are one CUDA-graph launch; its plan-owned outputs are gathered into the
                # batch-level buffers (115 KB per 16 images)
                d, c = model.infer_nms(buf[k * cb:(k + 1) * cb], a.conf, a.iou, a.classes, a.agnostic_nms, False,
                                       a.max_det, slot=li, augment=a.augment)
                if pipe["snap"] is not None:
                    ln.wait_event(pipe["snap"])  # the previous call's snapshot of the batch-level dets / counts is taken
                st["dets"][k * cb:(k + 1) * cb].copy_(d, non_blocking=True)
                st["counts"][k * cb:(k + 1) * cb].copy_(c, non_blocking=True)
        post = st["post"]
        for ln in lanes:
            post.wait_stream(ln)
        st["free"][j] = torch.cuda.Event()
        st["free"][j].record(post)
        if emb is not None:
            return buf, st["emb"], None, post
        return buf, st["dets"], st["counts"], post

    def _embed_rows(self, emb, stream=None):
        """Per-image rows of one clone of the (B, D) embeddings, taken on the current stream (after `stream`, the
        pipeline's post stream, when given)."""
        cur = torch.cuda.current_stream(self.device)
        if stream is not None:
            cur.wait_stream(stream)
        rows = torch.unbind(emb.clone(), 0)
        if stream is not None:
            pipe = self.model.__dict__["_yl_pipe"]
            pipe["snap"] = torch.cuda.Event()    # the next pipelined call may overwrite the batch-level buffer after this
            pipe["snap"].record(cur)
        return rows

    def postprocess(self, preds, img, orig_imgs, nms_out=None, stream=None):
        """`stream`: run the rescale + snapshot there (the asynchronous host-tensor pipeline) instead of on the
        caller's current stream."""
        if stream is not None:
            with torch.cuda.stream(stream):
                results = self.postprocess(preds, img, orig_imgs, nms_out=nms_out)
            pipe = self.model.__dict__.get("_yl_pipe")
            if pipe is not None:
                pipe["snap"] = results[0]._lazy[0].ready if results and results[0]._lazy else None
            return results
        a = self.args
        if nms_out is None:
            dets, counts = ops.nms_padded(preds, a.conf, a.iou, a.classes, a.agnostic_nms, False, a.max_det)
        else:
            dets, counts = nms_out
        B = dets.shape[0]
        tensor_src = isinstance(orig_imgs, torch.Tensor)
        shapes = [tuple(orig_imgs.shape[2:])] * B if tensor_src else [im.shape[:2] for im in orig_imgs]
        # per-image (gain, padx, pady, w0, h0) of scale_boxes: cached on the backend per geometry, so a steady stream
        # of same-shaped batches uploads nothing here
        cache = self.model.__dict__.setdefault("_yl_scale_params", {})
        ckey = (tuple(img.shape[2:]), tuple(shapes), str(dets.device))
        pd = cache.get(ckey)
        if pd is None:
            params = np.empty((B, 5), np.float32)
            for i, s0 in enumerate(shapes):
                gain, pad = ops.letterbox_params(tuple(img.shape[2:]), s0)
                params[i] = (gain, pad[0], pad[1], s0[1], s0[0])
            pd = torch.from_numpy(params).to(dets.device)
            if len(cache) > 64:
                cache.clear()
            cache[ckey] = pd
        _C.check(_C.load().yl_scale_boxes(dets.data_ptr(), counts.data_ptr(), B, dets.shape[1], pd.data_ptr(),
                                          _C.stream_ptr()), "yl_scale_boxes")
        # results must not alias the NMS output buffers of the next batch; the per-image counts are read from the
        # device when somebody first looks at a result (ONE host sync per batch), so this call never blocks
        batch = BatchDetections(dets.clone(), counts.clone())
        batch.ready.record()     # on the stream this runs on; consumers wait for it on THEIR stream
        results = []
        for i in range(B):
            orig = _LazyTensorImage(orig_imgs, i) if tensor_src else orig_imgs[i]
            results.append(Results(orig, path=self.batch[0][i], names=self.model.names, lazy=(batch, i)))
        return results

    # ------------------------------------------------------------------ driver
    def __call__(self, source=None, model=None, stream=False, *args, **kwargs):
        self.stream = stream
        gen = self.stream_inference(source, model, *args, **kwargs)
        return gen if stream else list(gen)

    def setup_source(self, source):
        s = self.args.imgsz
        s = [s, s] if isinstance(s, int) else list(s)
        stride = self.model.stride
        self.imgsz = [max(int(np.ceil(v / stride) * stride), stride) for v in s]
        self.dataset = load_inference_source(source=source, batch=self.args.batch, vid_stride=self.args.vid_stride,
                                             buffer=self.args.stream_buffer)
        self.source_type = self.dataset.source_type

    @smart_inference_mode()
    def stream_inference(self, source=None, model=None, *args, **kwargs):
        if not self.model:
            self.setup_model(model)
        if self.args.embed and isinstance(self.model.model, Ensemble):
            raise TypeError(_ENSEMBLE_NO_EMBED)
        with self._lock:
            self.setup_source(source if source is not None else self.args.source)
            self.seen, self.batch = 0, None
            # the reference's Profile synchronises the device on both edges of every stage (ops.py:18-63); that
            # would serialise upload, kernels and host work, so stage times here are HOST (enqueue) times unless
            # `verbose` asks for the per-image log, which needs device-accurate numbers
            profilers = tuple(ops.Profile(device=self.device if self.args.verbose else None) for _ in range(3))
            for self.batch in self.dataset:
                paths, im0s, s = self.batch
                n_chunks = self._chunking(im0s)
                if n_chunks != 1:
                    n_chunks = abs(n_chunks)
                    # host tensor batch: copy / model / NMS run chunk-pipelined (preprocess+inference timed together)
                    with profilers[1]:
                        im, dets, counts, post = self._pipelined(im0s, n_chunks)
                    if self.args.embed:
                        yield from self._embed_rows(dets, post)
                        continue
                    profilers[0].dt = 0.0
                    with profilers[2]:
                        self.results = self.postprocess(None, im, im0s, nms_out=(dets, counts), stream=post)
                else:
                    pipe = self.model.__dict__.get("_yl_pipe")
                    if pipe is not None:   # an asynchronous host-tensor batch may still own the plan slots
                        cur = torch.cuda.current_stream(self.device)
                        for side in (*pipe["lanes"], pipe["post"]):
                            cur.wait_stream(side)
                    with profilers[0]:
                        im = self.preprocess(im0s)
                    a = self.args
                    if a.embed:                 # the reference's stream loop yields the feature vectors, no postprocess
                        with profilers[1]:
                            rows = self._embed_rows(self.model.model.infer_embed(im, a.embed))
                        yield from rows
                        continue
                    with profilers[1]:
                        nms_out = self.model.model.infer_nms(im, a.conf, a.iou, a.classes, a.agnostic_nms, False, a.max_det,
                                                             augment=a.augment)
                    with profilers[2]:
                        self.results = self.postprocess(None, im, im0s, nms_out=nms_out)
                n = len(self.results)
                for i in range(n):
                    self.seen += 1
                    self.results[i].speed = {
                        "preprocess": profilers[0].dt * 1e3 / n,
                        "inference": profilers[1].dt * 1e3 / n,
                        "postprocess": profilers[2].dt * 1e3 / n,
                    }
                    if self.args.verbose:
                        LOGGER.info(f"{s[i]}{im.shape[2]}x{im.shape[3]} {self.results[i].verbose()}"
                                    f"{profilers[1].dt * 1e3 / n:.2f}ms")
                yield from self.results
        if self.args.verbose and self.seen:
            t = tuple(x.t / self.seen * 1e3 for x in profilers)
            LOGGER.info("Speed: %.2fms preprocess, %.2fms inference, %.2fms postprocess per image" % t)

    def setup_model(self, model, verbose=True):
        self.model = AutoBackend(weights=model or self.args.model, device=select_device(self.args.device),
                                 dnn=self.args.dnn, data=self.args.data, fp16=self.args.half, batch=self.args.batch,
                                 fuse=True, verbose=verbose and self.args.verbose)
        self.device = self.model.device
        self.args.half = self.model.fp16
        self.model.eval()
