"""COCO bbox evaluation with the names upstream `DetectionValidator.eval_json` calls (pycocotools 2.0.x `COCO`,
`COCO.loadRes`, `COCOeval(gt, dt, "bbox")`, `.evaluate()`, `.accumulate()`, `.summarize()`), evaluated on the GPU.

`evaluate()` and `accumulate()` are the pycocotools Python loops over images x categories x area ranges x IoU
thresholds; here they are two launches of csrc/cocoeval.cu (`yl_cocoeval_evaluate`, `yl_cocoeval_accumulate`) with one
stable device sort between them.  `summarize()` is pycocotools' own numpy code on the host.  `eval["precision"]`,
`eval["recall"]`, `eval["scores"]` and `stats` are bit-identical to pycocotools' (pinned against the numpy restatement in
oracle/cocoeval_ref.py), upstream quirks included: equal IoU goes to the later gt, crowd gts match any number of dts, a
gt with id 0 leaves its dt counted as a false positive, and both area-range bounds are inclusive.

Only iouType="bbox" with useCats=1 is implemented; anything else raises NotImplementedError.  The per-image result
dicts (`evalImgs`) are not materialised: the per-(image, category) results stay on the device between the two launches.
"""
from __future__ import annotations

import copy
import datetime
import json
import time
from collections import defaultdict

import numpy as np
import torch

from .. import _C
from . import LOGGER


class COCO:
    """pycocotools COCO: the annotation index (`anns` by id, `imgToAnns` in file order) from a json path or a dict."""

    def __init__(self, annotation_file=None):
        self.dataset, self.anns, self.cats, self.imgs = {}, {}, {}, {}
        self.imgToAnns = defaultdict(list)
        if annotation_file is not None:
            if isinstance(annotation_file, dict):
                dataset = annotation_file
            else:
                with open(annotation_file) as f:
                    dataset = json.load(f)
            assert isinstance(dataset, dict), f"annotation file format {type(dataset)} not supported"
            self.dataset = dataset
            self.createIndex()

    def createIndex(self):
        self.anns, self.cats, self.imgs = {}, {}, {}
        self.imgToAnns = defaultdict(list)
        for ann in self.dataset.get("annotations", []):
            self.imgToAnns[ann["image_id"]].append(ann)
            self.anns[ann["id"]] = ann
        for img in self.dataset.get("images", []):
            self.imgs[img["id"]] = img
        for cat in self.dataset.get("categories", []):
            self.cats[cat["id"]] = cat

    def getImgIds(self):
        return list(self.imgs.keys())

    def getCatIds(self):
        return [c["id"] for c in self.dataset.get("categories", [])]

    def getAnnIds(self, imgIds=(), catIds=()):
        """Annotation ids of `imgIds` (in that order, file order within an image) whose category is in `catIds`."""
        if len(imgIds):
            anns = [a for i in imgIds if i in self.imgToAnns for a in self.imgToAnns[i]]
        else:
            anns = self.dataset.get("annotations", [])
        if len(catIds):
            cats = set(catIds)
            anns = [a for a in anns if a["category_id"] in cats]
        return [a["id"] for a in anns]

    def loadAnns(self, ids):
        return [self.anns[i] for i in ids]

    def loadRes(self, resFile):
        """Detection results (json path or list of dicts) as a COCO object: the pycocotools bbox branch sets
        `area = w * h`, `id = index + 1` and `iscrowd = 0` on every result."""
        res = COCO()
        res.dataset["images"] = [img for img in self.dataset["images"]]
        LOGGER.info("Loading and preparing results...")
        tic = time.time()
        if isinstance(resFile, str) or hasattr(resFile, "__fspath__"):
            with open(resFile) as f:
                anns = json.load(f)
        else:
            anns = resFile
        assert isinstance(anns, list), "results in not an array of objects"
        annsImgIds = [ann["image_id"] for ann in anns]
        assert set(annsImgIds) == (set(annsImgIds) & set(self.getImgIds())), \
            "Results do not correspond to current coco set"
        if anns and not ("bbox" in anns[0] and anns[0]["bbox"] != []):
            raise NotImplementedError("only bbox results are supported (no captions, segmentations or keypoints)")
        res.dataset["categories"] = copy.deepcopy(self.dataset["categories"])
        for id, ann in enumerate(anns):
            bb = ann["bbox"]
            x1, x2, y1, y2 = [bb[0], bb[0] + bb[2], bb[1], bb[1] + bb[3]]
            if "segmentation" not in ann:
                ann["segmentation"] = [[x1, y1, x1, y2, x2, y2, x2, y1]]
            ann["area"] = bb[2] * bb[3]
            ann["id"] = id + 1
            ann["iscrowd"] = 0
        LOGGER.info(f"DONE (t={time.time() - tic:0.2f}s)")
        res.dataset["annotations"] = anns
        res.createIndex()
        return res


class Params:
    """COCOeval Params for iouType="bbox" (setDetParams)."""

    def __init__(self, iouType="bbox"):
        self.imgIds, self.catIds = [], []
        self.iouThrs = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
        self.recThrs = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
        self.maxDets = [1, 10, 100]
        self.areaRng = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
        self.areaRngLbl = ["all", "small", "medium", "large"]
        self.useCats = 1
        self.iouType = iouType


def _flat(anns, img_rank, cat_index, n_images, max_det=None):
    """(pair key = category index * n_images + image rank) of every annotation of the evaluated images and
    categories, grouped by a stable sort on the key.  Gts (max_det None) keep their given order inside a group.  Dts
    are ordered inside a group by descending score, ties in their given order (computeIoU / evaluateImg's
    np.argsort(-score, kind="mergesort")), and cut to the first `max_det`."""
    ri = np.fromiter((img_rank.get(a["image_id"], -1) for a in anns), np.int64, len(anns))
    ci = np.fromiter((cat_index.get(a["category_id"], -1) for a in anns), np.int64, len(anns))
    keep = np.nonzero((ri >= 0) & (ci >= 0))[0]
    key = ci[keep] * n_images + ri[keep]
    if max_det is None:
        o = np.argsort(key, kind="stable")
    else:
        score = np.fromiter((anns[i]["score"] for i in keep), np.float64, len(keep))
        _finite(score, "result scores")
        o = np.lexsort((-score, key))                      # stable: equal (key, score) keep their given order
        k = key[o]
        o = o[np.arange(len(o)) - np.searchsorted(k, k, "left") < max_det]
    return key[o], [anns[i] for i in keep[o]]


def _finite(a, what):
    """pycocotools compares NaN IoUs / scores in an order-dependent way that is not reproduced: reject them."""
    if not np.isfinite(a).all():
        raise ValueError(f"COCOeval: {what} must be finite (found NaN or inf)")
    return a


class COCOeval:
    """pycocotools COCOeval for iouType="bbox": `evaluate()` and `accumulate()` run on the current CUDA device,
    `summarize()` fills the 12 `stats`.  `evalImgs` is not materialised (see the module docstring)."""

    def __init__(self, cocoGt=None, cocoDt=None, iouType="segm"):
        if iouType != "bbox":
            raise NotImplementedError(f"COCOeval iouType={iouType!r}: only 'bbox' is implemented")
        self.cocoGt, self.cocoDt = cocoGt, cocoDt
        self.params = Params(iouType=iouType)
        self.eval, self.stats = {}, []
        self._dev = None
        if cocoGt is not None:
            self.params.imgIds = sorted(cocoGt.getImgIds())
            self.params.catIds = sorted(cocoGt.getCatIds())

    def evaluate(self):
        """computeIoU + evaluateImg of every (image, category) pair, in one launch."""
        tic = time.time()
        LOGGER.info("Running per image evaluation...")
        p = self.params
        if not p.useCats:
            raise NotImplementedError("COCOeval with useCats=0 is not implemented")
        LOGGER.info(f"Evaluate annotation type *{p.iouType}*")
        p.imgIds = list(np.unique(p.imgIds))
        p.catIds = list(np.unique(p.catIds))
        p.maxDets = sorted(p.maxDets)
        I, K, A, T = len(p.imgIds), len(p.catIds), len(p.areaRng), len(p.iouThrs)
        gts = self.cocoGt.loadAnns(self.cocoGt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        dts = self.cocoDt.loadAnns(self.cocoDt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        img_rank = {int(i) if isinstance(i, np.integer) else i: r for r, i in enumerate(p.imgIds)}
        cat_index = {int(c) if isinstance(c, np.integer) else c: k for k, c in enumerate(p.catIds)}
        gkey, gts = _flat(gts, img_rank, cat_index, I)
        dkey, dts = _flat(dts, img_rank, cat_index, I, p.maxDets[-1])
        pairs = np.union1d(gkey, dkey)
        n_gt = np.searchsorted(gkey, pairs, "right") - np.searchsorted(gkey, pairs, "left")
        n_slot = np.searchsorted(dkey, pairs, "right") - np.searchsorted(dkey, pairs, "left")
        csr = lambda c: np.concatenate([[0], np.cumsum(c)]).astype(np.int32)   # noqa: E731
        pair_cat = (pairs // max(I, 1)).astype(np.int32)
        cat_slots = np.bincount(pair_cat, weights=n_slot, minlength=K).astype(np.int64)

        f64 = np.float64
        gt_bbox = _finite(np.array([a["bbox"] for a in gts], f64).reshape(-1, 4), "gt boxes")
        gt_area = _finite(np.array([a["area"] for a in gts], f64), "gt areas")
        dt_bbox = _finite(np.array([a["bbox"] for a in dts], f64).reshape(-1, 4), "result boxes")

        self._dev = dev = torch.device("cuda", torch.cuda.current_device())
        _C.init(dev)
        put = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a, dt)).to(dev, non_blocking=True)   # noqa: E731
        g = {
            "pair_cat": put(pair_cat, np.int32), "gt_off": put(csr(n_gt), np.int32), "slot_off": put(csr(n_slot), np.int32),
            "gt_bbox": put(gt_bbox, f64), "gt_area": put(gt_area, f64),
            "gt_iscrowd": put([1 if a.get("iscrowd", 0) else 0 for a in gts], np.uint8),
            "gt_id": put([a["id"] for a in gts], np.int64),
            "dt_bbox": put(dt_bbox, f64),
            "dt_score": put([a["score"] for a in dts], f64),
            "dt_area": put([a["area"] for a in dts], f64),
            "dt_id": put([a["id"] for a in dts], np.int64),
            "iou_thrs": put(p.iouThrs, f64), "rec_thrs": put(p.recThrs, f64),
            "area_rng": put(np.array(p.areaRng, f64).reshape(-1, 2), f64), "max_dets": put(p.maxDets, np.int32),
            "cat_slot_off": put(csr(cat_slots), np.int32),
            "slot_cat": put(np.repeat(pair_cat, n_slot), np.int64),
        }
        S = int(n_slot.sum())
        g["key"] = torch.empty(S, dtype=torch.int64, device=dev)
        g["rank"] = torch.empty(S, dtype=torch.int32, device=dev)
        g["flags"] = torch.empty(S * A * T, dtype=torch.uint8, device=dev)
        g["npig"] = torch.empty(K * A, dtype=torch.int32, device=dev)
        ptr = lambda t: t.data_ptr() if t.numel() else None   # noqa: E731
        self._params = _C.CocoevalParams(ptr(g["iou_thrs"]), ptr(g["rec_thrs"]), ptr(g["area_rng"]), ptr(g["max_dets"]),
                                         T, len(p.recThrs), A, len(p.maxDets))
        self._slots = _C.CocoevalSlots(*(ptr(g[k]) for k in ("key", "rank", "flags", "npig")))
        cset = _C.CocoevalSet(len(pairs), K, S, int(n_gt.max(initial=0)), int(n_slot.max(initial=0)),
                              *(ptr(g[k]) for k in ("pair_cat", "gt_off", "gt_bbox", "gt_area", "gt_iscrowd", "gt_id",
                                                    "slot_off", "dt_bbox", "dt_score", "dt_area", "dt_id")))
        _C.check(_C.load().yl_cocoeval_evaluate(cset, self._params, self._slots, _C.stream_ptr()), "yl_cocoeval_evaluate")
        self._g, self._set = g, cset
        LOGGER.info(f"DONE (t={time.time() - tic:0.2f}s).")

    def accumulate(self, p=None):
        """Precision / recall / scores over every (category, area range, maxDet, IoU threshold), in one launch; the
        category's dts are put in score order (ties: image order, then rank in the image) by two stable device sorts
        and gathered once into that order."""
        LOGGER.info("Accumulating evaluation results...")
        tic = time.time()
        if not hasattr(self, "_g"):
            LOGGER.info("Please run evaluate() first")
            return
        p = self.params if p is None else p
        g = self._g
        T, R, K, A, M = len(p.iouThrs), len(p.recThrs), len(p.catIds), len(p.areaRng), len(p.maxDets)
        with torch.cuda.device(self._dev):
            by_score = torch.sort(g["key"], stable=True)[1]
            order = by_score[torch.sort(g["slot_cat"][by_score], stable=True)[1]]
            S = order.numel()
            score, rank = g["dt_score"][order], g["rank"][order]
            flags = g["flags"].view(A * T, S)[:, order].contiguous()
            precision = torch.empty((T, R, K, A, M), dtype=torch.float64, device=self._dev)
            recall = torch.empty((T, K, A, M), dtype=torch.float64, device=self._dev)
            scores = torch.empty((T, R, K, A, M), dtype=torch.float64, device=self._dev)
            ptr = lambda t: t.data_ptr() if t.numel() else None   # noqa: E731
            _C.check(_C.load().yl_cocoeval_accumulate(self._params, K, S, ptr(g["cat_slot_off"]), ptr(score), ptr(rank),
                                                      ptr(flags), ptr(g["npig"]), ptr(precision), ptr(recall),
                                                      ptr(scores), _C.stream_ptr()),
                     "yl_cocoeval_accumulate")
            self.eval = {"params": p, "counts": [T, R, K, A, M],
                         "date": datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S"),
                         "precision": precision.cpu().numpy(), "recall": recall.cpu().numpy(),
                         "scores": scores.cpu().numpy()}
        LOGGER.info(f"DONE (t={time.time() - tic:0.2f}s).")

    def summarize(self):
        """pycocotools _summarizeDets: the 12 AP / AR stats, each line logged."""
        if not self.eval:
            raise Exception("Please run accumulate() first")
        p = self.params

        def _summarize(ap=1, iouThr=None, areaRng="all", maxDets=100):
            iStr = " {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}"
            titleStr = "Average Precision" if ap == 1 else "Average Recall"
            typeStr = "(AP)" if ap == 1 else "(AR)"
            iouStr = "{:0.2f}:{:0.2f}".format(p.iouThrs[0], p.iouThrs[-1]) if iouThr is None else "{:0.2f}".format(iouThr)
            aind = [i for i, aRng in enumerate(p.areaRngLbl) if aRng == areaRng]
            mind = [i for i, mDet in enumerate(p.maxDets) if mDet == maxDets]
            if ap == 1:
                s = self.eval["precision"]
                if iouThr is not None:
                    t = np.where(iouThr == p.iouThrs)[0]
                    s = s[t]
                s = s[:, :, :, aind, mind]
            else:
                s = self.eval["recall"]
                if iouThr is not None:
                    t = np.where(iouThr == p.iouThrs)[0]
                    s = s[t]
                s = s[:, :, aind, mind]
            mean_s = -1 if len(s[s > -1]) == 0 else np.mean(s[s > -1])
            LOGGER.info(iStr.format(titleStr, typeStr, iouStr, areaRng, maxDets, mean_s))
            return mean_s

        stats = np.zeros((12,))
        stats[0] = _summarize(1)
        stats[1] = _summarize(1, iouThr=.5, maxDets=p.maxDets[2])
        stats[2] = _summarize(1, iouThr=.75, maxDets=p.maxDets[2])
        stats[3] = _summarize(1, areaRng="small", maxDets=p.maxDets[2])
        stats[4] = _summarize(1, areaRng="medium", maxDets=p.maxDets[2])
        stats[5] = _summarize(1, areaRng="large", maxDets=p.maxDets[2])
        stats[6] = _summarize(0, maxDets=p.maxDets[0])
        stats[7] = _summarize(0, maxDets=p.maxDets[1])
        stats[8] = _summarize(0, maxDets=p.maxDets[2])
        stats[9] = _summarize(0, areaRng="small", maxDets=p.maxDets[2])
        stats[10] = _summarize(0, areaRng="medium", maxDets=p.maxDets[2])
        stats[11] = _summarize(0, areaRng="large", maxDets=p.maxDets[2])
        self.stats = stats
