"""Plain numpy restatement of the COCO bbox evaluation that upstream `DetectionValidator.eval_json` runs: pycocotools
2.0.x `COCO.loadRes` (bbox branch), `COCOeval.computeIoU` (maskApi `bbIou`), `evaluateImg`, `accumulate` and
`summarize` for iouType="bbox", useCats=1; plus upstream's `pred_to_json` and `coco80_to_coco91_class`.

pycocotools cannot be installed where this project runs, so this file is the yardstick the GPU evaluation
(`yololite.utils.cocoeval`, csrc/cocoeval.cu) is compared against, bit for bit.  It follows the pycocotools code
line by line, quirks included: on equal IoU the later gt (in the ignore-sorted order) wins, crowd gts absorb any
number of dts, a gt whose id is 0 leaves `dtMatches = 0` (so accumulate counts its match as a false positive), and
both area bounds are inclusive (an area of exactly 32**2 is small and medium)."""
from __future__ import annotations

import copy
import json
from collections import defaultdict

import numpy as np


def coco80_to_coco91_class():
    """COCO 80-class index -> the 91-id category ids of the COCO annotation files (upstream converter.py)."""
    return [1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 27, 28, 31, 32, 33,
            34, 35, 36, 37, 38, 39, 40, 41, 42, 43, 44, 46, 47, 48, 49, 50, 51, 52, 53, 54, 55, 56, 57, 58, 59, 60, 61,
            62, 63, 64, 65, 67, 70, 72, 73, 74, 75, 76, 77, 78, 79, 80, 81, 82, 84, 85, 86, 87, 88, 89, 90]


def pred_to_json(predn, filename, class_map):
    """Upstream DetectionValidator.pred_to_json on one image's native-space predictions (n, 6) fp32
    [x1, y1, x2, y2, conf, cls]: xyxy -> xywh -> top-left xywh in fp32, then Python's round()."""
    from pathlib import Path

    predn = np.asarray(predn, np.float32).reshape(-1, 6)
    stem = Path(filename).stem
    image_id = int(stem) if stem.isnumeric() else stem
    box = np.empty((len(predn), 4), np.float32)
    box[:, 0] = (predn[:, 0] + predn[:, 2]) / 2
    box[:, 1] = (predn[:, 1] + predn[:, 3]) / 2
    box[:, 2] = predn[:, 2] - predn[:, 0]
    box[:, 3] = predn[:, 3] - predn[:, 1]
    box[:, :2] -= box[:, 2:] / 2
    return [{"image_id": image_id, "category_id": class_map[int(p[5])], "bbox": [round(x, 3) for x in b],
             "score": round(p[4], 5)} for p, b in zip(predn.tolist(), box.tolist())]


class Params:
    """COCOeval Params for iouType="bbox"."""

    def __init__(self):
        self.imgIds, self.catIds = [], []
        self.iouThrs = np.linspace(.5, 0.95, int(np.round((0.95 - .5) / .05)) + 1, endpoint=True)
        self.recThrs = np.linspace(.0, 1.00, int(np.round((1.00 - .0) / .01)) + 1, endpoint=True)
        self.maxDets = [1, 10, 100]
        self.areaRng = [[0 ** 2, 1e5 ** 2], [0 ** 2, 32 ** 2], [32 ** 2, 96 ** 2], [96 ** 2, 1e5 ** 2]]
        self.areaRngLbl = ["all", "small", "medium", "large"]
        self.useCats = 1


class COCO:
    """The index pycocotools' COCO builds (anns by id, imgToAnns in file order)."""

    def __init__(self, dataset=None):
        if isinstance(dataset, str):
            with open(dataset) as f:
                dataset = json.load(f)
        self.dataset = dataset or {}
        self.anns, self.imgs, self.cats = {}, {}, {}
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

    def getAnnIds(self, imgIds, catIds):
        lists = [self.imgToAnns[i] for i in imgIds if i in self.imgToAnns]
        anns = [a for lst in lists for a in lst]
        anns = anns if len(catIds) == 0 else [a for a in anns if a["category_id"] in catIds]
        return [a["id"] for a in anns]

    def loadAnns(self, ids):
        return [self.anns[i] for i in ids]

    def loadRes(self, resFile):
        res = COCO()
        res.dataset["images"] = [img for img in self.dataset["images"]]
        if isinstance(resFile, str):
            with open(resFile) as f:
                anns = json.load(f)
        else:
            anns = resFile
        assert isinstance(anns, list), "results in not an array of objects"
        annsImgIds = [ann["image_id"] for ann in anns]
        assert set(annsImgIds) == (set(annsImgIds) & set(self.getImgIds())), "Results do not correspond to current coco set"
        res.dataset["categories"] = copy.deepcopy(self.dataset["categories"])
        for id, ann in enumerate(anns):
            bb = ann["bbox"]
            x1, x2, y1, y2 = [bb[0], bb[0] + bb[2], bb[1], bb[1] + bb[3]]
            if "segmentation" not in ann:
                ann["segmentation"] = [[x1, y1, x1, y2, x2, y2, x2, y1]]
            ann["area"] = bb[2] * bb[3]
            ann["id"] = id + 1
            ann["iscrowd"] = 0
        res.dataset["annotations"] = anns
        return COCO(res.dataset)


def bb_iou(dt, gt, iscrowd):
    """maskApi bbIou: o[d, g], fp64, each element in its operation order (elementwise numpy, no reassociation)."""
    d = np.asarray(dt, np.float64).reshape(-1, 4)[:, None, :]
    g = np.asarray(gt, np.float64).reshape(-1, 4)[None, :, :]
    crowd = np.asarray(iscrowd, bool).reshape(1, -1)
    w = np.minimum(d[..., 2] + d[..., 0], g[..., 2] + g[..., 0]) - np.maximum(d[..., 0], g[..., 0])
    h = np.minimum(d[..., 3] + d[..., 1], g[..., 3] + g[..., 1]) - np.maximum(d[..., 1], g[..., 1])
    i = w * h
    da, ga = d[..., 2] * d[..., 3], g[..., 2] * g[..., 3]
    u = np.where(crowd, da, da + ga - i)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where((w > 0) & (h > 0), i / u, 0.0)


class COCOeval:
    def __init__(self, cocoGt, cocoDt):
        self.cocoGt, self.cocoDt = cocoGt, cocoDt
        self.params = Params()
        self.params.imgIds = sorted(cocoGt.getImgIds())
        self.params.catIds = sorted(cocoGt.getCatIds())
        self.eval, self.stats = {}, []

    def _prepare(self):
        p = self.params
        gts = self.cocoGt.loadAnns(self.cocoGt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        dts = self.cocoDt.loadAnns(self.cocoDt.getAnnIds(imgIds=p.imgIds, catIds=p.catIds))
        for gt in gts:
            gt["ignore"] = gt["ignore"] if "ignore" in gt else 0
            gt["ignore"] = "iscrowd" in gt and gt["iscrowd"]
        self._gts, self._dts = defaultdict(list), defaultdict(list)
        for gt in gts:
            self._gts[gt["image_id"], gt["category_id"]].append(gt)
        for dt in dts:
            self._dts[dt["image_id"], dt["category_id"]].append(dt)

    def evaluate(self):
        p = self.params
        p.imgIds = list(np.unique(p.imgIds))
        p.catIds = list(np.unique(p.catIds))
        p.maxDets = sorted(p.maxDets)
        self._prepare()
        self.ious = {(i, c): self.computeIoU(i, c) for i in p.imgIds for c in p.catIds}
        maxDet = p.maxDets[-1]
        self.evalImgs = [self.evaluateImg(i, c, a, maxDet) for c in p.catIds for a in p.areaRng for i in p.imgIds]

    def computeIoU(self, imgId, catId):
        p = self.params
        gt, dt = self._gts[imgId, catId], self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return []
        inds = np.argsort([-d["score"] for d in dt], kind="mergesort")
        dt = [dt[i] for i in inds]
        if len(dt) > p.maxDets[-1]:
            dt = dt[0:p.maxDets[-1]]
        if len(gt) == 0 or len(dt) == 0:
            return []
        return bb_iou([d["bbox"] for d in dt], [g["bbox"] for g in gt], [int(o["iscrowd"]) for o in gt])

    def evaluateImg(self, imgId, catId, aRng, maxDet):
        gt, dt = self._gts[imgId, catId], self._dts[imgId, catId]
        if len(gt) == 0 and len(dt) == 0:
            return None
        for g in gt:
            g["_ignore"] = 1 if (g["ignore"] or (g["area"] < aRng[0] or g["area"] > aRng[1])) else 0
        gtind = np.argsort([g["_ignore"] for g in gt], kind="mergesort")
        gt = [gt[i] for i in gtind]
        dtind = np.argsort([-d["score"] for d in dt], kind="mergesort")
        dt = [dt[i] for i in dtind[0:maxDet]]
        iscrowd = [int(o["iscrowd"]) for o in gt]
        ious = self.ious[imgId, catId][:, gtind] if len(self.ious[imgId, catId]) > 0 else self.ious[imgId, catId]
        T, G, D = len(self.params.iouThrs), len(gt), len(dt)
        gtm, dtm = np.zeros((T, G)), np.zeros((T, D))
        gtIg = np.array([g["_ignore"] for g in gt])
        dtIg = np.zeros((T, D))
        if not len(ious) == 0:
            for tind, t in enumerate(self.params.iouThrs):
                for dind, d in enumerate(dt):
                    iou = min([t, 1 - 1e-10])
                    m = -1
                    for gind, g in enumerate(gt):
                        if gtm[tind, gind] > 0 and not iscrowd[gind]:
                            continue
                        if m > -1 and gtIg[m] == 0 and gtIg[gind] == 1:
                            break
                        if ious[dind, gind] < iou:
                            continue
                        iou = ious[dind, gind]
                        m = gind
                    if m == -1:
                        continue
                    dtIg[tind, dind] = gtIg[m]
                    dtm[tind, dind] = gt[m]["id"]
                    gtm[tind, m] = d["id"]
        a = np.array([d["area"] < aRng[0] or d["area"] > aRng[1] for d in dt]).reshape((1, len(dt)))
        dtIg = np.logical_or(dtIg, np.logical_and(dtm == 0, np.repeat(a, T, 0)))
        return {"image_id": imgId, "category_id": catId, "aRng": aRng, "maxDet": maxDet,
                "dtIds": [d["id"] for d in dt], "gtIds": [g["id"] for g in gt], "dtMatches": dtm, "gtMatches": gtm,
                "dtScores": [d["score"] for d in dt], "gtIgnore": gtIg, "dtIgnore": dtIg}

    def accumulate(self):
        p = self.params
        T, R, K, A, M = len(p.iouThrs), len(p.recThrs), len(p.catIds), len(p.areaRng), len(p.maxDets)
        precision = -np.ones((T, R, K, A, M))
        recall = -np.ones((T, K, A, M))
        scores = -np.ones((T, R, K, A, M))
        I0, A0 = len(p.imgIds), len(p.areaRng)
        for k in range(K):
            Nk = k * A0 * I0
            for a in range(A):
                Na = a * I0
                for m, maxDet in enumerate(p.maxDets):
                    E = [self.evalImgs[Nk + Na + i] for i in range(I0)]
                    E = [e for e in E if e is not None]
                    if len(E) == 0:
                        continue
                    dtScores = np.concatenate([e["dtScores"][0:maxDet] for e in E])
                    inds = np.argsort(-dtScores, kind="mergesort")
                    dtScoresSorted = dtScores[inds]
                    dtm = np.concatenate([e["dtMatches"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    dtIg = np.concatenate([e["dtIgnore"][:, 0:maxDet] for e in E], axis=1)[:, inds]
                    gtIg = np.concatenate([e["gtIgnore"] for e in E])
                    npig = np.count_nonzero(gtIg == 0)
                    if npig == 0:
                        continue
                    tps = np.logical_and(dtm, np.logical_not(dtIg))
                    fps = np.logical_and(np.logical_not(dtm), np.logical_not(dtIg))
                    tp_sum = np.cumsum(tps, axis=1).astype(dtype=float)
                    fp_sum = np.cumsum(fps, axis=1).astype(dtype=float)
                    for t, (tp, fp) in enumerate(zip(tp_sum, fp_sum)):
                        tp, fp = np.array(tp), np.array(fp)
                        nd = len(tp)
                        rc = tp / npig
                        pr = tp / (fp + tp + np.spacing(1))
                        q, ss = np.zeros((R,)), np.zeros((R,))
                        recall[t, k, a, m] = rc[-1] if nd else 0
                        pr, q = pr.tolist(), q.tolist()
                        for i in range(nd - 1, 0, -1):
                            if pr[i] > pr[i - 1]:
                                pr[i - 1] = pr[i]
                        inds = np.searchsorted(rc, p.recThrs, side="left")
                        try:
                            for ri, pi in enumerate(inds):
                                q[ri] = pr[pi]
                                ss[ri] = dtScoresSorted[pi]
                        except IndexError:
                            pass
                        precision[t, :, k, a, m] = np.array(q)
                        scores[t, :, k, a, m] = np.array(ss)
        self.eval = {"params": p, "counts": [T, R, K, A, M], "precision": precision, "recall": recall, "scores": scores}

    def summarize(self):
        self.stats = summarize(self.eval, self.params)


def summarize(ev, p, log=None):
    """COCOeval.summarize / _summarizeDets: the 12 stats, with the lines it prints passed to `log`."""

    def _summarize(ap=1, iouThr=None, areaRng="all", maxDets=100):
        iStr = " {:<18} {} @[ IoU={:<9} | area={:>6s} | maxDets={:>3d} ] = {:0.3f}"
        titleStr = "Average Precision" if ap == 1 else "Average Recall"
        typeStr = "(AP)" if ap == 1 else "(AR)"
        iouStr = "{:0.2f}:{:0.2f}".format(p.iouThrs[0], p.iouThrs[-1]) if iouThr is None else "{:0.2f}".format(iouThr)
        aind = [i for i, aRng in enumerate(p.areaRngLbl) if aRng == areaRng]
        mind = [i for i, mDet in enumerate(p.maxDets) if mDet == maxDets]
        if ap == 1:
            s = ev["precision"]
            if iouThr is not None:
                t = np.where(iouThr == p.iouThrs)[0]
                s = s[t]
            s = s[:, :, :, aind, mind]
        else:
            s = ev["recall"]
            if iouThr is not None:
                t = np.where(iouThr == p.iouThrs)[0]
                s = s[t]
            s = s[:, :, aind, mind]
        mean_s = -1 if len(s[s > -1]) == 0 else np.mean(s[s > -1])
        if log is not None:
            log(iStr.format(titleStr, typeStr, iouStr, areaRng, maxDets, mean_s))
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
    return stats


def evaluate(gt_dataset, results, img_ids=None):
    """COCO(gt) -> loadRes(results) -> COCOeval(bbox).evaluate/accumulate/summarize; returns the COCOeval."""
    gt = COCO(copy.deepcopy(gt_dataset))
    dt = gt.loadRes(copy.deepcopy(results))
    ev = COCOeval(gt, dt)
    if img_ids is not None:
        ev.params.imgIds = list(img_ids)
    ev.evaluate()
    ev.accumulate()
    ev.summarize()
    return ev


def synthetic_coco(seed, n_images=40, n_cats=6, gts_per_image=8, dts_per_image=60, fixed_dts=False, crowd_frac=0.05,
                   id_zero=False):
    """Seeded COCO-style (annotation dict, results list).  Gts: 0 .. 2 * gts_per_image per image, sides spanning all
    three area classes, some with w * h of exactly 32**2 or 96**2, json areas that differ from w * h, `crowd_frac` crowd
    gts; ids start at 0 when `id_zero`.  Dts (`dts_per_image` each with `fixed_dts`, else 0 .. 2 * dts_per_image): 70 %
    jittered copies of a gt (some exact, so IoUs tie; 20 % with a wrong category), the rest clutter; scores rounded to
    5 digits from a small set, so score ties within and across images are common.  Image ids are shuffled, sparse."""
    rng = np.random.default_rng(seed)
    img_ids = [int(x) for x in rng.choice(np.arange(1, 10 * n_images + 1), n_images, replace=False)]
    cat_ids = np.sort(rng.choice(np.arange(1, 3 * n_cats + 1), n_cats, replace=False))
    side = np.array([4.0, 12.0, 31.5, 32.0, 50.0, 96.0, 120.0, 260.0])
    levels = np.linspace(0.05, 0.95, 19)
    anns, res = [], []
    aid = 0 if id_zero else 1
    for im in img_ids:
        ng = int(rng.integers(0, 2 * gts_per_image + 1))
        wh = rng.choice(side, (ng, 2)) * rng.uniform(0.5, 1.5, (ng, 2))
        exact = rng.random(ng) < 0.1
        wh[exact] = rng.choice([32.0, 96.0], (int(exact.sum()), 1))
        xy = rng.uniform(0, 1, (ng, 2)) * np.maximum(np.array([640.0, 480.0]) - wh, 0)
        area = wh[:, 0] * wh[:, 1] * np.where(rng.random(ng) < 0.7, 1.0, rng.uniform(0.3, 1.0, ng))
        gcat = rng.choice(cat_ids, ng)
        crowd = rng.random(ng) < crowd_frac
        for j in range(ng):
            anns.append({"id": aid, "image_id": im, "category_id": int(gcat[j]),
                         "bbox": [float(xy[j, 0]), float(xy[j, 1]), float(wh[j, 0]), float(wh[j, 1])],
                         "area": float(area[j]), "iscrowd": int(crowd[j])})
            aid += 1
        nd = dts_per_image if fixed_dts else int(rng.integers(0, 2 * dts_per_image + 1))
        near = (rng.random(nd) < 0.7) & (ng > 0)
        src = rng.integers(0, max(ng, 1), nd)
        bb = np.empty((nd, 4))
        cat = rng.choice(cat_ids, nd)
        if ng:
            gb = np.concatenate([xy, wh], 1)[src]
            jit = rng.normal(0, 0.08, (nd, 4)) * gb[:, [2, 3, 2, 3]]
            jit[rng.random(nd) < 0.05] = 0.0                                  # exact copies: equal IoUs
            nb = gb + jit
            nb[:, 2:] = np.maximum(nb[:, 2:], 1.0)
            keep_cat = rng.random(nd) >= 0.2
            cat = np.where(near & keep_cat, gcat[src], cat)
            bb[near] = nb[near]
        far = ~near
        bb[far] = np.concatenate([rng.uniform(0, 1, (int(far.sum()), 2)) * [600, 440],
                                  rng.choice(side, (int(far.sum()), 2))], 1)
        bb = np.round(bb, 3)
        score = np.round(rng.choice(levels, nd) + (rng.random(nd) < 0.5) * rng.uniform(0, 0.04, nd), 5)
        res += [{"image_id": im, "category_id": int(c), "bbox": b, "score": float(sc)}
                for c, b, sc in zip(cat.tolist(), bb.tolist(), score.tolist())]
    gt = {"images": [{"id": i, "width": 640, "height": 480, "file_name": f"{i:012d}.jpg"} for i in img_ids],
          "annotations": anns, "categories": [{"id": int(c), "name": f"c{c}", "supercategory": "x"} for c in cat_ids]}
    return gt, res
