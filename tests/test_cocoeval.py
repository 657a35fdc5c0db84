"""COCO evaluation (`save_json=True`), CPU half: the numpy restatement of pycocotools' bbox COCOeval
(oracle/cocoeval_ref.py) pinned on hand-worked cases, upstream `pred_to_json` rows byte for byte, the coco80 -> coco91
map, `.txt` split loading, and the input checks that need no device."""
import json
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]

from oracle import cocoeval_ref as R  # noqa: E402

RECTHRS = np.linspace(.0, 1.00, 101)
EPS = np.spacing(1)       # pr = tp / (fp + tp + eps): a perfect prefix has precision 1 / (1 + eps), not 1


def _set(images, anns, cats=(1,)):
    """Annotation dict: anns are (id, image_id, category_id, [x, y, w, h], area or None for w * h, iscrowd)."""
    return {"images": [{"id": i} for i in images], "categories": [{"id": c} for c in cats],
            "annotations": [{"id": a, "image_id": i, "category_id": c, "bbox": list(map(float, b)),
                             "area": float(b[2] * b[3] if ar is None else ar), "iscrowd": cr}
                            for a, i, c, b, ar, cr in anns]}


def _dt(image_id, bbox, score, cat=1):
    return {"image_id": image_id, "category_id": cat, "bbox": list(map(float, bbox)), "score": score}


def _img_eval(ev, img, cat=1, area=0):
    p = ev.params
    return ev.evalImgs[(p.catIds.index(cat) * len(p.areaRng) + area) * len(p.imgIds) + p.imgIds.index(img)]


def test_one_image_known_ap():
    # d1 hits g1 exactly, d2 hits nothing, d3 hits g2 exactly: tp 1 1 2, fp 0 1 1 -> rc .5 .5 1, pr 1 .5 2/3
    gt = _set([1], [(1, 1, 1, [0, 0, 200, 200], None, 0), (2, 1, 1, [300, 300, 150, 150], None, 0)])
    ev = R.evaluate(gt, [_dt(1, [0, 0, 200, 200], .9), _dt(1, [500, 0, 100, 100], .8), _dt(1, [300, 300, 150, 150], .7)])
    want = np.where(RECTHRS <= 0.5, 1 / (1 + EPS), 2 / (3 + EPS))
    for t in range(10):
        np.testing.assert_array_equal(ev.eval["precision"][t, :, 0, 0, 2], want)
        np.testing.assert_array_equal(ev.eval["scores"][t, :, 0, 0, 2], np.where(RECTHRS <= 0.5, .9, .7))
    assert ev.eval["recall"][:, 0, 0, 2].tolist() == [1.0] * 10
    assert ev.stats[0] == pytest.approx((51 + 50 * 2 / 3) / 101, abs=1e-12)   # the mean of the 1010 values above
    assert ev.eval["recall"][0, 0, 0, 0] == 0.5          # maxDets = 1: only d1
    assert ev.stats[6] == 0.5 and ev.stats[8] == 1.0


def test_equal_iou_later_gt_wins():
    gt = _set([1], [(1, 1, 1, [0, 0, 100, 100], None, 0), (2, 1, 1, [0, 0, 100, 100], None, 0)])
    ev = R.evaluate(gt, [_dt(1, [0, 0, 100, 100], .9), _dt(1, [0, 0, 100, 100], .8)])
    e = _img_eval(ev, 1)
    assert e["dtMatches"][:, 0].tolist() == [2] * 10 and e["dtMatches"][:, 1].tolist() == [1] * 10


def test_crowd_gt_absorbs_several_dts():
    gt = _set([1], [(5, 1, 1, [0, 0, 100, 100], None, 1), (6, 1, 1, [300, 300, 50, 50], None, 0)])
    dts = [_dt(1, [10, 10, 20, 20], .9), _dt(1, [40, 40, 20, 20], .8), _dt(1, [60, 10, 30, 30], .7),
           _dt(1, [300, 300, 50, 50], .6)]
    ev = R.evaluate(gt, dts)
    e = _img_eval(ev, 1)
    assert e["dtMatches"][0].tolist() == [5, 5, 5, 6] and e["dtIgnore"][0].tolist() == [1, 1, 1, 0]
    # the crowd-matched dts count neither as tp nor fp: AP of the one real match is 1
    assert ev.stats[0] == pytest.approx(1.0, abs=1e-12)


def test_ignore_break():
    # the dt overlaps the regular gt at IoU .68 and the crowd gt (listed first) at crowd IoU 1
    gt = _set([1], [(7, 1, 1, [0, 0, 10, 6.8], None, 1), (8, 1, 1, [0, 0, 10, 10], None, 0)])
    ev = R.evaluate(gt, [_dt(1, [0, 0, 10, 6.8], .9)])
    e = _img_eval(ev, 1)
    assert e["dtMatches"][:, 0].tolist() == [8] * 4 + [7] * 6
    assert e["dtIgnore"][:, 0].tolist() == [0] * 4 + [1] * 6


def test_area_bounds_inclusive():
    gt = _set([1], [(1, 1, 1, [0, 0, 32, 32], None, 0), (2, 1, 2, [100, 100, 96, 96], None, 0)], cats=(1, 2))
    ev = R.evaluate(gt, [_dt(1, [0, 0, 32, 32], .9, 1), _dt(1, [100, 100, 96, 96], .9, 2)])
    rec = ev.eval["recall"][0, :, :, 2]      # [category, area: all small medium large]
    assert rec.tolist() == [[1, 1, 1, -1], [1, -1, 1, 1]]


def test_max_dets_truncation():
    # 12 gts each hit by one dt; the 11th-ranked dt is the only one that finds gt 11
    gts = [(g + 1, 1, 1, [60 * g, 0, 50, 50], None, 0) for g in range(12)]
    dts = [_dt(1, [60 * g, 0, 50, 50], round(.99 - .01 * g, 2)) for g in range(12)]
    ev = R.evaluate(_set([1], gts), dts)
    assert ev.eval["recall"][0, 0, 0, :].tolist() == [1 / 12, 10 / 12, 1.0]
    e = _img_eval(ev, 1)
    assert e["dtMatches"][0, 10] == 11


def test_gt_with_id_zero_counts_as_false_positive():
    gt = _set([1], [(0, 1, 1, [0, 0, 50, 50], None, 0)])
    ev = R.evaluate(gt, [_dt(1, [0, 0, 50, 50], .9), _dt(1, [0, 0, 50, 50], .8)])
    e = _img_eval(ev, 1)
    assert e["dtMatches"][0].tolist() == [0, 0] and e["gtMatches"][0].tolist() == [1]   # matched, yet dtm = 0
    assert ev.eval["recall"][0, 0, 0, 2] == 0 and (ev.eval["precision"][:, :, 0, 0, 2] == 0).all()
    ev1 = R.evaluate(_set([1], [(1, 1, 1, [0, 0, 50, 50], None, 0)]), [_dt(1, [0, 0, 50, 50], .9)])
    assert ev1.stats[0] == pytest.approx(1.0, abs=1e-12)


def test_category_without_gts_is_excluded():
    gt = _set([1], [(1, 1, 1, [0, 0, 50, 50], None, 0)], cats=(1, 2))
    ev = R.evaluate(gt, [_dt(1, [0, 0, 50, 50], .9, 1), _dt(1, [0, 0, 50, 50], .8, 2)])
    assert (ev.eval["precision"][:, :, 1] == -1).all() and (ev.eval["recall"][:, 1] == -1).all()
    assert (ev.eval["scores"][:, :, 1] == -1).all()
    assert ev.stats[0] == pytest.approx(1.0, abs=1e-12)


def test_recall_thresholds_beyond_max_recall_are_zero():
    gt = _set([1], [(1, 1, 1, [0, 0, 50, 50], None, 0), (2, 1, 1, [100, 100, 50, 50], None, 0)])
    ev = R.evaluate(gt, [_dt(1, [0, 0, 50, 50], .9)])
    q, s = ev.eval["precision"][0, :, 0, 0, 2], ev.eval["scores"][0, :, 0, 0, 2]
    np.testing.assert_array_equal(q, np.where(RECTHRS <= .5, 1 / (1 + EPS), 0.0))
    np.testing.assert_array_equal(s, np.where(RECTHRS <= .5, .9, 0.0))


def test_score_ties_across_images_follow_image_order():
    # equal scores: the false positive of image 3 comes before the true positive of image 7 (image ids ascending,
    # whatever the order of the images in the file or of the results)
    gt = _set([7, 3], [(1, 7, 1, [0, 0, 50, 50], None, 0)])
    ev = R.evaluate(gt, [_dt(7, [0, 0, 50, 50], .5), _dt(3, [0, 0, 50, 50], .5)])
    np.testing.assert_array_equal(ev.eval["precision"][0, :, 0, 0, 2], np.full(101, 1 / (2 + EPS)))


def test_pred_to_json_rows():
    from yololite.engine.validator import DetectionValidator

    predn = np.array([[0.0625, 0.1875, 2.625, 1.1875, 0.5, 3],      # exact binary halves: round half to even
                      [10.0, 20.0, 30.5, 41.0, 0.123455, 0],         # fp32 0.123455 lies above the half
                      [1.0005, 0.0, 2.0, 1.0, 0.000005, 79]], np.float32)   # fp32 1.0005 and 5e-6: just below
    cmap = R.coco80_to_coco91_class()
    want = [{"image_id": 42, "category_id": 4, "bbox": [0.062, 0.188, 2.562, 1.0], "score": 0.5},
            {"image_id": 42, "category_id": 1, "bbox": [10.0, 20.0, 20.5, 21.0], "score": 0.12346},
            {"image_id": 42, "category_id": 90, "bbox": [1.0, 0.0, 1.0, 1.0], "score": 0.0}]
    rows = R.pred_to_json(predn, "/data/images/val2017/000000000042.jpg", cmap)
    assert json.dumps(rows) == json.dumps(want)
    v = DetectionValidator(dataloader=[])
    v.class_map = cmap
    v.pred_to_json(torch.from_numpy(predn), "/data/images/val2017/000000000042.jpg")
    assert json.dumps(v.jdict) == json.dumps(want)
    assert R.pred_to_json(predn[:1], "x/abc.jpg", list(range(1, 81)))[0]["image_id"] == "abc"


def test_coco80_to_coco91_class():
    from yololite.utils import ops

    m = ops.coco80_to_coco91_class()
    assert m == R.coco80_to_coco91_class() and len(m) == 80 and m == sorted(set(m))
    assert set(range(1, 91)) - set(m) == {12, 26, 29, 30, 45, 66, 68, 69, 71, 83}


def _coco_layout(tmp_path, n=3):
    import cv2

    root = tmp_path / "coco"
    (root / "images" / "val2017").mkdir(parents=True)
    (root / "labels" / "val2017").mkdir(parents=True)
    (root / "annotations").mkdir()
    names = [f"{i:012d}" for i in (139, 285, 632)[:n]]
    for k, s in enumerate(names):
        cv2.imwrite(str(root / "images" / "val2017" / f"{s}.jpg"), np.full((48 + 16 * k, 64, 3), 90, np.uint8))
        (root / "labels" / "val2017" / f"{s}.txt").write_text(f"{k} 0.5 0.5 0.25 0.5\n")
    (root / "val2017.txt").write_text("".join(f"./images/val2017/{s}.jpg\n" for s in reversed(names)))
    (root / "annotations" / "instances_val2017.json").write_text(json.dumps(_set([int(s) for s in names], [])))
    yaml = tmp_path / "coco.yaml"
    yaml.write_text(f"path: {root}\nval: val2017.txt\nnames:\n  0: a\n  1: b\n  2: c\n")
    return root, yaml, names


def test_txt_split_loading(tmp_path):
    from yololite.data import build_val_loader
    from yololite.engine.validator import DetectionValidator

    root, yaml, names = _coco_layout(tmp_path)
    loader, cls_names = build_val_loader(yaml, imgsz=64, batch_size=2)
    assert sorted(Path(f).stem for f in loader.im_files) == names and cls_names == {0: "a", 1: "b", 2: "c"}
    for f, lb in zip(loader.im_files, loader.labels):
        k = names.index(Path(f).stem)
        np.testing.assert_array_equal(lb, np.array([[k, .5, .5, .25, .5]], np.float32))
    assert sum(len(b["im_file"]) for b in loader) == 3
    v = DetectionValidator(dataloader=[], args={"data": str(yaml), "save_json": True})
    assert v._coco_annotations() == root / "annotations" / "instances_val2017.json"
    (root / "annotations" / "instances_val2017.json").unlink()
    assert v._coco_annotations() is None


def test_save_dir_numbering(tmp_path, monkeypatch):
    from yololite.cfg import get_cfg, get_save_dir

    monkeypatch.chdir(tmp_path)
    args = get_cfg(overrides={"mode": "val"})
    assert get_save_dir(args) == Path("runs/detect/val")
    Path("runs/detect/val").mkdir(parents=True)
    assert get_save_dir(args) == Path("runs/detect/val2")
    assert get_save_dir(get_cfg(overrides={"mode": "val", "exist_ok": True})) == Path("runs/detect/val")
    assert get_save_dir(get_cfg(overrides={"mode": "val", "project": "p", "name": "n"})) == Path("p/n")


def test_unsupported_evaluations_raise():
    from yololite.utils.cocoeval import COCO, COCOeval

    gt = COCO(_set([1], [(1, 1, 1, [0, 0, 10, 10], None, 0)]))
    dt = gt.loadRes([_dt(1, [0, 0, 10, 10], .5)])
    assert dt.anns[1]["area"] == 100.0 and dt.anns[1]["iscrowd"] == 0
    for t in ("segm", "keypoints"):
        with pytest.raises(NotImplementedError):
            COCOeval(gt, dt, t)
    ev = COCOeval(gt, dt, "bbox")
    ev.params.useCats = 0
    with pytest.raises(NotImplementedError):
        ev.evaluate()
    with pytest.raises(AssertionError):
        gt.loadRes([_dt(2, [0, 0, 10, 10], .5)])      # image 2 is not in the annotations


def test_results_grouping_orders_by_score_and_cuts():
    from yololite.utils.cocoeval import _flat

    dts = [{"image_id": i, "category_id": c, "score": sc} for i, c, sc in
           [(5, 1, .3), (2, 1, .3), (5, 1, .9), (5, 1, .3), (5, 2, .1), (9, 1, .5), (5, 1, -0.0), (5, 1, 0.0)]]
    key, rows = _flat(dts, {2: 0, 5: 1}, {1: 0, 2: 1}, 2, max_det=3)
    # (cat 1, image 2), (cat 1, image 5) cut to its 3 best with the tie in list order, (cat 2, image 5); image 9 dropped
    assert key.tolist() == [0, 1, 1, 1, 3]
    assert [[id(d) for d in dts].index(id(r)) for r in rows] == [1, 2, 0, 3, 4]
    key, rows = _flat(dts, {2: 0, 5: 1}, {1: 0, 2: 1}, 2, max_det=100)
    assert [[id(d) for d in dts].index(id(r)) for r in rows] == [1, 2, 0, 3, 6, 7, 4]      # -0.0 and 0.0 tie


@pytest.mark.parametrize("bad", ["gt_box", "gt_area", "dt_box", "score"])
def test_non_finite_inputs_raise(bad):
    from yololite.utils.cocoeval import COCO, COCOeval

    gt = _set([1], [(1, 1, 1, [0, 0, 10, float("nan") if bad == "gt_box" else 10],
                     float("inf") if bad == "gt_area" else None, 0)])
    g = COCO(gt)
    dt = g.loadRes([_dt(1, [0, 0, float("nan") if bad == "dt_box" else 10, 10], float("nan") if bad == "score" else .5)])
    with pytest.raises(ValueError, match="finite"):
        COCOeval(g, dt, "bbox").evaluate()
