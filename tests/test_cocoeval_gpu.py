"""COCO evaluation (`save_json=True`) on the GPU: `yololite.utils.cocoeval.COCOeval` (csrc/cocoeval.cu) bit-identical to
the numpy restatement of pycocotools (oracle/cocoeval_ref.py) on seeded synthetic sets up to COCO val2017 size, and the
validator's predictions.json + COCO mAP against the oracle, alone and with augment, an ensemble and save_hybrid."""
import copy
import json
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]

from oracle import cocoeval_ref as R  # noqa: E402

pytestmark = pytest.mark.gpu


def _gpu_eval(gt, res, img_ids=None, max_dets=None):
    from yololite.utils.cocoeval import COCO, COCOeval

    g = COCO(copy.deepcopy(gt))
    ev = COCOeval(g, g.loadRes(copy.deepcopy(res)), "bbox")
    if img_ids is not None:
        ev.params.imgIds = list(img_ids)
    if max_dets is not None:
        ev.params.maxDets = list(max_dets)
    ev.evaluate()
    ev.accumulate()
    ev.summarize()
    return ev


def _ref_eval(gt, res, img_ids=None, max_dets=None):
    g = R.COCO(copy.deepcopy(gt))
    ev = R.COCOeval(g, g.loadRes(copy.deepcopy(res)))
    if img_ids is not None:
        ev.params.imgIds = list(img_ids)
    if max_dets is not None:
        ev.params.maxDets = list(max_dets)
    ev.evaluate()
    ev.accumulate()
    ev.summarize()
    return ev


def _assert_same(ev, ref):
    for k in ("precision", "recall", "scores"):
        assert ev.eval[k].dtype == np.float64 and ev.eval[k].shape == ref.eval[k].shape, k
        assert np.array_equal(ev.eval[k], ref.eval[k]), (k, np.argwhere(ev.eval[k] != ref.eval[k])[:5])
    assert np.array_equal(ev.stats, ref.stats), (ev.stats, ref.stats)


@pytest.mark.parametrize("seed,kw", [
    (0, {}),
    (1, dict(crowd_frac=0.3)),                                   # many crowds: ignore break, many-to-one matches
    (2, dict(id_zero=True, gts_per_image=20, dts_per_image=150)),   # dense overlaps, a gt with id 0
    (3, dict(n_images=8, dts_per_image=400)),                    # > maxDets[-1] dts in one (image, category)
    (4, dict(n_images=100, n_cats=20, gts_per_image=3, dts_per_image=30)),
])
def test_cocoeval_bit_identical_to_oracle(seed, kw):
    gt, res = R.synthetic_coco(seed, **kw)
    _assert_same(_gpu_eval(gt, res), _ref_eval(gt, res))


def test_cocoeval_params_subset_and_other_max_dets():
    gt, res = R.synthetic_coco(5, n_images=30)
    ids = sorted(i["id"] for i in gt["images"])[::2] + [sorted(i["id"] for i in gt["images"])[0]]   # duplicates too
    _assert_same(_gpu_eval(gt, res, ids, [20, 1, 5]), _ref_eval(gt, res, ids, [20, 1, 5]))


def test_cocoeval_val2017_size():
    """5000 images, 80 categories, ~35k gts, 300 dts per image (1.5M results)."""
    gt, res = R.synthetic_coco(2017, n_images=5000, n_cats=80, gts_per_image=7, dts_per_image=300, fixed_dts=True)
    assert len(res) == 1_500_000 and 30_000 < len(gt["annotations"]) < 40_000
    _assert_same(_gpu_eval(gt, res), _ref_eval(gt, res))


def test_cocoeval_empty_inputs():
    gt = {"images": [{"id": 1}, {"id": 2}], "annotations": [], "categories": [{"id": 1}, {"id": 3}]}
    ev = _gpu_eval(gt, [])
    for k in ("precision", "recall", "scores"):
        assert (ev.eval[k] == -1).all()
    assert (ev.stats == -1).all()
    # results but no gts: still -1 everywhere
    ev = _gpu_eval(gt, [{"image_id": 1, "category_id": 3, "bbox": [0.0, 0.0, 5.0, 5.0], "score": 0.5}])
    assert (ev.eval["precision"] == -1).all() and (ev.stats == -1).all()


# ------------------------------------------------------------------------------------------------ validator
def _model():
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    return yl


def _coco_layout(root, yl):
    """COCO val2017 layout (images/val2017, labels/val2017, val2017.txt, annotations/instances_val2017.json) of 6
    noise images.  The gts are some of the validator's own detections (from a probe run on the same loader), shrunk
    a little, one of them crowd, so the COCO mAP is not 0."""
    import cv2

    from yololite.utils import ops

    cmap = ops.coco80_to_coco91_class()
    for d in ("images/val2017", "labels/val2017", "annotations"):
        (root / d).mkdir(parents=True)
    rng = np.random.default_rng(0)
    images, lines = [], []
    for k, (h, w) in enumerate([(64, 64), (48, 80), (80, 48), (64, 96), (40, 40), (72, 64)]):
        iid = 1000 + 37 * k
        f = root / "images" / "val2017" / f"{iid:012d}.png"
        cv2.imwrite(str(f), rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        images.append({"id": iid, "width": w, "height": h, "file_name": f.name})
        lines.append(f"./images/val2017/{f.name}\n")
    (root / "val2017.txt").write_text("".join(lines))
    yaml = root / "coco.yaml"
    yaml.write_text(f"path: {root}\nval: val2017.txt\nnames:\n" + "".join(f"  {i}: c{i}\n" for i in range(80)))
    probe, _ = _run(yl.model, yaml, root / "probe", save_json=True)
    anns = []
    for predn, f in probe.calls:
        k = [im["file_name"] for im in images].index(Path(f).name)
        h, w = images[k]["height"], images[k]["width"]
        rows = []
        for j, b in enumerate(predn.numpy()[: 1 + k % 3]):
            x1, y1, x2, y2 = (float(v) for v in b[:4])
            s = 0.9 - 0.05 * j
            cx, cy, bw, bh = (x1 + x2) / 2, (y1 + y2) / 2, (x2 - x1) * s, (y2 - y1) * s
            rows.append(f"{int(b[5])} {cx / w} {cy / h} {bw / w} {bh / h}\n")
            anns.append({"id": len(anns) + 1, "image_id": images[k]["id"], "category_id": cmap[int(b[5])],
                         "bbox": [cx - bw / 2, cy - bh / 2, bw, bh], "area": bw * bh * 0.8, "iscrowd": int(j == 2)})
        (root / "labels" / "val2017" / f"{Path(f).stem}.txt").write_text("".join(rows))
    assert len(anns) >= 6
    gt = {"images": images, "annotations": anns, "categories": [{"id": c, "name": str(c)} for c in cmap]}
    (root / "annotations" / "instances_val2017.json").write_text(json.dumps(gt))
    return yaml, gt


def _run(model, yaml, save_dir, **extra):
    """DetectionValidator over the yaml's split, recording what pred_to_json receives."""
    from yololite.data import build_val_loader
    from yololite.engine.validator import DetectionValidator

    class Rec(DetectionValidator):
        def pred_to_json(self, predn, filename):
            self.calls.append((predn.clone(), filename))
            return super().pred_to_json(predn, filename)

    loader, _ = build_val_loader(yaml, imgsz=64, batch_size=4, stride=32)
    args = dict(data=str(yaml), imgsz=64, batch=4, conf=0.001, iou=0.7, device=0, verbose=False, **extra)
    v = Rec(dataloader=loader, save_dir=save_dir, args=args)
    v.calls = []
    stats = v(model=model)
    return v, stats


def _check_against_oracle(model, yaml, gt, save_dir, **extra):
    v, stats = _run(model, yaml, save_dir, save_json=True, **extra)
    cmap = R.coco80_to_coco91_class()
    want = [row for predn, f in v.calls for row in R.pred_to_json(predn.numpy(), f, cmap)]
    assert len(want) > 0
    assert (save_dir / "predictions.json").read_text() == json.dumps(want)
    ref = R.evaluate(gt, want, img_ids=[im["id"] for im in gt["images"]])
    assert v.coco_eval is not None
    _assert_same(v.coco_eval, ref)
    assert stats["metrics/mAP50-95(B)"] == ref.stats[0] and stats["metrics/mAP50(B)"] == ref.stats[1]
    assert ref.stats[1] > 0
    return v, stats


def test_val_save_json_matches_oracle(tmp_path):
    yl = _model()
    yaml, gt = _coco_layout(tmp_path / "coco", yl)
    v, stats = _check_against_oracle(yl.model, yaml, gt, tmp_path / "out")
    assert v.is_coco and v.class_map == R.coco80_to_coco91_class()
    # the public API: runs/<project>/<name>, numbered when it exists
    yl.val(data=str(yaml), imgsz=64, batch=4, conf=0.001, device=0, verbose=False, save_json=True,
           project=str(tmp_path / "p"), name="val")
    yl.val(data=str(yaml), imgsz=64, batch=4, conf=0.001, device=0, verbose=False, save_json=True,
           project=str(tmp_path / "p"), name="val")
    want = (tmp_path / "out" / "predictions.json").read_text()
    assert (tmp_path / "p" / "val" / "predictions.json").read_text() == want
    assert (tmp_path / "p" / "val2" / "predictions.json").read_text() == want


def test_val_save_json_off_changes_nothing(tmp_path, monkeypatch):
    yl = _model()
    yaml, gt = _coco_layout(tmp_path / "coco", yl)
    monkeypatch.chdir(tmp_path)
    v_off, off = _run(yl.model, yaml, None)
    _, plain = _run(yl.model, yaml, None, save_json=False)
    assert off == plain and v_off.jdict == [] and v_off.coco_eval is None
    assert not (tmp_path / "runs").exists()
    # the detections are the same with the switch on: only the two COCO keys are replaced
    v_on, on = _run(yl.model, yaml, None, save_json=True)
    assert (tmp_path / "runs" / "detect" / "val" / "predictions.json").is_file()
    for k in ("metrics/precision(B)", "metrics/recall(B)"):
        assert on[k] == off[k]


def test_val_save_json_composes_with_augment_ensemble_and_hybrid(tmp_path):
    from oracle.weights import fill_state_dict_
    from yololite.nn.tasks import DetectionModel, Ensemble

    yl = _model()
    yaml, gt = _coco_layout(tmp_path / "coco", yl)
    _check_against_oracle(yl.model, yaml, gt, tmp_path / "aug", augment=True)
    _, plain = _check_against_oracle(yl.model, yaml, gt, tmp_path / "plain")
    _, hyb = _check_against_oracle(yl.model, yaml, gt, tmp_path / "hyb", save_hybrid=True)
    assert hyb["metrics/mAP50-95(B)"] > plain["metrics/mAP50-95(B)"]   # the gts are in the predictions
    other = fill_state_dict_(DetectionModel("yolo11n.yaml", verbose=False), 1).eval()
    ens = Ensemble([yl.model, other]).cuda().eval()
    _check_against_oracle(ens, yaml, gt, tmp_path / "ens")
