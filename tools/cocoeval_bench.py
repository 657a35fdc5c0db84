"""Cost of COCO evaluation (`save_json=True`) on a synthetic set of COCO val2017 size: 5000 images, 80 categories,
~35k gts, 300 detections per image (1.5M results, the validator's max_det).

    python tools/cocoeval_bench.py [--rounds 5] [--out FILE.json]

1. `COCOeval.evaluate()` + `accumulate()` on the GPU, host clock around work that ends in a device synchronise:
   the whole calls (host-side grouping of the result dicts and uploads included), and the device part alone
   (`yl_cocoeval_evaluate`, the stable sorts and gathers, `yl_cocoeval_accumulate`) with CUDA events, relaunched on the same inputs.
2. The numpy restatement of pycocotools (oracle/cocoeval_ref.py) on the same input, once; its arrays are checked
   bit-identical to the GPU's.  pycocotools itself is not installed here and is not timed.
3. The host side around it: building the predictions.json rows with `DetectionValidator.pred_to_json` from 5000
   per-image (300, 6) fp32 tensors, `json.dump` to a temporary file, `COCO(...)` + `loadRes(...)` of that file.

The card name, power limit and max SM clock are read in the same run.
"""
import argparse
import copy
import json
import statistics
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]
from oracle import cocoeval_ref as R  # noqa: E402
from yololite import _C  # noqa: E402
from yololite.utils import LOGGER  # noqa: E402
from yololite.utils.cocoeval import COCO, COCOeval  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def gpu_eval(gt_coco, dt_coco):
    ev = COCOeval(gt_coco, dt_coco, "bbox")
    ev.evaluate()
    ev.accumulate()
    return ev


def device_ms(ev, reps):
    """CUDA-event time of evaluate launch + sorts + accumulate launch on the evaluator's resident inputs."""
    lib, g = _C.load(), ev._g
    p = ev.params
    T, R_, K, A, M = len(p.iouThrs), len(p.recThrs), len(p.catIds), len(p.areaRng), len(p.maxDets)
    prec = torch.empty((T, R_, K, A, M), dtype=torch.float64, device="cuda")
    rec = torch.empty((T, K, A, M), dtype=torch.float64, device="cuda")
    sc = torch.empty_like(prec)

    def once():
        _C.check(lib.yl_cocoeval_evaluate(ev._set, ev._params, ev._slots, _C.stream_ptr()), "yl_cocoeval_evaluate")
        by_score = torch.sort(g["key"], stable=True)[1]
        order = by_score[torch.sort(g["slot_cat"][by_score], stable=True)[1]]
        S = order.numel()
        score, rank = g["dt_score"][order], g["rank"][order]
        flags = g["flags"].view(A * T, S)[:, order].contiguous()
        _C.check(lib.yl_cocoeval_accumulate(ev._params, K, S, g["cat_slot_off"].data_ptr(), score.data_ptr(),
                                            rank.data_ptr(), flags.data_ptr(), g["npig"].data_ptr(), prec.data_ptr(),
                                            rec.data_ptr(), sc.data_ptr(), _C.stream_ptr()), "yl_cocoeval_accumulate")

    for _ in range(2):
        once()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        once()
    e1.record()
    torch.cuda.synchronize()
    assert np.array_equal(prec.cpu().numpy(), ev.eval["precision"]) and np.array_equal(rec.cpu().numpy(), ev.eval["recall"])
    return e0.elapsed_time(e1) / reps


def json_case(gt, rounds):
    from yololite.engine.validator import DetectionValidator
    from yololite.utils import ops

    g = torch.Generator().manual_seed(7)
    ids = [im["id"] for im in gt["images"]]
    predn = torch.zeros((len(ids), 300, 6))
    xy = torch.rand((len(ids), 300, 2), generator=g) * 560
    predn[..., :2], predn[..., 2:4] = xy, xy + torch.rand((len(ids), 300, 2), generator=g) * 200 + 2
    predn[..., 4] = torch.sort(torch.rand((len(ids), 300), generator=g), 1, descending=True)[0]
    predn[..., 5] = torch.randint(0, 80, (len(ids), 300), generator=g).float()
    files = [f"/coco/images/val2017/{i:012d}.jpg" for i in ids]
    out = {"rows_ms": [], "dump_ms": [], "load_ms": []}
    with tempfile.TemporaryDirectory() as d:
        for _ in range(rounds):
            v = DetectionValidator(dataloader=[])
            v.class_map = ops.coco80_to_coco91_class()
            t0 = time.perf_counter()
            for i, f in enumerate(files):
                v.pred_to_json(predn[i], f)
            t1 = time.perf_counter()
            with open(Path(d) / "predictions.json", "w") as fh:
                json.dump(v.jdict, fh)
            t2 = time.perf_counter()
            anno = COCO(copy.deepcopy(gt))
            anno.loadRes(str(Path(d) / "predictions.json"))
            t3 = time.perf_counter()
            out["rows_ms"].append((t1 - t0) * 1e3)
            out["dump_ms"].append((t2 - t1) * 1e3)
            out["load_ms"].append((t3 - t2) * 1e3)
    return {"images": len(ids), "rows": len(v.jdict), **{k: round(statistics.median(x), 1) for k, x in out.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--images", type=int, default=5000)
    ap.add_argument("--skip-oracle", action="store_true")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "cocoeval_bench_val2017size.json"))
    a = ap.parse_args()
    LOGGER.setLevel("WARNING")
    torch.cuda.init()
    _C.init(0)
    gt, res = R.synthetic_coco(2017, n_images=a.images, n_cats=80, gts_per_image=7, dts_per_image=300, fixed_dts=True)
    gt_coco = COCO(copy.deepcopy(gt))
    dt_coco = gt_coco.loadRes(copy.deepcopy(res))
    ev = gpu_eval(gt_coco, dt_coco)                      # warm-up (module load, sort kernels)
    walls = []
    for _ in range(a.rounds):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ev = gpu_eval(gt_coco, dt_coco)
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
    dev_ms = [device_ms(ev, a.reps) for _ in range(a.rounds)]
    result = {
        "card": card(),
        "set": {"images": len(gt["images"]), "categories": len(gt["categories"]), "gts": len(gt["annotations"]),
                "results": len(res), "pairs": int(ev._g["pair_cat"].numel()), "kept_dt_slots": int(ev._g["key"].numel())},
        "gpu_evaluate_accumulate_wall_ms": round(statistics.median(walls), 1),
        "gpu_evaluate_accumulate_wall_ms_all": [round(x, 1) for x in walls],
        "gpu_device_ms": round(statistics.median(dev_ms), 3),
        "gpu_device_ms_all": [round(x, 3) for x in dev_ms],
    }
    if not a.skip_oracle:
        t0 = time.perf_counter()
        g = R.COCO(copy.deepcopy(gt))
        ref = R.COCOeval(g, g.loadRes(copy.deepcopy(res)))
        ref.evaluate()
        ref.accumulate()
        result["oracle_numpy_evaluate_accumulate_s"] = round(time.perf_counter() - t0, 1)
        result["bit_identical"] = all(np.array_equal(ev.eval[k], ref.eval[k]) for k in ("precision", "recall", "scores"))
    result["predictions_json"] = json_case(gt, max(1, a.rounds // 2))
    print(json.dumps(result, indent=1))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
