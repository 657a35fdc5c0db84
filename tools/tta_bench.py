"""Cost of test-time augmentation on the B200: plain `infer_nms` against `infer_nms(augment=True)` in one process, plus
CUDA-event times of the two TTA kernels and of the NMS on the merged prediction.

    python tools/tta_bench.py [--bs 64] [--imgsz 640] [--steps 50] [--out FILE.json]

yolo11n with seeded weights, device-resident fp32 inputs (two batches, alternated).  Each kernel is timed over `--reps`
back-to-back launches between two events; its working set (>= 300 MB at bs=64) is larger than L2, so every launch
streams from HBM.  Algorithmic bytes count every element the kernel must read or write once.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]
import bench  # noqa: E402
from oracle.weights import fill_state_dict_  # noqa: E402
from yololite import _ops  # noqa: E402
from yololite.nn.tasks import DetectionModel, tta_geometry  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def event_ms(fn, reps):
    """Mean device time of one call of `fn` over `reps` back-to-back calls (after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--bs", type=int, default=64)
    ap.add_argument("--imgsz", type=int, default=640)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    m = fill_state_dict_(DetectionModel("yolo11n.yaml", verbose=False)).eval().to(dev)
    B, S = a.bs, a.imgsz
    g = torch.Generator(device=dev).manual_seed(0)
    xs = [torch.rand(B, 3, S, S, device=dev, generator=g) for _ in range(2)]
    kw = dict(conf=0.25, iou=0.7)

    def rate(augment):
        for x in xs:                                    # build / capture every plan first
            m.infer_nms(x, augment=augment, **kw)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.steps):
            m.infer_nms(xs[i % 2], augment=augment, **kw)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.steps
        return ms, B / ms * 1e3

    # alternate the two arms twice: other work on the host shows up as a spread between the repeats
    runs = {"plain": [], "tta": []}
    for _ in range(2):
        runs["plain"].append(rate(False))
        runs["tta"].append(rate(True))

    # the kernels on the real buffers of the last TTA step
    geo = tta_geometry(S, S, m.model[-1].stride.tolist())
    x = xs[0]
    canv = [torch.empty(B, 3, p.H, p.W, device=dev) for p in geo[1:]]
    scale_ms = event_ms(lambda: _ops.tta_scale_img(x, [(c, (p.h, p.w), p.flip) for c, p in zip(canv, geo[1:])]), a.reps)
    preds = [m.infer(torch.rand(B, 3, p.H, p.W, device=dev, generator=g))[0].clone() for p in geo]
    merged = torch.empty(B, preds[0].shape[1], sum(p.n for p in geo), device=dev)
    merge_ms = event_ms(lambda: _ops.tta_merge([(t, p.a0, p.n, p.scale, p.flip) for t, p in zip(preds, geo)], S, merged),
                        a.reps)
    nms_merged_ms = event_ms(lambda: _ops.nms_batched(merged, **dict(conf=kw["conf"], iou=kw["iou"])), a.reps)
    nms_plain_ms = event_ms(lambda: _ops.nms_batched(preds[0], **dict(conf=kw["conf"], iou=kw["iou"])), a.reps)

    hbm_gbs, _, peak_src = bench.peaks()
    rows = preds[0].shape[1]
    scale_bytes = x.numel() * 4 + sum(c.numel() * 4 for c in canv)
    merge_bytes = 2 * B * rows * merged.shape[2] * 4
    kernels = {}
    for name, ms, nbytes in (("yl_tta_scale_img", scale_ms, scale_bytes), ("yl_tta_merge", merge_ms, merge_bytes)):
        bound_ms = nbytes / (hbm_gbs * 1e9) * 1e3
        kernels[name] = {"ms": round(ms, 4), "bytes": nbytes, "GB/s": round(nbytes / ms / 1e6, 1),
                         "hbm_bound_ms": round(bound_ms, 4), "fraction_of_hbm_bound": round(bound_ms / ms, 3)}
    res = {
        "card": card(), "model": "yolo11n (seeded weights)", "batch": B, "imgsz": S, "input": "fp32, device-resident",
        "nms": kw, "steps": a.steps,
        "plain": {"ms_per_step": [round(r[0], 3) for r in runs["plain"]], "images_per_s": [round(r[1]) for r in runs["plain"]]},
        "tta": {"ms_per_step": [round(r[0], 3) for r in runs["tta"]], "images_per_s": [round(r[1]) for r in runs["tta"]]},
        "anchors": {"plain": geo[0].A, "tta_merged": merged.shape[2],
                    "passes": [{"canvas": [p.H, p.W], "content": [p.h, p.w], "A": p.A, "kept": p.n} for p in geo]},
        "kernels": kernels, "hbm_peak_GBps": hbm_gbs, "hbm_peak_source": peak_src,
        "nms_ms": {"merged": round(nms_merged_ms, 4), "plain_prediction": round(nms_plain_ms, 4)},
    }
    if a.out:
        out = Path(a.out)
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
