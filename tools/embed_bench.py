"""Cost of feature embeddings on the B200: the plain `infer_nms` step against `infer_embed` steps in one process, plus
CUDA-event times of yl_embed_pool on one tap larger than L2 and one that is not.

    python tools/embed_bench.py [--bs 64] [--imgsz 640] [--steps 50] [--out FILE.json]

yolo11n with seeded weights, device-resident fp32 inputs (two batches, alternated).  The pool kernel is timed over
`--reps` back-to-back launches between two events on the real layer outputs of the last step.  The layer-2 tap (160² x 64
channels, 210 MB at bs 64) is larger than the 126 MB L2, so every launch streams it from HBM; the layer-22 tap (20² x 256,
13 MB) stays in L2 across launches, so its rate is an L2 rate and is reported against the HBM figure for scale only.
Algorithmic bytes count every tap element read once and every output element written once.
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
from yololite._ops import View  # noqa: E402
from yololite.nn.tasks import DetectionModel  # noqa: E402

SETS = {"embed_22": [22], "embed_4_6_10_16_19_22": [4, 6, 10, 16, 19, 22]}


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
    arms = {"plain_infer_nms": lambda x: m.infer_nms(x, **kw)}
    for name, idx in SETS.items():
        arms[name] = lambda x, idx=idx: m.infer_embed(x, idx)

    def rate(step):
        for x in xs:                                    # build / capture every plan first
            step(x)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(a.steps):
            step(xs[i % 2])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / a.steps
        return ms, B / ms * 1e3

    # alternate the arms twice: other work on the host shows up as a spread between the repeats
    runs = {k: [] for k in arms}
    for _ in range(2):
        for k, step in arms.items():
            runs[k].append(rate(step))

    # the pool kernel alone, on the layer outputs the [4, 6, 10, 16, 19, 22] plan and a layer-2 plan hold
    plans = m.__dict__["_yl_plans"]
    m.infer_embed(xs[0], [2])
    torch.cuda.synchronize()

    def taps_of(idx):
        plan = plans[next(k for k in plans if k[0] == tuple(xs[0].shape) and k[-1] == tuple(idx))][0]
        fn, args, keep = plan.calls[-1]
        assert fn.__name__ == "yl_embed_pool"
        arr = keep[0]
        return [View(next(b for b in plan.buffers if b.dim() == 4 and b.data_ptr() == t.x.data), t.x.coff, t.x.c)
                for t in arr]

    hbm_gbs, _, peak_src = bench.peaks()
    kernels = {}
    for name, idx, where in (("layer2_160x160x64", [2], "HBM (tap > L2)"), ("layer22_20x20x256", [22], "L2-resident"),
                             ("layers_4_6_10_16_19_22", SETS["embed_4_6_10_16_19_22"], "mixed")):
        views = taps_of(idx)
        D = sum(v.c for v in views)
        out = torch.empty((B, D), device=dev)
        taps, _ = _ops.embed_pool_taps(views)
        ws = _ops.embed_pool_workspace(taps, B, D, dev)
        ms = event_ms(lambda: _ops.embed_pool(views, out, ws), a.reps)
        nbytes = sum(v.n * v.h * v.w * v.c * 2 for v in views) + B * D * 4
        bound_ms = nbytes / (hbm_gbs * 1e9) * 1e3
        kernels[name] = {"layers": idx, "D": D, "ms": round(ms, 4), "bytes": nbytes, "GB/s": round(nbytes / ms / 1e6, 1),
                         "hbm_bound_ms": round(bound_ms, 4), "fraction_of_hbm_bound": round(bound_ms / ms, 3),
                         "read_from": where}
    res = {
        "card": card(), "model": "yolo11n (seeded weights)", "batch": B, "imgsz": S, "input": "fp32, device-resident",
        "nms": kw, "steps": a.steps,
        "steps_ms": {k: [round(r[0], 3) for r in v] for k, v in runs.items()},
        "images_per_s": {k: [round(r[1]) for r in v] for k, v in runs.items()},
        "launches": {k: plans[next(p for p in plans if p[0] == tuple(xs[0].shape) and p[-1] == tuple(idx))][0].n_launches
                     for k, idx in SETS.items()},
        "kernels": {"yl_embed_pool": kernels}, "hbm_peak_GBps": hbm_gbs, "hbm_peak_source": peak_src,
    }
    if a.out:
        out = Path(a.out)
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
