"""Cost of a model ensemble on the B200: the ensemble's `infer_nms` step against each member's own step (and their sum)
in one process, for yolo11n x 2 (differently seeded) and yolo11n + yolo11s at bs 64 and bs 1; the members on parallel
graph branches against the members recorded one after the other; CUDA-event times of yl_detect_decode_into for an nc = 3
member and of the NMS on the ensemble's prediction next to the NMS on one member's.

    python tools/ensemble_bench.py [--imgsz 640] [--steps 50] [--out FILE.json]

Seeded weights, device-resident fp32 inputs (two batches, alternated), conf 0.25, iou 0.7.  Every arm is timed twice,
alternating, so that other work on the host shows up as a spread between the repeats.  A bs 1 arm runs 10x the steps.
The decode is timed over `--reps` back-to-back launches between two events; its working set at bs 64 (~260 MB) is larger
than L2, so every launch streams from HBM.  Algorithmic bytes count every element the kernel must read or write once.
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
from yololite.nn.tasks import DetectionModel, Ensemble  # noqa: E402


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


def step_ms(model, xs, steps, kw):
    """Device time of one infer_nms step of `model`, alternating the batches `xs` (plans built and captured first)."""
    for x in xs:
        model.infer_nms(x, **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        model.infer_nms(xs[i % len(xs)], **kw)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--imgsz", type=int, default=640)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    S = a.imgsz
    kw = dict(conf=0.25, iou=0.7)

    def model(cfg, salt, nc=None):
        return fill_state_dict_(DetectionModel(cfg, nc=nc, verbose=False), salt).eval().to(dev)

    n0, n1, s0 = model("yolo11n.yaml", 0), model("yolo11n.yaml", 1), model("yolo11s.yaml", 0)
    pairs = {"yolo11n x 2": [n0, n1], "yolo11n + yolo11s": [n0, s0]}
    g = torch.Generator(device=dev).manual_seed(0)
    results = {}
    for bs in (64, 1):
        xs = [torch.rand(bs, 3, S, S, device=dev, generator=g) for _ in range(2)]
        steps = a.steps * (10 if bs == 1 else 1)
        for name, ms in pairs.items():
            parallel = Ensemble(ms)
            serial = Ensemble(ms)
            serial._member_lanes = 0          # every member on the same lanes: stream order runs them one after another
            arms = {"ensemble": parallel, "ensemble_serial_members": serial, **{f"member{k}": m for k, m in enumerate(ms)}}
            runs = {k: [] for k in arms}
            for _ in range(2):
                for k, m in arms.items():
                    runs[k].append(step_ms(m, xs, steps, kw))
            best = {k: min(v) for k, v in runs.items()}
            member_sum = sum(best[f"member{k}"] for k in range(len(ms)))
            nms_key = tuple(parallel._yl_plans)[-1][4]
            plan = parallel._get_plan(xs[0].shape, dev, 0, nms_key)[0]
            member_plans = [m._get_plan(xs[0].shape, dev, False, 0, nms_key)[0] for m in ms]
            results[f"{name}, bs {bs}"] = {
                "ms_per_step": {k: [round(t, 4) for t in v] for k, v in runs.items()},
                "images_per_s": {k: round(bs / t * 1e3) for k, t in best.items()},
                "member_sum_ms": round(member_sum, 4),
                "ensemble_over_member_sum": round(best["ensemble"] / member_sum, 3),
                "serial_members_over_parallel": round(best["ensemble_serial_members"] / best["ensemble"], 3),
                "launches": {"ensemble": plan.n_launches, "ensemble_eager_ingests": plan.n_ingest,
                             "members": [p.n_launches for p in member_plans]},
            }

    # yl_detect_decode_into: the unfused head of an nc = 3 yolo11n (raw maps of its three levels) at bs 64, writing the
    # second member's window of a two-member prediction
    B, nc = 64, 3
    no = 64 + nc
    levels = [View(torch.randn(B, S // s, S // s, no, device=dev, generator=g), 0, no) for s in (8, 16, 32)]
    A = sum(v.h * v.w for v in levels)
    y = torch.empty(B, 4 + nc, 2 * A, device=dev)
    dec_ms = event_ms(lambda: _ops.detect_decode(levels, (8, 16, 32), 16, nc, y, anchor_base=A), a.reps)
    dec_bytes = B * A * (no + 4 + nc) * 4
    hbm_gbs, _, peak_src = bench.peaks()
    bound_ms = dec_bytes / (hbm_gbs * 1e9) * 1e3

    # NMS on the ensemble's prediction (yolo11n x 2) next to NMS on one member's
    xb = torch.rand(64, 3, S, S, device=dev, generator=g)
    one = n0.infer(xb)[0].clone()
    both = Ensemble([n0, n1]).infer(xb)[0].clone()
    nms_both = event_ms(lambda: _ops.nms_batched(both, **kw), a.reps)
    nms_one = event_ms(lambda: _ops.nms_batched(one, **kw), a.reps)

    res = {
        "card": card(), "imgsz": S, "input": "fp32, device-resident", "nms": kw, "steps_bs64": a.steps,
        "steps_bs1": a.steps * 10, "weights": "name-keyed seeded (oracle/weights.py); yolo11n x 2 = salts 0 and 1",
        "steps": results,
        "yl_detect_decode_into": {"model": "yolo11n nc=3 head", "batch": B, "anchors": A, "window": [A, 2 * A],
                                  "ms": round(dec_ms, 4), "bytes": dec_bytes, "GB/s": round(dec_bytes / dec_ms / 1e6, 1),
                                  "hbm_bound_ms": round(bound_ms, 4), "fraction_of_hbm_bound": round(bound_ms / dec_ms, 3)},
        "hbm_peak_GBps": hbm_gbs, "hbm_peak_source": peak_src,
        "nms_ms_bs64": {"ensemble_prediction": round(nms_both, 4), "anchors": both.shape[2],
                        "one_member_prediction": round(nms_one, 4), "member_anchors": one.shape[2]},
    }
    if a.out:
        out = Path(a.out)
        out.parent.mkdir(parents=True, exist_ok=True)
        out.write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
