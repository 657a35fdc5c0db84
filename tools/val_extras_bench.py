"""Cost of the validator switches on the B200: NMS with ground-truth priors (save_hybrid), the confusion kernel (plots)
and one validator batch with both switches off and on.

    python tools/val_extras_bench.py [--parent-lib PATH] [--out FILE.json]

1. `yl_nms_batched` without priors against `yl_nms_batched_priors` with 20 priors per image, at validator settings:
   B = 64, A = 8400, nc = 80, conf 0.001, multi-label, iou 0.7, max_det 300 (the sparse score regime of bench.py's
   nms_stress: sigmoid(N(-12, 1.5)) class scores, a few % of anchors above conf).
2. `yl_confusion_matrix` at B = 64, max_det = 300 with ~8 labels per image.
3. One DetectionValidator batch (postprocess + update_metrics on a fixed 64-image prediction), switches off and on.
4. With `--parent-lib` (a libyl11.so built from the parent commit): bench.py's nms_stress cases (B = 256, dense and
   sparse, both label modes), `yl_nms_batched` of this tree and of the parent library alternated round by round in
   this one process, through the same C call.

Times are CUDA events around `--reps` back-to-back calls after warm-up, median over `--rounds` rounds.  The card name,
power limit and max SM clock are read in the same run.
"""
import argparse
import ctypes as C
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]
from yololite import _C, _ops  # noqa: E402
from yololite.utils import ops  # noqa: E402
from yololite.utils.metrics import ConfusionMatrix  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or torch.cuda.get_device_name(0)


def event_ms(fn, reps):
    """Mean device time of one call of `fn` over `reps` back-to-back calls (after 3 warm-up calls)."""
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def pred_tensor(B, A, nc, mean, std, seed=2):
    g = torch.Generator(device="cuda").manual_seed(seed)
    pred = torch.empty((B, 4 + nc, A), device="cuda")
    pred[:, 0:2] = torch.rand((B, 2, A), device="cuda", generator=g) * 640
    pred[:, 2:4] = torch.rand((B, 2, A), device="cuda", generator=g) * 248 + 8
    pred[:, 4:] = torch.sigmoid(torch.randn((B, nc, A), device="cuda", generator=g) * std + mean)
    return pred


def priors(B, per_image, nc, seed=3):
    g = torch.Generator().manual_seed(seed)
    lb = [torch.cat([torch.randint(0, nc, (per_image, 1)).float(), torch.rand((per_image, 2), generator=g) * 640,
                     torch.rand((per_image, 2), generator=g) * 248 + 8], 1) for _ in range(B)]
    xywh, cls, offs = ops.pack_priors(lb)
    return xywh.cuda().contiguous(), cls.cuda().to(torch.int32), offs


def nms_priors_case(rounds, reps):
    B, A, nc = 64, 8400, 80
    pred = pred_tensor(B, A, nc, -12.0, 1.5)
    lab = priors(B, 20, nc)
    plain = lambda: _ops.nms_batched(pred, 0.001, 0.7, multi_label=True, max_det=300)  # noqa: E731
    with_priors = lambda: _ops.nms_batched(pred, 0.001, 0.7, multi_label=True, max_det=300, labels=lab)  # noqa: E731
    a, b = [], []
    for _ in range(rounds):
        a.append(event_ms(plain, reps))
        b.append(event_ms(with_priors, reps))
    d0, c0 = plain()
    d1, c1 = with_priors()
    return {"B": B, "A": A, "nc": nc, "conf": 0.001, "iou": 0.7, "multi_label": True, "priors_per_image": 20,
            "no_priors_ms": round(statistics.median(a), 4), "priors_ms": round(statistics.median(b), 4),
            "ratio": round(statistics.median(b) / statistics.median(a), 4),
            "detections_no_priors": int(c0.sum()), "detections_priors": int(c1.sum())}


def confusion_case(rounds, reps):
    B, max_det, nc = 64, 300, 80
    g = torch.Generator().manual_seed(4)
    dets = torch.zeros((B, max_det, 6))
    xy = torch.rand((B, max_det, 2), generator=g) * 600
    dets[..., :2], dets[..., 2:4] = xy, xy + torch.rand((B, max_det, 2), generator=g) * 200 + 10
    dets[..., 4] = torch.sort(torch.rand((B, max_det), generator=g), 1, descending=True)[0]
    dets[..., 5] = torch.randint(0, nc, (B, max_det), generator=g).float()
    counts = torch.full((B,), max_det, dtype=torch.int32)
    L = 8 * B
    gt = dets[torch.arange(L) % B, torch.arange(L) % 50, :4] + torch.randn((L, 4), generator=g) * 4
    gtc = dets[torch.arange(L) % B, torch.arange(L) % 50, 5]
    order = torch.argsort(torch.arange(L) % B, stable=True)
    gt, gtc = gt[order].cuda(), gtc[order].cuda()
    offs = [8 * i for i in range(B + 1)]
    dets, counts = dets.cuda(), counts.cuda()
    cm = ConfusionMatrix(nc, 0.001)
    fn = lambda: cm.process_batched(dets, counts, gt, gtc, offs)  # noqa: E731
    ts = [event_ms(fn, reps) for _ in range(rounds)]
    return {"B": B, "max_det": max_det, "nc": nc, "labels_per_image": 8, "ms": round(statistics.median(ts), 4),
            "matrix_sum": float(cm.matrix.sum())}


def validator_case(rounds):
    """postprocess + update_metrics of one 64-image batch at 640², host clock around work that ends in a sync."""
    import time

    from yololite.engine.validator import DetectionValidator

    B, A, nc = 64, 8400, 80
    pred = pred_tensor(B, A, nc, -12.0, 1.5, seed=5)
    g = torch.Generator().manual_seed(6)
    n = 20 * B
    batch = {"img": torch.zeros((B, 3, 640, 640), dtype=torch.uint8), "cls": torch.randint(0, nc, (n, 1), generator=g).float(),
             "bboxes": torch.rand((n, 4), generator=g) * 0.3 + 0.1, "batch_idx": (torch.arange(n) % B).float(),
             "ori_shape": [(640, 640)] * B, "ratio_pad": [None] * B}
    out = {"off": [], "on": []}
    for _ in range(rounds):
        for tag, sw in (("off", False), ("on", True)):
            v = DetectionValidator(dataloader=[], args={"save_hybrid": sw, "plots": sw, "verbose": False})
            v.device = torch.device("cuda", 0)
            v.init_metrics(type("M", (), {"names": {i: str(i) for i in range(nc)}})())
            for k in range(4):
                b = v.preprocess(dict(batch))
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                v.update_metrics(v.postprocess(pred), b)
                if v.confusion_matrix is not None:
                    v.confusion_matrix.tp_fp()   # the host read of the matrix
                torch.cuda.synchronize()
                if k:
                    out[tag].append((time.perf_counter() - t0) * 1e3)
    return {"B": B, "labels_per_image": 20, "conf": 0.001, "iou": 0.7,
            "off_ms": round(statistics.median(out["off"]), 3), "on_ms": round(statistics.median(out["on"]), 3),
            "note": "postprocess + update_metrics (+ the matrix read when on), host clock, synchronised"}


def nms_stress_ab(parent_lib, rounds, reps):
    """bench.py's nms_stress cases through `yl_nms_batched` of this tree's library and of `parent_lib`, alternated."""
    libs = {}
    for tag, path in (("this", _C.lib_path()), ("parent", Path(parent_lib))):
        lib = C.CDLL(str(path))
        lib.yl_init.argtypes = [C.c_int]
        lib.yl_nms_workspace_bytes.restype = C.c_size_t
        lib.yl_nms_workspace_bytes.argtypes = [C.c_int] * 4
        lib.yl_nms_batched.argtypes = _C._PROTOTYPES["yl_nms_batched"][1]
        assert lib.yl_init(0) == 0, tag
        libs[tag] = lib
    B, A, nc = 256, 8400, 80
    out = torch.empty((B, 300, 6), device="cuda")
    cnt = torch.empty((B,), dtype=torch.int32, device="cuda")
    res = {}
    for regime, (mean, std) in (("dense", (-5.0, 2.0)), ("sparse", (-12.0, 1.5))):
        pred = pred_tensor(B, A, nc, mean, std)
        for multi in (0, 1):
            ws = torch.empty(libs["this"].yl_nms_workspace_bytes(B, A, nc, multi), dtype=torch.uint8, device="cuda")
            ts = {"this": [], "parent": []}
            dumps = {}
            for _ in range(rounds):
                for tag, lib in libs.items():
                    def fn(lib=lib):
                        rc = lib.yl_nms_batched(pred.data_ptr(), B, nc, A, 0.001, 0.7, None, 0, 0, multi, 300, 30000,
                                                7680.0, ws.data_ptr(), ws.numel(), out.data_ptr(), cnt.data_ptr(),
                                                _C.stream_ptr())
                        assert rc == 0
                    ts[tag].append(event_ms(fn, reps))
                    dumps[tag] = (out.clone(), cnt.clone())
            same = torch.equal(dumps["this"][0], dumps["parent"][0]) and torch.equal(dumps["this"][1], dumps["parent"][1])
            t, p = statistics.median(ts["this"]), statistics.median(ts["parent"])
            res[f"{regime}_{'multi' if multi else 'single'}_label"] = {
                "this_ms": round(t, 4), "parent_ms": round(p, 4), "ratio": round(t / p, 4), "outputs_identical": same,
                "this_spread_ms": [round(min(ts["this"]), 4), round(max(ts["this"]), 4)],
                "parent_spread_ms": [round(min(ts["parent"]), 4), round(max(ts["parent"]), 4)]}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "val_extras_bench_b64_a8400_nc80.json"))
    a = ap.parse_args()
    torch.cuda.set_device(0)
    _C.init(0)
    res = {"card": card(), "torch": torch.__version__, "rounds": a.rounds, "reps": a.reps,
           "nms_priors": nms_priors_case(a.rounds, a.reps), "confusion_matrix": confusion_case(a.rounds, a.reps),
           "validator_batch": validator_case(a.rounds)}
    if a.parent_lib:
        res["nms_stress_ab"] = nms_stress_ab(a.parent_lib, a.rounds, 5)
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text(json.dumps(res, indent=1) + "\n")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
