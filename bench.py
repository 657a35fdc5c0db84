#!/usr/bin/env python
"""bench.py — YOLO11 inference hot path on B200: preprocessed tensor in -> NMS'd detections out.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model n|s|m] [--batch B]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...       (one rank per GPU, weak scaling)

One "step" = one pass of the hot path over one batch of synthetic 640x640 images (BASELINE.json config 3:
yolo11n, bs=64 per GPU, bf16 storage / fp32 accumulate): image ingest (NCHW fp32 -> NHWC bf16), the whole
model as one CUDA-graph replay of this repo's sm_100a kernels, DFL/anchor decode, and batched NMS
(conf=0.25, iou=0.7, max_det=300: the predictor defaults).  Rank 0 prints ONE JSON line.

  value      images/s, inputs resident in HBM, CUDA-event timed on the launching stream, max over ranks
  e2e        images/s through the public API (YOLOLite.predict) from a pinned HOST tensor, H2D + D2H inside
  roofline   dominant kernel (conv_tc_kernel, all its launches of a step): algorithmic bytes / measured time
             vs MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the oracle port of the reference's CPU path (oracle/yolo11_ref.py + oracle/nms_ref.py) timed
             on this box's host cores on a bounded sample

`--impl reference` times that same CPU path alone (the reference is pure Python/ATen, there is nothing to
compile into oracle/_ref; /root/reference does not exist on the GPU box, so the oracle port stands in).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]

CONF, IOU, MAX_DET = 0.25, 0.7, 300
IMG = 640


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="n", choices=["n", "s", "m"])
    ap.add_argument("--batch", type=int, default=64, help="images per GPU per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-latency", action="store_true", help="skip the bs=1 latency measurement")
    ap.add_argument("--no-roofline", action="store_true", help="skip the per-launch timing pass (for ncu launch lists)")
    ap.add_argument("--repeats", type=int, default=5, help="repeat the K-step timed region; value = the median repeat")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the secondary BASELINE configs (yolo11m bs=256 sharded, NMS stress, eager GPU baseline, H2D ceiling)")
    ap.add_argument("--inflight", type=int, default=2,
                    help="batches in flight per GPU (each on its own stream with its own plan buffers)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0's batch) as DIR/*.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


# ------------------------------------------------------------------------------------------------ synthetic
def randomise_model_(model, seed=1):
    """SURVEY §8d: BN gamma~U(.5,1.5), beta,mean~N(0,.1), var~U(.5,1.5); Detect class bias ~N(-4,1.5) so
    scores spread over (0,1) (default bias_init gives ~1e-5 and zero candidates)."""
    g = torch.Generator().manual_seed(seed)
    for name, m in model.named_modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.weight.data.copy_(torch.rand(m.weight.shape, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.bias.shape, generator=g) * 0.1)
            m.running_mean.copy_(torch.randn(m.running_mean.shape, generator=g) * 0.1)
            m.running_var.copy_(torch.rand(m.running_var.shape, generator=g) + 0.5)
    det = model.model[-1]
    for seq in det.cv3:
        seq[-1].bias.data.copy_(torch.randn(seq[-1].bias.shape, generator=g) * 1.5 - 4.0)
    return model


def synth_images(batch, n_sets, seed=0):
    g = torch.Generator().manual_seed(seed)
    return [torch.rand(batch, 3, IMG, IMG, generator=g) for _ in range(n_sets)]


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index, self._mark = [], None, index, 0

    def n_samples(self, since_mark=False):
        return len(self.rows) - (self._mark if since_mark else 0)

    def mark(self):
        """Samples from here on belong to the timed region (+ the identical untimed load that follows it)."""
        self._mark = len(self.rows)

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        rows = self.rows[self._mark:] or self.rows
        sm = [float(r[0]) for r in rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU path
def cpu_reference_step(sd, x):
    """The reference's CPU hot path restated: unfused fp32 forward + non_max_suppression (oracle port)."""
    from oracle import nms_ref, yolo11_ref

    y, _ = yolo11_ref.forward(sd, x)
    return nms_ref.non_max_suppression(y.numpy(), conf_thres=CONF, iou_thres=IOU, max_det=MAX_DET)


def time_cpu(model_sd, batch, reps, warm=1, budget_s=None):
    """Median images/s of the CPU path on `batch`-image steps; with `budget_s` keep repeating (>= reps) until about
    that much CPU wall time has been spent, so the baseline is a 10-30 s sample, not a single cold step.
    Also returns the last step's detections (a list of (n, 6) arrays, one per image)."""
    x = synth_images(batch, 1, seed=0)[0]
    for _ in range(warm):
        cpu_reference_step(model_sd, x)
    ts = []
    t_start = time.perf_counter()
    while len(ts) < reps or (budget_s is not None and time.perf_counter() - t_start < budget_s and len(ts) < 400):
        t0 = time.perf_counter()
        out = cpu_reference_step(model_sd, x)
        ts.append(time.perf_counter() - t0)
    return batch / statistics.median(ts), ts, out


def dump_outputs(out_dir, dets, counts, limit_bytes=64 << 20):
    """Write one step's result as `out_dir`/dets.npy ((B, MAX_DET, 6) float32: x1, y1, x2, y2, conf, class) and
    counts.npy ((B,) float64).  Rows at or past an image's count are not part of the result (the GPU path leaves
    them unwritten), so they are stored as zeros and two builds compare equal exactly when their detections do.
    A batch too large for `limit_bytes` is cut to its first images."""
    keep = max(1, limit_bytes // (MAX_DET * 6 * 4 + 8))
    dets = np.array(dets[:keep], dtype=np.float32)
    counts = np.asarray(counts[:keep], dtype=np.int64)
    dets[np.arange(MAX_DET)[None, :] >= counts[:, None]] = 0
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "dets.npy", dets)
    np.save(out / "counts.npy", counts.astype(np.float64))


def ncu_traffic(kernel, model_name, batch):
    """DRAM bytes per launch of `kernel` (dram__bytes_read.sum + dram__bytes_write.sum) from the committed
    `ncu` capture of this workload (profiles/traffic.json, written by tools/ncu_traffic.py), or None."""
    p = ROOT / "profiles" / "traffic.json"
    if not p.exists():
        return None
    d = json.loads(p.read_text())
    e = d.get(f"{model_name}_bs{batch}", {}).get(kernel)
    return None if e is None else round(e["dram_bytes_per_launch"], 1)


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured"
    return 6650.0, 1400.0, "fallback"


def pin_to_gpu_numa(local):
    """Bind this rank (and therefore the first-touch placement of its pinned host buffers) to the CPU cores NVML
    reports as local to its GPU: with one process per GPU on a multi-socket host, uploads otherwise cross the
    inter-socket link for half of the ranks.  Returns (all_cpus, chosen_cpus) or None when unavailable."""
    try:
        import pynvml

        pynvml.nvmlInit()
        pr = torch.cuda.get_device_properties(local)
        bus = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
        words = (os.cpu_count() + 63) // 64
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, words)
        cpus = {i * 64 + b for i, w in enumerate(mask) for b in range(64) if (w >> b) & 1}
        allc = os.sched_getaffinity(0)
        cpus &= allc
        if cpus and cpus != allc:
            os.sched_setaffinity(0, cpus)
            return allc, cpus
    except Exception:
        pass
    return None



# ------------------------------------------------------------------------------------------------ secondary configs
def bench_yolo11m_sharded(dev, rank, world, dist, ydist, steps=6, warm=3, total=256):
    """BASELINE config 4: yolo11m (random init from the yaml), synthetic 640x640, GLOBAL batch 256 sharded over the ranks
    (strong scaling: 256 / N images per GPU), same step as the headline (ingest + model + decode + batched NMS, two
    batches in flight).  Rank 0 adds the conv kernel's roofline / tensor-pipe fraction from per-launch event timing."""
    from yololite.nn.tasks import DetectionModel

    b = total // world
    torch.manual_seed(0)
    m = randomise_model_(DetectionModel("yolo11m.yaml", verbose=False)).eval().to(dev)
    g = torch.Generator().manual_seed(100 + rank)
    xs = [torch.rand(b, 3, IMG, IMG, generator=g).to(dev) for _ in range(2)]
    lanes = [torch.cuda.Stream(device=dev) for _ in range(2)]

    def run(k):
        main = torch.cuda.current_stream(dev)
        for s_ in lanes:
            s_.wait_stream(main)
        for i in range(k):
            with torch.cuda.stream(lanes[i % 2]):
                out = m.infer_nms(xs[i % 2], CONF, IOU, None, False, False, MAX_DET, slot=i % 2)
        for s_ in lanes:
            main.wait_stream(s_)
        return out

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    run(2 * warm)
    barrier()
    times = []
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        dets, counts = run(steps)
        e1.record()
        barrier()
        times.append(ydist.max_over_ranks(e0.elapsed_time(e1), dev))
    ms = statistics.median(times)
    out = {"value": round(total * steps / (ms / 1e3), 1), "unit": "images/s", "scaling": "strong",
           "global_batch": total, "per_gpu_batch": b, "steps": steps, "warmup": warm, "ms_per_step": round(ms / steps, 4),
           "runs_ms": [round(t, 3) for t in times], "in_flight": 2, "detections_last_step_rank0": int(counts.sum().item()),
           "workload": f"yolo11m synthetic {IMG}x{IMG}, global bs={total} sharded {b}/GPU over {world} GPU(s), predict NMS"}
    if rank == 0:
        nms_key = (float(CONF), float(IOU), None, False, False, int(MAX_DET), 30000, 7680.0)
        plan = m._get_plan(xs[0].shape, dev, False, 0, nms_key)[0]
        lt = plan.time_launches(reps=1, inner=2)
        hbm, tf, _ = peaks()
        tot = {"ms": 0.0, "bytes": 0, "flops": 0, "n": 0}
        all_ms = 0.0
        for md, t in zip(plan.meta, lt):
            all_ms += t
            if md["kind"] == "conv_tc":
                tot["ms"] += t
                tot["bytes"] += md["bytes"]
                tot["flops"] += md["flops"]
                tot["n"] += 1
        out["conv_tc"] = {"launches": tot["n"], "ms": round(tot["ms"], 3), "share_of_step": round(tot["ms"] / all_ms, 3),
                          "achieved_GBps": round(tot["bytes"] / 1e9 / (tot["ms"] / 1e3), 1),
                          "hbm_frac": round(tot["bytes"] / 1e9 / (tot["ms"] / 1e3) / hbm, 4),
                          "tensor_tflops": round(tot["flops"] / 1e12 / (tot["ms"] / 1e3), 1),
                          "tensor_frac": round(tot["flops"] / 1e12 / (tot["ms"] / 1e3) / tf, 4), "tensor_peak_tflops": tf}
    del m, xs
    torch.cuda.empty_cache()
    return out


def bench_nms_stress(dev, B=256, A=8400, nc=80):
    """BASELINE config 5: NMS stress at B=256, A=8400, nc=80, conf=0.001, iou=0.7, max_det=300 (SURVEY 8d inputs: dense =
    every anchor a candidate, multi-label > 30000 pairs -> the max_nms path; sparse = ~2.7 % of anchors), both label
    modes.  Algorithmic bytes = the (B, 84, A) fp32 prediction read once = 722 MB; time = the whole yl_nms_batched call
    (filter + select kernels), CUDA events, median of 5."""
    from yololite import _ops as ops

    hbm = peaks()[0]
    res = {"algorithmic_MB": round(B * (4 + nc) * A * 4 / 1e6, 1), "B": B, "A": A, "nc": nc, "conf": 0.001, "iou": IOU,
           "max_det": MAX_DET, "cases": {}}
    for regime, (mean, std) in (("dense", (-5.0, 2.0)), ("sparse", (-12.0, 1.5))):
        g = torch.Generator(device=dev).manual_seed(2)
        pred = torch.empty((B, 4 + nc, A), device=dev)
        pred[:, 0:2] = torch.rand((B, 2, A), device=dev, generator=g) * 640
        pred[:, 2:4] = torch.rand((B, 2, A), device=dev, generator=g) * 248 + 8
        pred[:, 4:] = torch.sigmoid(torch.randn((B, nc, A), device=dev, generator=g) * std + mean)
        cand = int((pred[:, 4:].amax(1) > 0.001).sum().item())
        for multi in (False, True):
            ts = []
            for i in range(7):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                dets, counts = ops.nms_batched(pred, 0.001, IOU, multi_label=multi, max_det=MAX_DET)
                e1.record()
                torch.cuda.synchronize(dev)
                if i >= 2:
                    ts.append(e0.elapsed_time(e1))
            ms = statistics.median(ts)
            gbs = B * (4 + nc) * A * 4 / 1e9 / (ms / 1e3)
            res["cases"][f"{regime}_{'multi' if multi else 'single'}_label"] = {
                "ms": round(ms, 4), "achieved_GBps": round(gbs, 1), "hbm_frac": round(gbs / hbm, 4),
                "candidate_anchors_per_image": round(cand / B, 1), "detections": int(counts.sum().item())}
        # the filter kernel alone: conf = 1.0 leaves no candidate, so the select kernel has nothing to do
        ts = []
        for i in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ops.nms_batched(pred, 1.0, IOU, max_det=MAX_DET)
            e1.record()
            torch.cuda.synchronize(dev)
            ts.append(e0.elapsed_time(e1))
        ms = statistics.median(ts[1:])
        res["cases"][f"{regime}_filter_only(conf=1)"] = {"ms": round(ms, 4),
                                                         "achieved_GBps": round(B * (4 + nc) * A * 4 / 1e9 / (ms / 1e3), 1),
                                                         "hbm_frac": round(B * (4 + nc) * A * 4 / 1e9 / (ms / 1e3) / hbm, 4)}
        del pred
    torch.cuda.empty_cache()
    return res


def gpu_eager_baseline(local, batch):
    """The honest GPU bar (SURVEY 8d): the same architecture on stock PyTorch eager kernels (ATen / cuDNN conv, BN, SiLU
    unfused like the reference; torchvision CUDA nms per image) on this B200, run in a SUBPROCESS (tools/
    eager_gpu_baseline.py) after all of this repo's measurements, so no library kernel ever runs in the bench process."""
    env = dict(os.environ)
    vis = env.get("CUDA_VISIBLE_DEVICES")
    env["CUDA_VISIBLE_DEVICES"] = (vis.split(",")[local] if vis else str(local))
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, str(ROOT / "tools" / "eager_gpu_baseline.py"), str(batch)], env=env,
                           capture_output=True, text=True, timeout=240)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        if r.returncode != 0 or not line:
            return {"unavailable": (r.stderr or r.stdout)[-300:]}
        d = json.loads(line[-1])
        d["what"] = ("reference architecture on stock PyTorch eager + cuDNN + torchvision CUDA nms on this GPU (subprocess); "
                     "a reported GPU baseline, none of this repo's kernels")
        return d
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"}


# ------------------------------------------------------------------------------------------------ main
def main():
    a = parse()
    # the contract is ONE JSON line on stdout: park the real stdout and send everything else that writes to fd 1
    # (NCCL's version banner, library chatter) to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    rank = int(os.environ.get("RANK", 0))
    local = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    model_name = f"yolo11{a.model}"
    workload = f"{model_name} synthetic {IMG}x{IMG} bs={a.batch}/GPU, predict NMS conf={CONF} iou={IOU} max_det={MAX_DET}"

    from yololite.nn.tasks import DetectionModel

    torch.manual_seed(0)
    model = randomise_model_(DetectionModel(f"{model_name}.yaml", verbose=False)).eval()
    n_sets = 3                                              # rotate inputs: 3 x 315 MB >> 126 MB L2
    # identical in both arms (the driver compares it): what is computed, on which inputs, with which weights
    config = {"workload": workload, "global_batch": a.batch * max(world, a.gpus if a.impl == "reference" else 1),
              "inputs": f"synthetic torch.rand images; {n_sets} rotating batches of {a.batch * 3 * IMG * IMG * 4 / 1e6:.0f} MB "
                        f"per GPU (> the 126 MB L2), so no timed step finds its input in cache",
              "weights": "random init from cfg/yolo11.yaml, BN statistics randomised (seed 1)"}

    if a.impl == "reference":
        if rank != 0:
            return
        threads = max(1, min(os.cpu_count() or 1, 64))
        torch.set_num_threads(threads)
        sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
        sample_b = 8
        t_probe0 = time.perf_counter()
        cpu_reference_step(sd, synth_images(sample_b, 1)[0])
        probe = time.perf_counter() - t_probe0
        steps = a.steps
        warm = min(a.warmup, max(0, int(20.0 / max(probe, 1e-3))))
        v, ts, last = time_cpu(sd, sample_b, steps, warm)
        if a.dump_outputs:
            dets = np.zeros((sample_b, MAX_DET, 6), np.float32)
            for i, d in enumerate(last):
                dets[i, :len(d)] = d
            dump_outputs(a.dump_outputs, dets, [len(d) for d in last])
        line = {
            "impl": "reference", "metric": "images_per_sec", "value": round(v, 3), "unit": "images/s",
            "n_gpus": a.gpus, "steps": steps, "warmup": warm, "ms_per_step": round(statistics.median(ts) * 1e3, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config,
            "cpu_baseline": {"value": round(v, 3), "unit": "images/s", "cores": threads, "kind": "port",
                             "sample": f"oracle port (yolo11_ref fp32 unfused + nms_ref), {sample_b}-image steps x{steps}"},
            "e2e": {"value": round(v, 3), "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        }
        emit(line)
        return

    # ---------------------------------------------------------------- ours
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the B200 path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = pin_to_gpu_numa(local) if world > 1 else None
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from yololite import _C
    from yololite.utils import dist as ydist
    from yololite.utils import ops

    _C.init(dev)
    sd_cpu = {k: v.detach().clone() for k, v in model.state_dict().items()}
    model = model.to(dev)
    host = [t.pin_memory() for t in synth_images(a.batch, n_sets, seed=rank)]
    devx = [t.to(dev) for t in host]

    n_fly = max(1, a.inflight)
    lanes = [torch.cuda.Stream(device=dev) for _ in range(n_fly)]

    def step(x, slot=0):
        # ingest + ONE graph launch: the whole model and the batched NMS are recorded in the same plan
        return model.infer_nms(x, CONF, IOU, None, False, False, MAX_DET, slot=slot)

    def run_steps(k, fly):
        """k steps with `fly` batches in flight: step i runs on lane i % fly (own stream, own plan slot), so the
        small latency-bound layers of one batch overlap the large layers of the other.  fly == 1 is strictly
        serial on the current stream."""
        if fly == 1:
            for i in range(k):
                out = step(devx[i % n_sets], 0)
            return out
        main = torch.cuda.current_stream(dev)
        for s_ in lanes[:fly]:
            s_.wait_stream(main)
        for i in range(k):
            with torch.cuda.stream(lanes[i % fly]):
                out = step(devx[i % n_sets], i % fly)
        for s_ in lanes[:fly]:
            main.wait_stream(s_)
        return out

    for fly in sorted({1, n_fly}):
        dets, counts = run_steps(max(a.warmup, 3) * fly, fly)
    torch.cuda.synchronize(dev)
    nms_key = (float(CONF), float(IOU), None, False, False, int(MAX_DET), 30000, 7680.0)
    plan = model._get_plan(devx[0].shape, dev, False, 0, nms_key)[0]
    launches_per_step = plan.n_launches + 1                 # the NMS entry launches two kernels (filter + select)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(k, fly):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        out = run_steps(k, fly)
        e1.record()
        barrier()
        return ydist.max_over_ranks(e0.elapsed_time(e1), dev), out

    # ---- timed region: K steps, CUDA events on the launching (current) stream, max over ranks
    # nvidia-smi needs a few hundred ms to deliver its first sample and the K timed steps may last only ~60 ms, so the
    # sampler is started under load BEFORE the timed region and keeps sampling through it and through the serial
    # re-measurement; every sample it reports was taken while this workload was running on the GPU.
    with ClockSampler(local) as clk:
        t_wait = time.perf_counter()
        while clk.n_samples() < 2 and time.perf_counter() - t_wait < 3.0:      # untimed load until the sampler is live
            run_steps(10, n_fly)
            torch.cuda.synchronize(dev)
        clk.mark()
        rep_ms = []
        for _ in range(max(1, a.repeats)):
            ms_r, (dets, counts) = timed(a.steps, n_fly)
            rep_ms.append(ms_r)
        if a.dump_outputs and rank == 0:
            # the returned tensors alias plan buffers that the steps below overwrite: copy the last timed step now
            dump_outputs(a.dump_outputs, dets.cpu().numpy(), counts.cpu().numpy())
        ms_max = statistics.median(rep_ms)
        ms_serial = ms_max
        if n_fly > 1:
            ms_serial = statistics.median([timed(a.steps, 1)[0] for _ in range(min(3, max(1, a.repeats)))])
        t_wait = time.perf_counter()
        while clk.n_samples(since_mark=True) < 10 and time.perf_counter() - t_wait < 2.0:   # same load, untimed
            run_steps(10, n_fly)
            torch.cuda.synchronize(dev)
    n_det_local = int(counts.sum().item())

    # ---- bs=1 latency (BASELINE metric: "bs1 p50 latency"): ingest + model + NMS + counts on the host
    lat = None
    if rank == 0 and not a.no_latency:
        x1 = devx[0][:1].contiguous()
        for _ in range(10):
            step(x1)[1].tolist()
        ts = []
        for i in range(200):
            torch.cuda.synchronize(dev)
            t0 = time.perf_counter()
            step(x1)[1].tolist()                            # host has the detection count = result delivered
            ts.append((time.perf_counter() - t0) * 1e3)
        ts.sort()
        lat = {"p50": round(ts[len(ts) // 2], 4), "p90": round(ts[int(len(ts) * 0.9)], 4), "min": round(ts[0], 4),
               "unit": "ms", "what": f"{model_name} bs=1 640x640 device-resident input -> NMS'd count on host, 200 reps"}

    # ---- e2e through the public API, host tensors, H2D + D2H inside the timed region
    e2e = e2e_half = e2e_u8 = h2d_ceiling = None
    if not a.no_e2e:
        from yololite import YOLOLite

        yl = YOLOLite(f"{model_name}.yaml")
        yl.model.load_state_dict(sd_cpu)
        yl.model.to(dev)
        kw = dict(conf=CONF, iou=IOU, max_det=MAX_DET, verbose=False, device=dev, batch=a.batch)
        steps_e = max(3, min(a.steps, 20))

        def read_all(res):
            """Device->host read of EVERY image's detections of a step: one batched copy of the padded (B, 300, 6)
            detections + the (B,) counts (Results.batch.host()); returns the detection count and the bytes moved."""
            d, c = res[0].batch.host()
            return int(c.sum()), d.nbytes + c.nbytes

        def e2e_run(host_batches, label):
            for i in range(max(3, steps_e // 2)):              # warm-up: plan build, pinned pages, copy-engine queues
                read_all(yl.predict(host_batches[i % n_sets], **kw))
            best = None
            for _ in range(5):                                  # 5 x steps_e steps; the median run is reported
                barrier()
                t0 = time.perf_counter()
                nd, d2h = 0, 0
                prev = None
                for i in range(steps_e):
                    res = yl.predict(host_batches[i % n_sets], **kw)   # asynchronous: upload + kernels only enqueued
                    if prev is not None:
                        n_, b_ = read_all(prev)                 # D2H of the PREVIOUS step's results (all B images)
                        nd += n_
                        d2h = b_
                    prev = res
                n_, d2h = read_all(prev)
                nd += n_
                barrier()
                dt = ydist.max_over_ranks(time.perf_counter() - t0, dev)
                best = (best or []) + [dt]
            dt = statistics.median(best)
            hb = host_batches[0]
            return {"value": round(a.batch * world * steps_e / dt, 1), "unit": "images/s",
                    "h2d_bytes_per_step": hb.numel() * hb.element_size(), "d2h_bytes_per_step": d2h, "steps": steps_e,
                    "runs_s": [round(t, 4) for t in best], "input": label, "detections": nd,
                    "api": "YOLOLite.predict(pinned host BCHW tensor); EVERY image's detections of every step are read on the "
                           "host (one batched D2H of dets + counts), one step behind the upload of the next batch "
                           "(predict() is asynchronous, Results resolve lazily)"}

        e2e = e2e_run(host, "pinned host fp32 BCHW tensor in [0, 1] (the reference arm's input)")
        # secondary: the same API fed narrower host tensors — fp16 (the reference accepts it: `.float()` on the device,
        # predictor.py:83) and uint8 image bytes (/255 on the device inside the fused stem; the reference's own uint8
        # route is the numpy-image path, predictor.py:76-84): 2x / 4x fewer PCIe bytes, so the link stops being the bound
        host_h = [t.half().pin_memory() for t in host]
        e2e_half = e2e_run(host_h, "pinned host fp16 BCHW tensor")
        del host_h
        host_u8 = [(t * 255).round().to(torch.uint8).pin_memory() for t in host]
        e2e_u8 = e2e_run(host_u8, "pinned host uint8 BCHW tensor (image bytes, /255 on the device)")
        del host_u8

        # ---- the box's pinned host->device ceiling at this rank count: the same bytes per step as the fp32 e2e, plain
        # cudaMemcpyAsync on one stream per GPU, all ranks at once (max over ranks)
        if not a.no_extras:
            dst = torch.empty_like(devx[0])
            cs = torch.cuda.Stream(device=dev)
            with torch.cuda.stream(cs):
                for i in range(3):
                    dst.copy_(host[i % n_sets], non_blocking=True)
            cs.synchronize()
            barrier()
            t0 = time.perf_counter()
            with torch.cuda.stream(cs):
                for i in range(steps_e):
                    dst.copy_(host[i % n_sets], non_blocking=True)
            cs.synchronize()
            dt = ydist.max_over_ranks(time.perf_counter() - t0, dev)
            gbs = world * steps_e * dst.numel() * 4 / dt / 1e9
            h2d_ceiling = {"aggregate_GBps": round(gbs, 1), "per_gpu_GBps": round(gbs / world, 1),
                           "images_per_s_fp32": round(gbs * 1e9 / (3 * IMG * IMG * 4), 1),
                           "e2e_frac_of_ceiling": round(e2e["value"] / (gbs * 1e9 / (3 * IMG * IMG * 4)), 3),
                           "what": f"pinned host -> device cudaMemcpyAsync of {dst.numel() * 4 / 1e6:.0f} MB batches, one stream per "
                                   f"GPU, {world} rank(s) concurrently, wall clock max over ranks"}
            del dst

    # ---- image preprocess (SURVEY §8f rank 1): uint8 HWC BGR images -> letterboxed fp32 NCHW batch on the GPU
    prep = None
    if rank == 0 and not a.no_e2e:
        from yololite.data import letterbox_batch_cuda
        from yololite.data.augment import _Staging

        rng = np.random.default_rng(0)
        imgs = [rng.integers(0, 256, (1080, 810, 3), dtype=np.uint8) for _ in range(a.batch)]
        stg = _Staging()
        out = letterbox_batch_cuda(imgs, (IMG, IMG), auto=True, stride=32, device=dev, staging=stg)
        torch.cuda.synchronize(dev)
        from yololite import _C as _c

        descs_dev = stg.dev                                   # descriptors + pixels are already resident
        ek0, ek1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 20
        ek0.record()
        for _ in range(reps):
            _c.check(_c.load().yl_letterbox_u8(descs_dev.data_ptr(), a.batch, out.data_ptr(), out.shape[2], out.shape[3],
                                               114, _c.stream_ptr()), "yl_letterbox_u8")
        ek1.record()
        torch.cuda.synchronize(dev)
        k_ms = ek0.elapsed_time(ek1) / reps
        byts = a.batch * (1080 * 810 * 3 + out.shape[1] * out.shape[2] * out.shape[3] * 4)
        t0 = time.perf_counter()
        for _ in range(3):
            letterbox_batch_cuda(imgs, (IMG, IMG), auto=True, stride=32, device=dev, staging=stg, out=out)
        torch.cuda.synchronize(dev)
        host_ms = (time.perf_counter() - t0) / 3 * 1e3
        hbm_pk = peaks()[0]
        prep = {"kernel": "letterbox_u8", "workload": f"{a.batch} x 1080x810 BGR uint8 -> {tuple(out.shape)} fp32",
                "kernel_ms": round(k_ms, 4), "kernel_images_per_s": round(a.batch / k_ms * 1e3, 1),
                "algorithmic_GBps": round(byts / 1e9 / (k_ms / 1e3), 1), "hbm_frac": round(byts / 1e9 / (k_ms / 1e3) / hbm_pk, 4),
                "from_host_ms": round(host_ms, 3), "from_host_images_per_s": round(a.batch / host_ms * 1e3, 1),
                "h2d_bytes": a.batch * 1080 * 810 * 3,
                "note": "from_host = pinned pack + one H2D + kernel (host memcpy bound)"}
        del imgs, out

    # ---- roofline of the dominant kernel (rank 0): per-launch CUDA-event times of one eager pass
    roof, breakdown = None, None
    if rank == 0 and not a.no_roofline:
        step(devx[0])
        torch.cuda.synchronize(dev)
        lt = plan.time_launches(reps=3)
        kinds = {}
        for m_, t_ in zip(plan.meta, lt):
            k = kinds.setdefault(m_["kind"], {"ms": 0.0, "bytes": 0, "flops": 0, "launches": 0})
            k["ms"] += t_
            k["bytes"] += m_["bytes"]
            k["flops"] += m_["flops"]
            k["launches"] += 1
        total_ms = sum(k["ms"] for k in kinds.values())
        breakdown = {k: {"ms": round(v["ms"], 4), "share": round(v["ms"] / total_ms, 3), "launches": v["launches"],
                         "GB": round(v["bytes"] / 1e9, 4), "GFLOP": round(v["flops"] / 1e9, 2)}
                     for k, v in sorted(kinds.items(), key=lambda kv: -kv[1]["ms"])}
        hbm, tf, src = peaks()
        top = max(kinds.items(), key=lambda kv: kv[1]["ms"])[0]
        tk = kinds[top]
        ach = tk["bytes"] / 1e9 / (tk["ms"] / 1e3)
        roof = {"kernel": top, "bound": "hbm", "achieved": round(ach, 1), "peak": hbm, "unit": "GB/s",
                "frac": round(ach / hbm, 4), "traffic": ncu_traffic(top, model_name, a.batch),
                "algorithmic_bytes_per_launch": round(tk["bytes"] / tk["launches"], 1),
                "peak_source": f"MEASURED_PEAKS.json ({src})",
                "timing": "CUDA events around 4 back-to-back launches of every plan launch (eager pass in plan order), /4",
                "launches_per_step": tk["launches"], "avg_launch_us": round(tk["ms"] * 1e3 / tk["launches"], 2),
                "tensor_tflops": round(tk["flops"] / 1e12 / (tk["ms"] / 1e3), 1), "tensor_peak_tflops": tf,
                "tensor_frac": round(tk["flops"] / 1e12 / (tk["ms"] / 1e3) / tf, 4)}

    # ---- detections gathered for the metric only (no collective on the hot path)
    gd, gc = ydist.gather_detections(dets, counts, total=a.batch * world)     # (B*world, 300, 6) + counts: 7.2 KB/img
    n_det = int(gc.sum().item())
    assert n_det == ydist.sum_over_ranks(n_det_local, dev)

    # ---- the other BASELINE configs, after every headline measurement (they free the headline's buffers first)
    m256 = nms_stress = eager = None
    if not a.no_extras:
        if not a.no_e2e:
            del yl
        for k_ in [k_ for k_ in model.__dict__ if k_.startswith("_yl_")]:
            del model.__dict__[k_]
        del devx, host
        torch.cuda.synchronize(dev)
        torch.cuda.empty_cache()
        # a failure in a secondary config must not cost the headline line (collectives inside m256 stay matched: every
        # rank runs the same code and an exception there is a bug on all of them)
        try:
            m256 = bench_yolo11m_sharded(dev, rank, world, dist, ydist)
        except Exception as e:  # noqa: BLE001
            m256 = {"error": f"{type(e).__name__}: {e}"[:300]}
        if rank == 0:
            try:
                nms_stress = bench_nms_stress(dev)
            except Exception as e:  # noqa: BLE001
                nms_stress = {"error": f"{type(e).__name__}: {e}"[:300]}
        if dist is not None:
            dist.barrier()
        if rank == 0:
            eager = gpu_eager_baseline(local, a.batch)

    cpu_b = None
    if rank == 0 and not a.no_cpu_baseline:
        if numa is not None:
            os.sched_setaffinity(0, numa[0])            # the CPU baseline may use every host core again
        threads = max(1, min(os.cpu_count() or 1, 64))
        torch.set_num_threads(threads)
        v, ts, _ = time_cpu(sd_cpu, 8, reps=3, warm=1, budget_s=12.0)
        cpu_b = {"value": round(v, 3), "unit": "images/s", "cores": threads, "kind": "port",
                 "sample": f"oracle port (yolo11_ref fp32 unfused + nms_ref), 8-image steps of the bs={a.batch} "
                           f"workload x{len(ts)} reps, {sum(ts):.1f}s CPU wall, median step"}

    if rank == 0:
        total_images = a.batch * world * a.steps
        line = {
            "metric": "images_per_sec", "value": round(total_images / (ms_max / 1e3), 1), "unit": "images/s",
            "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": round(ms_max / a.steps, 4),
            "in_flight": n_fly, "value_serial": round(total_images / (ms_serial / 1e3), 1),
            "bs1_latency_ms": lat,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": config,
            "run": {"parallelism": f"dp{world} batch-sharded, no collective",
                    "cpu_affinity": (f"rank bound to the {len(numa[1])} cores NVML reports local to its GPU" if numa else "default"),
                    "in_flight": f"{n_fly} batches in flight per GPU (one stream + one plan slot each)"},
            "repeats": {"n": len(rep_ms), "ms_per_step_median": round(ms_max / a.steps, 4),
                        "ms_per_step_min": round(min(rep_ms) / a.steps, 4), "ms_per_step_max": round(max(rep_ms) / a.steps, 4)},
            "clocks": clk.summary(), "e2e": e2e, "e2e_fp16_input": e2e_half, "e2e_u8_input": e2e_u8,
            "h2d_ceiling": h2d_ceiling, "yolo11m_bs256": m256, "nms_stress": nms_stress, "gpu_eager_baseline": eager,
            "gpu_launches": launches_per_step * a.steps,
            "launches_per_step": launches_per_step, "detections_last_step": n_det,
            "roofline": roof, "preprocess": prep, "cpu_baseline": cpu_b, "kernel_breakdown": breakdown,
        }
        emit(line)
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
