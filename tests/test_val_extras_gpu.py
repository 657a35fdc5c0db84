"""Validator switches `save_hybrid=True` and `plots=True` on the GPU: NMS with ground-truth priors
(`yl_nms_batched_priors`) bit-exact against oracle/val_extras_ref.py, the confusion kernel (`yl_confusion_matrix`)
equal to its `ConfusionMatrix` as integer counts, and both switches through DetectionValidator / YOLOLite.val."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]

from oracle import metrics_ref, nms_ref, val_extras_ref  # noqa: E402

pytestmark = pytest.mark.gpu


def _seeded_pred(seed, B, nc, A, dense=False):
    """(B, 4+nc, A) prediction on a 1/64 grid; `dense`: many near-identical boxes with saturated scores."""
    g = np.random.default_rng(seed)
    p = np.zeros((B, 4 + nc, A), np.float32)
    p[:, 0:2] = g.integers(0, 600 * 64, (B, 2, A)) / 64.0
    p[:, 2:4] = g.integers(4 * 64, 120 * 64, (B, 2, A)) / 64.0
    p[:, 4:] = g.random((B, nc, A)).astype(np.float32) ** 6
    if dense:
        p[:, 0:2] = 300 + g.integers(0, 64, (B, 2, A)) / 64.0
        p[:, 4 + 3, : A // 2] = 1.0
    return p


def _seeded_labels(seed, B, nc, counts, pred=None):
    """B arrays (n, 5) [cls, cx, cy, w, h]; with `pred`, label 0 of each image copies anchor 5's box and its class
    gets score 1.0 there, so anchor and prior tie at 1.0 on the same box."""
    g = np.random.default_rng(seed + 1000)
    out = []
    for b, n in enumerate(counts):
        lb = np.zeros((n, 5), np.float32)
        lb[:, 0] = g.integers(0, nc, n)
        lb[:, 1:3] = g.integers(0, 600 * 64, (n, 2)) / 64.0
        lb[:, 3:5] = g.integers(4 * 64, 120 * 64, (n, 2)) / 64.0
        if pred is not None and n:
            lb[0, 1:5] = pred[b, :4, 5]
            pred[b, 4 + int(lb[0, 0]), 5] = 1.0
        out.append(lb)
    return out


def _check(pred, labels, **kw):
    from yololite.utils import ops

    got = ops.non_max_suppression(torch.from_numpy(pred).cuda(), labels=[torch.from_numpy(lb) for lb in labels], **kw)
    want = val_extras_ref.non_max_suppression(pred, labels=labels, **kw)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a.cpu().numpy(), b)
    return want


KW = [
    dict(conf_thres=0.5, iou_thres=0.45),                                              # class-wise select path
    dict(conf_thres=0.001, iou_thres=0.7, multi_label=True),                           # validator settings
    dict(conf_thres=0.1, iou_thres=0.5, multi_label=True, classes=[0, 3, 7]),
    dict(conf_thres=0.25, iou_thres=0.45, agnostic=True),                              # general select path
    dict(conf_thres=0.05, iou_thres=0.6, multi_label=True, max_det=7),                 # max_det < candidates
]


@pytest.mark.parametrize("kw", KW)
def test_nms_priors_bitexact(kw):
    B, nc, A = 5, 10, 2000
    pred = _seeded_pred(1, B, nc, A)
    labels = _seeded_labels(1, B, nc, [0, 1, 20, 300, 0], pred=pred)
    want = _check(pred, labels, **kw)
    if "classes" not in kw:
        assert (want[3][:, 4] == 1.0).sum() > 0          # priors reached the output


@pytest.mark.parametrize("multi_label", [False, True])
def test_nms_priors_dense_max_nms_cut(multi_label):
    """The max_nms top-k cut falls among score-1.0 rows: anchors first, then the priors in label order."""
    B, nc, A = 3, 8, 4000
    pred = _seeded_pred(2, B, nc, A, dense=True)
    labels = _seeded_labels(2, B, nc, [50, 0, 700])
    for b in range(B):
        labels[b][:, 1:3] = 300 + np.float32(labels[b][:, 1:3] % 1)
    for max_nms in (1000, 2500):
        _check(pred, labels, conf_thres=0.2, iou_thres=0.9, multi_label=multi_label, max_nms=max_nms, max_det=300)
        _check(pred, labels, conf_thres=0.2, iou_thres=0.9, multi_label=multi_label, max_nms=max_nms, max_det=300,
               agnostic=True)


def test_nms_priors_only_candidates():
    pred = np.zeros((2, 4 + 3, 64), np.float32)
    pred[:, :4] = 10
    labels = [np.array([[1, 50, 50, 20, 20], [2, 300, 300, 10, 10]], np.float32), np.zeros((0, 5), np.float32)]
    want = _check(pred, labels, conf_thres=0.25, iou_thres=0.45)
    assert len(want[0]) == 2 and len(want[1]) == 0


def test_no_labels_is_bit_identical_to_yl_nms_batched():
    from yololite import _C, _ops
    from yololite.utils import ops

    B, nc, A = 4, 80, 8400
    pred = torch.from_numpy(_seeded_pred(3, B, nc, A)).cuda()
    lib = _C.init(pred.device)
    for ml in (0, 1):
        ws = torch.empty(lib.yl_nms_workspace_bytes(B, A, nc, ml), dtype=torch.uint8, device="cuda")
        out = torch.zeros((B, 300, 6), device="cuda")
        cnt = torch.zeros((B,), dtype=torch.int32, device="cuda")
        _C.check(lib.yl_nms_batched(pred.data_ptr(), B, nc, A, 0.001, 0.7, None, 0, 0, ml, 300, 30000, 7680.0,
                                    ws.data_ptr(), ws.numel(), out.data_ptr(), cnt.data_ptr(), _C.stream_ptr()))
        assert lib.yl_nms_priors_workspace_bytes(B, A, nc, ml, 0) == ws.numel()
        for labels in (None, ops.pack_priors([torch.zeros((0, 5))] * B)):
            d, c = ops.nms_padded(pred, 0.001, 0.7, multi_label=bool(ml), labels=labels)
            assert torch.equal(c, cnt)
            assert torch.equal(d, out)
        d, c = _ops.nms_batched(pred, 0.001, 0.7, multi_label=bool(ml))
        assert torch.equal(c, cnt) and torch.equal(d, out)


def test_prior_class_out_of_range_on_device():
    from yololite.utils import ops

    pred = torch.zeros((1, 7, 16), device="cuda")
    with pytest.raises(ValueError, match="outside"):
        ops.non_max_suppression(pred, labels=[torch.tensor([[3.0, 5, 5, 2, 2]], device="cuda")])


# ------------------------------------------------------------------------------------------------ confusion kernel
def _cm_gpu(nc, dets, counts, gtb, gtc, offs, conf=0.001):
    from yololite.utils.metrics import ConfusionMatrix

    cm = ConfusionMatrix(nc, conf)
    cm.process_batched(torch.from_numpy(dets).cuda(), torch.from_numpy(counts).cuda(), torch.from_numpy(gtb),
                       torch.from_numpy(gtc), list(offs))
    return cm


def _seeded_conf(dets, counts, seed):
    g = np.random.default_rng(seed)
    for b in range(dets.shape[0]):
        dets[b, : counts[b], 4] = np.sort(g.random(counts[b]).astype(np.float32))[::-1]
    return dets


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_confusion_kernel_equals_oracle(seed):
    from oracle.gen_golden import val_case

    dets, counts, gtb, gtc, offs = val_case(100 + seed, B=64, max_det=300, nc=80)
    dets = _seeded_conf(dets, counts, seed)
    want = val_extras_ref.batch_confusion(val_extras_ref.ConfusionMatrix(80, 0.001), dets, counts, gtb, gtc, offs).matrix
    assert (np.diff(offs) == 0).any() and (counts == 0).any()
    got = _cm_gpu(80, dets, counts, gtb, gtc, offs)
    np.testing.assert_array_equal(got.matrix, want)
    assert want.sum() > 0 and want[:80, :80].trace() > 0
    tp, fp = got.tp_fp()
    assert tp.shape == fp.shape == (80,)


def test_confusion_kernel_tie_rule():
    # identical labels and detections: label 0 pairs with detection 0 (lower indices win the exact ties)
    dets = np.zeros((1, 4, 6), np.float32)
    dets[0, :3] = [[0, 0, 10, 10, 0.9, 1], [0, 0, 10, 10, 0.8, 2], [0, 0, 20, 10, 0.7, 0]]
    gtb = np.float32([[0, 0, 10, 10], [0, 0, 10, 10], [0, 0, 9, 10]])   # label 2: IoU exactly 0.45 with det 2
    gtc = np.float32([0, 2, 0])
    counts = np.int32([3])
    want = val_extras_ref.batch_confusion(val_extras_ref.ConfusionMatrix(3, 0.25), dets, counts, gtb, gtc, [0, 3]).matrix
    got = _cm_gpu(3, dets, counts, gtb, gtc, [0, 3], conf=0.25).matrix
    np.testing.assert_array_equal(got, want)
    assert got[1, 0] == 1 and got[3, 2] == 1 and got[2, 3] == 1 and got[3, 0] == 1 and got[0, 3] == 1


def test_confusion_kernel_on_coco8(golden):
    """The reference's own native-space predictions of the coco8 rect batch against its labels."""
    from yololite.engine.validator import DetectionValidator

    real = golden("real_images.npz")
    counts = real["coco8.nms_counts"].astype(np.int32)
    off = np.concatenate([[0], np.cumsum(counts)])
    dets = np.zeros((4, 300, 6), np.float32)
    for i in range(4):
        dets[i, : counts[i]] = real["coco8.predn"][off[i]:off[i + 1]]
    batch = {"img": torch.empty(tuple(int(v) for v in real["coco8.img_shape"])),
             "cls": torch.from_numpy(real["coco8.cls"]), "bboxes": torch.from_numpy(real["coco8.bboxes"]),
             "batch_idx": torch.from_numpy(real["coco8.batch_idx"]),
             "ori_shape": [tuple(int(v) for v in s) for s in real["coco8.ori_shape"]],
             "ratio_pad": [(tuple(r), tuple(p)) for r, p in zip(real["coco8.ratio"], real["coco8.pad"])]}
    v = DetectionValidator(dataloader=[])
    v.device = torch.device("cuda", 0)
    for k in ("cls", "bboxes", "batch_idx"):
        batch[k] = batch[k].cuda()
    gtb, gtc, offs = v._labels_native(batch)
    gtb, gtc = gtb.cpu().numpy(), gtc.cpu().numpy()
    want = val_extras_ref.batch_confusion(val_extras_ref.ConfusionMatrix(80, 0.001), dets, counts, gtb, gtc, offs).matrix
    got = _cm_gpu(80, dets, counts, gtb, gtc, offs)
    np.testing.assert_array_equal(got.matrix, want)
    assert want.sum() >= len(gtc)


# ------------------------------------------------------------------------------------------------ validator
def _model_and_batches():
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    batches = []
    for k in range(2):
        x = torch.rand(4, 3, 64, 64, generator=torch.Generator().manual_seed(k))
        res = yl.predict(x, imgsz=64, conf=0.05, iou=0.5, verbose=False, device=0)
        cls, boxes, bidx = [], [], []
        for i, r in enumerate(res):
            b = r.boxes.data.cpu()[: 2 + 2 * i]
            if len(b) and i != 1:                          # image 1 has no labels
                xyxy = b[:, :4]
                xywh = torch.stack([(xyxy[:, 0] + xyxy[:, 2]) / 2, (xyxy[:, 1] + xyxy[:, 3]) / 2,
                                    xyxy[:, 2] - xyxy[:, 0], xyxy[:, 3] - xyxy[:, 1]], 1) / 64.0
                # shrunk about the detection's centre, by a different factor per label: every label lies inside the
                # image (nothing clips two labels onto one box) and no IoU ties exactly, so the matching tie order,
                # which the reference leaves to np.argsort, never decides a result
                xywh[:, 2:] *= (0.85 - 0.07 * torch.arange(len(b), dtype=torch.float32))[:, None]
                cls.append((b[:, 5:6] + i) % 80)
                boxes.append(xywh)
                bidx.append(torch.full((len(b),), float(i)))
        perm = torch.randperm(len(torch.cat(bidx)), generator=torch.Generator().manual_seed(k))   # image-interleaved
        batches.append({"img": x, "cls": torch.cat(cls)[perm], "bboxes": torch.cat(boxes)[perm],
                        "batch_idx": torch.cat(bidx)[perm], "ori_shape": [(64, 64)] * 4, "ratio_pad": [None] * 4,
                        "im_file": [f"im{i}.jpg" for i in range(4)]})
    return yl, batches


def _fresh(batches):
    return [dict(b) for b in batches]


def _recording_validator(args, batches):
    from yololite.engine.validator import DetectionValidator

    class Rec(DetectionValidator):
        seen_preds = []

        def postprocess(self, preds):
            self.seen_preds.append(preds.clone())
            return super().postprocess(preds)

    v = Rec(dataloader=_fresh(batches), args=args)
    v.seen_preds = []
    return v


def _oracle_pipeline(preds, batches, conf, iou, save_hybrid, cm=None):
    """oracle NMS (with priors) -> identity rescale + clip to 64 x 64 -> match_predictions -> ap_per_class."""
    from yololite.utils.metrics import DetMetrics

    iouv = np.linspace(0.5, 0.95, 10).astype(np.float32)
    stats = dict(tp=[], conf=[], pred_cls=[], target_cls=[])
    for y, batch in zip(preds, batches):
        bi = batch["batch_idx"].long()
        order = torch.argsort(bi, stable=True)
        cls = batch["cls"].view(-1)[order].numpy()
        xywh = batch["bboxes"].view(-1, 4)[order]
        offs = [0] + torch.cumsum(torch.bincount(bi, minlength=4), 0).tolist()
        labels = ()
        if save_hybrid:
            px = (xywh * torch.tensor((64, 64, 64, 64))).numpy()
            labels = [np.concatenate([cls[offs[i]:offs[i + 1], None], px[offs[i]:offs[i + 1]]], 1) for i in range(4)]
        out = val_extras_ref.non_max_suppression(y.cpu().numpy(), conf, iou, multi_label=True, labels=labels, max_det=300)
        gtb = np.clip(nms_ref.xywh2xyxy(xywh.numpy()) * np.float32(64), 0, 64)   # scale_boxes' clip_boxes
        for i in range(4):
            d = out[i].copy()
            d[:, :4] = np.clip(d[:, :4], 0, 64)
            s, e = offs[i], offs[i + 1]
            if cm is not None and (len(d) or e > s):
                cm.process_batch(d if len(d) else None, gtb[s:e], cls[s:e])
            if not len(d) and e == s:
                continue
            tp = np.zeros((len(d), 10), bool)
            if len(d) and e > s:
                tp = metrics_ref.match_predictions(d[:, 5], cls[s:e], metrics_ref.box_iou(gtb[s:e], d[:, :4]), iouv)
            stats["tp"].append(tp)
            stats["conf"].append(d[:, 4])
            stats["pred_cls"].append(d[:, 5])
            stats["target_cls"].append(cls[s:e])
    st = {k: np.concatenate(v, 0) for k, v in stats.items()}
    m = DetMetrics(names={i: str(i) for i in range(80)})
    m.process(**st)
    return m.results_dict


@pytest.mark.parametrize("save_hybrid", [False, True])
def test_validator_stats_equal_oracle_pipeline(save_hybrid):
    yl, batches = _model_and_batches()
    args = dict(conf=0.001, iou=0.7, device=0, verbose=False, save_hybrid=save_hybrid, plots=True)
    v = _recording_validator(args, batches)
    got = v(model=yl.model)
    cm = val_extras_ref.ConfusionMatrix(80, 0.001)
    want = _oracle_pipeline(v.seen_preds, batches, 0.001, 0.7, save_hybrid, cm)
    assert got == pytest.approx(want, abs=1e-12), (got, want)
    np.testing.assert_array_equal(v.metrics.confusion_matrix.matrix, cm.matrix)
    assert v.confusion_matrix is v.metrics.confusion_matrix and cm.matrix.sum() > 0


def test_val_plots_off_changes_nothing():
    yl, batches = _model_and_batches()
    m_on = yl.val(dataloader=_fresh(batches), conf=0.001, iou=0.7, device=0, verbose=False, plots=True)
    d_on, cm = m_on.results_dict, m_on.confusion_matrix
    assert cm.matrix.shape == (81, 81) and cm.matrix.dtype == np.float64 and cm.matrix.sum() > 0
    m_off = yl.val(dataloader=_fresh(batches), conf=0.001, iou=0.7, device=0, verbose=False)
    assert m_off.results_dict == d_on and m_off.confusion_matrix is None


def test_val_switches_with_augment_and_ensemble():
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite
    from yololite.nn.tasks import DetectionModel, Ensemble

    yl, batches = _model_and_batches()
    kw = dict(conf=0.001, iou=0.7, device=0, verbose=False)

    def check(**extra):
        plain = yl.val(dataloader=_fresh(batches), **kw, **extra).results_dict["metrics/mAP50-95(B)"]
        m = yl.val(dataloader=_fresh(batches), save_hybrid=True, plots=True, **kw, **extra)
        # the priors are the labels themselves at score 1.0: hybrid mAP is inflated, as the reference warns
        assert m.results_dict["metrics/mAP50-95(B)"] > plain, (m.results_dict, plain)
        assert m.confusion_matrix.matrix.sum() > 0

    check(augment=True)
    other = fill_state_dict_(DetectionModel("yolo11n.yaml", verbose=False), 1).eval()
    yl.model = Ensemble([yl.model, other]).cuda().eval()
    check()
