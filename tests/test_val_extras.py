"""Validator switches `save_hybrid=True` (ground-truth priors in NMS) and `plots=True` (confusion matrix), CPU half:
the oracle restatements (oracle/val_extras_ref.py: `non_max_suppression(labels=...)`, `ConfusionMatrix`) on hand-worked
known-answer cases, and the input checks that run before any device is needed."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path[:0] = [str(ROOT / "yolo-lite_b200"), str(ROOT)]

from oracle import metrics_ref, nms_ref, val_extras_ref  # noqa: E402


def _pred(rows, nc):
    """(1, 4+nc, A) prediction from rows (cx, cy, w, h, {cls: score})."""
    p = np.zeros((1, 4 + nc, len(rows)), np.float32)
    for a, (cx, cy, w, h, sc) in enumerate(rows):
        p[0, :4, a] = (cx, cy, w, h)
        for c, v in sc.items():
            p[0, 4 + c, a] = v
    return p


# ------------------------------------------------------------------------------------------------ NMS priors (oracle)
def test_priors_come_after_the_anchors():
    # an anchor at score 1.0 and a prior of the same class on an overlapping box: equal scores, the anchor's row comes
    # first, so it is kept and suppresses the prior
    p = _pred([(50, 50, 20, 20, {0: 1.0})], nc=3)
    lb = [np.array([[0, 51, 50, 20, 20]], np.float32)]
    out = val_extras_ref.non_max_suppression(p, 0.25, 0.45, labels=lb)[0]
    np.testing.assert_array_equal(out, [[40, 40, 60, 60, 1, 0]])


@pytest.mark.parametrize("multi_label", [False, True])
def test_prior_is_a_one_hot_row_in_both_label_modes(multi_label):
    p = _pred([(10, 10, 4, 4, {0: 0.5, 1: 0.6})], nc=3)
    lb = [np.array([[2, 100, 100, 10, 20]], np.float32)]
    out = val_extras_ref.non_max_suppression(p, 0.25, 0.45, multi_label=multi_label, labels=lb)[0]
    anchors = [[8, 8, 12, 12, 0.6, 1]] + ([[8, 8, 12, 12, 0.5, 0]] if multi_label else [])
    np.testing.assert_array_equal(out, np.array([[95, 90, 105, 110, 1, 2]] + anchors, np.float32))


def test_class_filter_and_agnostic_apply_to_priors():
    p = _pred([(50, 50, 20, 20, {0: 0.9})], nc=3)
    lb = [np.array([[1, 50, 50, 20, 20], [2, 200, 200, 8, 8]], np.float32)]
    # class-aware: the prior of class 1 sits on the class-0 anchor without suppressing it
    out = val_extras_ref.non_max_suppression(p, 0.25, 0.45, labels=lb)[0]
    np.testing.assert_array_equal(out[:, 5], [1, 2, 0])
    # agnostic: the prior (score 1.0) suppresses the anchor
    out = val_extras_ref.non_max_suppression(p, 0.25, 0.45, agnostic=True, labels=lb)[0]
    np.testing.assert_array_equal(out[:, 5], [1, 2])
    # classes: only class 2 survives
    out = val_extras_ref.non_max_suppression(p, 0.25, 0.45, classes=[2], labels=lb)[0]
    np.testing.assert_array_equal(out, [[196, 196, 204, 204, 1, 2]])


@pytest.mark.parametrize("multi_label", [False, True])
def test_conf_one_drops_the_priors(multi_label):
    p = _pred([(50, 50, 20, 20, {0: 0.9})], nc=3)
    lb = [np.array([[1, 50, 50, 20, 20]], np.float32)]
    assert val_extras_ref.non_max_suppression(p, 1.0, 0.45, multi_label=multi_label, labels=lb)[0].shape == (0, 6)


def test_image_with_priors_only():
    p = _pred([(50, 50, 20, 20, {0: 0.1})], nc=3)
    lb = [np.array([[1, 50, 50, 20, 20], [1, 52, 50, 20, 20], [0, 300, 300, 10, 10]], np.float32)]
    out = val_extras_ref.non_max_suppression(p, 0.25, 0.45, labels=lb)[0]
    # the second prior of class 1 overlaps the first (IoU 0.82): suppressed; label order is the tie order
    np.testing.assert_array_equal(out, [[40, 40, 60, 60, 1, 1], [295, 295, 305, 305, 1, 0]])


def test_empty_labels_equal_the_plain_oracle():
    g = np.random.default_rng(3)
    p = g.random((3, 4 + 5, 200)).astype(np.float32)
    p[:, :2] *= 300
    p[:, 2:4] *= 40
    for ml in (False, True):
        want = nms_ref.non_max_suppression(p, 0.5, 0.45, multi_label=ml)
        for labels in ((), [np.zeros((0, 5), np.float32)] * 3):
            got = val_extras_ref.non_max_suppression(p, 0.5, 0.45, multi_label=ml, labels=labels)
            assert all(np.array_equal(a, b) for a, b in zip(got, want))


# ------------------------------------------------------------------------------------------------ confusion (oracle)
def _cm(dets, gtb, gtc, nc=3, conf=0.25):
    cm = val_extras_ref.ConfusionMatrix(nc, conf)
    cm.process_batch(None if dets is None else np.asarray(dets, np.float32), np.asarray(gtb, np.float32).reshape(-1, 4),
                     np.asarray(gtc, np.float32))
    return cm.matrix


def test_confusion_keeps_the_highest_iou_detection_not_the_lowest_index():
    gt = [[0, 0, 10, 10]]
    dets = [[0, 0, 10, 16, 0.9, 1],     # IoU 0.625 with the label, higher confidence
            [0, 0, 10, 11, 0.8, 2]]     # IoU 0.909
    m = _cm(dets, gt, [2])
    assert m[2, 2] == 1 and m[1, 3] == 1 and m.sum() == 2
    # match_predictions (same class only) picks by the lowest index instead: with both of class 2, detection 0 wins
    iou = metrics_ref.box_iou(np.float32(gt), np.float32(dets)[:, :4])
    tp = metrics_ref.match_predictions(np.float32([2, 2]), np.float32([2]), iou, np.float32([0.5]))
    assert tp[:, 0].tolist() == [True, False]


def test_confusion_default_conf_substitution():
    assert val_extras_ref.ConfusionMatrix(3, 0.001).conf == 0.25
    assert val_extras_ref.ConfusionMatrix(3, None).conf == 0.25
    assert val_extras_ref.ConfusionMatrix(3, 0.1).conf == 0.1
    m = _cm([[0, 0, 10, 10, 0.2, 0]], [[0, 0, 10, 10]], [0], conf=0.001)
    assert m[3, 0] == 1 and m.sum() == 1    # the 0.2 detection is below the substituted 0.25


def test_confusion_iou_exactly_at_threshold_is_no_match():
    # inter 90, union 200 (+1e-7 vanishes in fp32): IoU == float32(0.45)
    assert metrics_ref.box_iou(np.float32([[0, 0, 9, 10]]), np.float32([[0, 0, 20, 10]]))[0, 0] == np.float32(0.45)
    m = _cm([[0, 0, 20, 10, 0.9, 0]], [[0, 0, 9, 10]], [0])
    assert m[3, 0] == 1 and m[0, 3] == 1 and m[0, 0] == 0
    m = _cm([[0, 0, 20, 10, 0.9, 0]], [[0, 0, 9.5, 10]], [0])
    assert m[0, 0] == 1 and m.sum() == 1


def test_confusion_no_labels_and_no_detections():
    m = _cm([[0, 0, 5, 5, 0.9, 1], [0, 0, 5, 5, 0.1, 2]], np.zeros((0, 4)), [])
    assert m[1, 3] == 1 and m.sum() == 1
    m = _cm(None, [[0, 0, 5, 5], [1, 1, 6, 6]], [0, 2])
    assert m[3, 0] == 1 and m[3, 2] == 1 and m.sum() == 2


def test_confusion_ties_go_to_the_lower_indices():
    # two identical labels and two identical detections: label 0 pairs with detection 0, label 1 stays unmatched
    m = _cm([[0, 0, 10, 10, 0.9, 1], [0, 0, 10, 10, 0.8, 2]], [[0, 0, 10, 10], [0, 0, 10, 10]], [0, 2])
    assert m[1, 0] == 1 and m[3, 2] == 1 and m[2, 3] == 1 and m.sum() == 3


def test_confusion_sum_invariant():
    g = np.random.default_rng(7)
    for _ in range(20):
        n, L = g.integers(0, 30), g.integers(0, 12)
        xy = g.random((L, 2)).astype(np.float32) * 100
        gtb = np.concatenate([xy, xy + 5 + g.random((L, 2)).astype(np.float32) * 30], 1)
        base = gtb[g.integers(0, max(L, 1), n)] if L else np.zeros((n, 4), np.float32)
        dets = np.zeros((n, 6), np.float32)
        dets[:, :4] = base + g.normal(0, 3, (n, 4)).astype(np.float32)
        dets[:, 4] = np.sort(g.random(n).astype(np.float32))[::-1]
        dets[:, 5] = g.integers(0, 4, n)
        gtc = g.integers(0, 4, L).astype(np.float32)
        cm = val_extras_ref.ConfusionMatrix(4, 0.25)
        cm.process_batch(dets, gtb, gtc)
        kept = int((dets[:, 4] > np.float32(0.25)).sum())
        matched = int(cm.matrix[:4, :4].sum())
        assert cm.matrix.sum() == L + (kept - matched)
        assert cm.matrix[4].sum() == L - matched


# ------------------------------------------------------------------------------------------------ input checks
@pytest.mark.parametrize("bad", [3, -1])
def test_prior_class_out_of_range_raises_before_launch(bad):
    from yololite.utils import ops

    pred = torch.zeros((1, 4 + 3, 8))
    with pytest.raises(ValueError, match="outside"):
        ops.non_max_suppression(pred, labels=[torch.tensor([[float(bad), 5, 5, 2, 2]])])
    with pytest.raises(ValueError, match="outside"):
        ops.nms_padded(pred, labels=ops.pack_priors([torch.tensor([[float(bad), 5, 5, 2, 2]])]))


def test_priors_count_must_match_the_batch():
    from yololite.utils import ops

    with pytest.raises(ValueError, match="entries"):
        ops.non_max_suppression(torch.zeros((2, 7, 8)), labels=[torch.zeros((1, 5))])


def test_confusion_matrix_needs_a_device():
    from yololite.utils.metrics import ConfusionMatrix

    cm = ConfusionMatrix(3, conf=0.001)
    assert cm.conf == 0.25 and cm.matrix.shape == (4, 4) and cm.matrix.dtype == np.float64
    with pytest.raises(RuntimeError, match="CUDA"):
        cm.process_batch(torch.zeros((1, 6)), torch.zeros((1, 4)), torch.zeros(1))


def test_validator_switches_default_off():
    from yololite.engine.validator import DetectionValidator

    v = DetectionValidator(dataloader=[], args={"plots": False})
    assert v.confusion_matrix is None and v.lb is None
    v = DetectionValidator(dataloader=[], args={"save_hybrid": True, "plots": True})
    assert v.args.save_hybrid and v.args.plots
