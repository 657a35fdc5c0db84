"""Model ensembles without a GPU: `attempt_load_weights` on lists of checkpoints (the reference's `Ensemble` semantics),
the `Ensemble` attributes and checks, the fp32 oracle of `Ensemble.forward`, the `YOLOLite([...])` facade and the
`embed` refusal."""
from pathlib import Path

import pytest
import torch

from conftest import model_state_dict

ROOT = Path(__file__).resolve().parents[1]
TINY = str(ROOT / "tests" / "golden" / "ckpt_tiny.pt")


def _ckpt(tmp_path, name, cfg="yolo11n.yaml", nc=None, ch=3, salt=0, train_args=None):
    """A checkpoint in the reference's layout: {"model": DetectionModel, "train_args": {...}}."""
    from oracle.weights import fill_state_dict_
    from yololite.nn.tasks import DetectionModel

    m = fill_state_dict_(DetectionModel(cfg, ch=ch, nc=nc, verbose=False), salt)
    path = tmp_path / name
    torch.save({"model": m, "train_args": train_args or {}}, path)
    return str(path)


def test_two_checkpoints_make_an_ensemble(tmp_path):
    from yololite.nn.tasks import DetectionModel, Ensemble, attempt_load_weights

    a = _ckpt(tmp_path, "a.pt", train_args={"imgsz": 320})
    b = _ckpt(tmp_path, "b.pt", "yolo11s.yaml", salt=1)
    e = attempt_load_weights([a, b])
    assert type(e) is Ensemble and len(e) == 2
    assert all(type(m) is DetectionModel and not m.training for m in e)
    assert e[0].pt_path == a and e[1].pt_path == b and e[0].args["imgsz"] == 320
    assert e.names is e[0].names and e.yaml is e[0].yaml and e.nc == 80
    assert e.stride.tolist() == [8.0, 16.0, 32.0]
    keys = set(e.state_dict())
    assert {k.split(".", 1)[0] for k in keys} == {"0", "1"}
    assert {k[2:] for k in keys if k.startswith("0.")} == set(e[0].state_dict())
    assert "0.model.0.conv.weight" in keys and "1.model.23.dfl.conv.weight" in keys


def test_reference_checkpoint_twice():
    from yololite.nn.tasks import Ensemble, attempt_load_one_weight, attempt_load_weights

    e = attempt_load_weights([TINY, TINY])
    alone, _ = attempt_load_one_weight(TINY)
    assert type(e) is Ensemble and len(e) == 2 and e[0] is not e[1]
    assert e.nc == alone.model[-1].nc == 16       # the reference's model carries no `nc`: the head's counts
    assert e.names == alone.names and e.yaml == alone.yaml and e.stride.tolist() == alone.stride.tolist()
    assert set(e.state_dict()) == {f"{i}.{k}" for i in (0, 1) for k in alone.state_dict()}


def test_one_weight_is_the_model_itself(tmp_path):
    from yololite.nn.tasks import DetectionModel, attempt_load_weights

    a = _ckpt(tmp_path, "a.pt")
    for w in (a, [a]):
        m = attempt_load_weights(w)
        assert type(m) is DetectionModel and m.pt_path == a


def test_class_counts_must_agree(tmp_path):
    from yololite.nn.tasks import attempt_load_weights

    a, b = _ckpt(tmp_path, "a.pt"), _ckpt(tmp_path, "b.pt", nc=3)
    with pytest.raises(AssertionError, match=r"Models differ in class counts \[80, 3\]"):
        attempt_load_weights([a, b])


def test_input_channels_must_agree(tmp_path):
    from yololite.nn.tasks import attempt_load_weights

    a, b = _ckpt(tmp_path, "a.pt"), _ckpt(tmp_path, "b.pt", ch=1)
    with pytest.raises(ValueError, match="input channel"):
        attempt_load_weights([a, b])


def test_stride_is_the_largest_members():
    from yololite.nn.tasks import DetectionModel, Ensemble

    a, b = DetectionModel("yolo11n.yaml", verbose=False), DetectionModel("yolo11n.yaml", verbose=False)
    b.stride = torch.tensor([8.0, 16.0, 32.0, 64.0])
    assert Ensemble([a, b]).stride is b.stride and Ensemble([b, a]).stride is b.stride


def test_oracle_concatenates_member_outputs(golden):
    from oracle import ensemble_ref, yolo11_ref

    sds = [model_state_dict(golden("model_yolo11n.npz")), model_state_dict(golden("model_yolo11s.npz"))]
    x = torch.rand(2, 3, 64, 64, generator=torch.Generator().manual_seed(3))
    y, none = ensemble_ref.forward(sds, x)
    parts = [yolo11_ref.forward(sd, x)[0] for sd in sds]
    assert none is None and y.shape == (2, 84, 2 * 84)
    assert torch.equal(y, torch.cat(parts, 2))


def test_yololite_loads_a_list(tmp_path):
    from yololite import YOLOLite
    from yololite.nn.tasks import Ensemble

    a = _ckpt(tmp_path, "a.pt", train_args={"imgsz": 320})
    b = _ckpt(tmp_path, "b.pt", salt=1)
    yl = YOLOLite([a, b])
    assert type(yl.model) is Ensemble and len(yl.model) == 2
    assert yl.ckpt_path == a and yl.overrides["imgsz"] == 320 and yl.overrides["model"] == [a, b]
    assert yl.task == "detect"
    one = YOLOLite([a])
    assert type(one.model) is not Ensemble and one.ckpt_path == a


def test_embed_is_refused(tmp_path):
    from yololite import YOLOLite
    from yololite.nn.tasks import attempt_load_weights

    a, b = _ckpt(tmp_path, "a.pt"), _ckpt(tmp_path, "b.pt", salt=1)
    e = attempt_load_weights([a, b])
    x = torch.zeros(1, 3, 64, 64)                 # a CPU batch: the refusal comes before any device check
    with pytest.raises(TypeError, match="ensemble"):
        e(x, embed=[22])
    with pytest.raises(TypeError, match="ensemble"):
        e.infer_embed(x, [22])
    with pytest.raises(TypeError, match="ensemble"):
        YOLOLite([a, b]).embed(x)
