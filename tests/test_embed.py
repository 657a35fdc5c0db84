"""Feature embeddings (`embed=[...]`) without a GPU: index validation and ordering, the embedding width per model scale,
the oracle against a literal restatement of the reference's `_predict_once` loop, argument checks of yl_embed_pool
(host-side, before any launch), and the predictor / facade wiring."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from conftest import model_state_dict

WIDTH_22 = {"n": 256, "s": 512, "m": 512}


def test_indices_are_sorted_and_deduplicated():
    import numpy as np

    from yololite.nn.tasks import embed_indices

    assert embed_indices([22], 24) == (22,)
    assert embed_indices([22, 4, 4, 10, 0], 24) == (0, 4, 10, 22)
    assert embed_indices((np.int64(6), torch.tensor(3)), 24) == (3, 6)


@pytest.mark.parametrize("bad,err", [([23], ValueError), ([-1], ValueError), ([4, 30], ValueError), ([], ValueError),
                                     (22, TypeError), ("22", TypeError), ([1.5], TypeError), ([True], TypeError)])
def test_index_validation(bad, err):
    from yololite.nn.tasks import embed_indices

    with pytest.raises(err):
        embed_indices(bad, 24)


@pytest.mark.parametrize("scale", ["n", "s", "m"])
def test_width_is_the_sum_of_the_tapped_channels(golden, scale):
    from oracle import embed_ref, yolo11_ref
    from yololite.nn.tasks import DetectionModel

    m = DetectionModel(f"yolo11{scale}.yaml", verbose=False)
    layers = list(m.model)
    sd = model_state_dict(golden(f"model_yolo11{scale}.npz"))
    _, _, ys = yolo11_ref.forward(sd, torch.rand(1, 3, 64, 64, generator=torch.Generator().manual_seed(0)),
                                  return_features=True)
    assert len(ys) == len(layers) - 1
    for k, y in enumerate(ys):
        assert m._out_channels(layers, k, {}) == y.shape[1] and y.shape[1] % 8 == 0, k
    assert m._out_channels(layers, 22, {}) == WIDTH_22[scale]
    idx = [4, 6, 10, 16, 19, 22]
    assert embed_ref.from_features(ys, idx).shape == (1, sum(m._out_channels(layers, k, {}) for k in idx))


def _reference_predict_once(sd, x, embed):
    """The reference's BaseModel._predict_once (nn/tasks.py:118-145) with `embed`, over the oracle's layer functions."""
    from oracle import yolo11_ref as r

    y, embeddings = [], []
    max_idx = max(embed)
    for i, (f, t) in enumerate(r.LAYERS):
        p = f"model.{i}"
        if f != -1:
            x = y[f] if isinstance(f, int) else [x if j == -1 else y[j] for j in f]
        if t == "Conv":
            x = r.conv(sd, p, x, s=2)
        elif t == "C3k2":
            x = r.c3k2(sd, p, x)
        elif t == "SPPF":
            x = r.sppf(sd, p, x)
        elif t == "C2PSA":
            x = r.c2psa(sd, p, x)
        elif t == "Upsample":
            x = F.interpolate(x, scale_factor=2.0, mode="nearest")
        elif t == "Concat":
            x = torch.cat(x, 1)
        else:
            raise AssertionError("the head is never reached")
        y.append(x)
        if i in embed:
            embeddings.append(F.adaptive_avg_pool2d(x, (1, 1)).squeeze(-1).squeeze(-1))
            if i == max_idx:
                return torch.unbind(torch.cat(embeddings, 1), 0)


@pytest.mark.parametrize("idx", [[22], [0], [12, 11], [22, 4, 4, 16, 10, 19, 6]])
def test_oracle_matches_the_reference_loop(golden, idx):
    from oracle import embed_ref

    sd = {k: v.float() for k, v in model_state_dict(golden("model_yolo11n.npz")).items()}
    x = torch.rand(2, 3, 64, 96, generator=torch.Generator().manual_seed(1))
    want = torch.stack(_reference_predict_once(sd, x, idx))
    got = embed_ref.embed(sd, x, idx)
    assert torch.equal(got, want)
    assert embed_ref.embed(sd, x, []) is None               # an empty list is falsy: normal prediction


def _tap(ptr, n, h, w, c, cstride, coff, col):
    from yololite import _C

    return _C.EmbedTap(_C.Tensor(ptr, n, h, w, c, cstride, coff, _C.YL_BF16, 0), col, 0)


def test_c_abi_argument_checks_and_workspace_query():
    """Host-side checks of yl_embed_pool, which run before anything touches the device: a misaligned channel slice is
    refused, and the workspace query sizes the chunk partials + one counter per multi-chunk (image, group tile)."""
    from yololite import _C

    lib = _C.load()

    def query(taps, B, D):
        arr = (_C.EmbedTap * len(taps))(*taps)
        need = ctypes.c_size_t(12345)
        rc = lib.yl_embed_pool(arr, len(taps), B, D, None, None, ctypes.byref(need), None)
        return rc, need.value

    # 20x20x256 at B=2: 32 groups -> 8 pixel lanes, 64 KB / 512 B = 128 pixels per chunk -> 4 chunks
    rc, need = query([_tap(0x10000, 2, 20, 20, 256, 256, 0, 0)], 2, 256)
    assert rc == 0 and need == 2 * 4 * 256 * 4 + 2 * 4
    # 4x4x64: one chunk per image -> no workspace
    assert query([_tap(0x10000, 2, 4, 4, 64, 64, 0, 0)], 2, 64) == (0, 0)
    for bad in (_tap(0x10000, 2, 20, 20, 64, 128, 4, 0),     # coff % 8
                _tap(0x10000, 2, 20, 20, 60, 64, 0, 0),      # c % 8
                _tap(0x10000, 2, 20, 20, 64, 100, 0, 0),     # cstride % 8
                _tap(0x10008, 2, 20, 20, 64, 64, 0, 0),      # data not 16-byte aligned
                _tap(0x10000, 3, 20, 20, 64, 64, 0, 0),      # n != B
                _tap(0x10000, 2, 20, 20, 64, 64, 0, 8)):     # columns beyond D
        assert query([bad], 2, 64)[0] == -1


def test_facade_embed_defaults_to_the_last_neck_layer(monkeypatch):
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    seen = []
    monkeypatch.setattr(YOLOLite, "predict", lambda self, source=None, stream=False, **kw: seen.append((source, stream, kw)))
    yl.embed("src")
    yl.embed("src", stream=True, embed=[4, 6])
    yl.embed("src", embed=[])
    assert seen == [("src", False, {"embed": [22]}), ("src", True, {"embed": [4, 6]}), ("src", False, {"embed": [22]})]


def test_predictor_refuses_augment_with_embed():
    from yololite import YOLOLite
    from yololite.engine.predictor import DetectionPredictor

    with pytest.raises(ValueError, match="augment"):
        DetectionPredictor(overrides=dict(augment=True, embed=[22]))
    with pytest.raises(ValueError, match="augment"):
        YOLOLite("yolo11n.yaml").predict(torch.zeros(1, 3, 64, 64), augment=True, embed=[22])
    DetectionPredictor(overrides=dict(augment=True, embed=[]))        # an empty list is falsy
