"""Test-time augmentation geometry (no GPU): the host-side pass geometry of `augment=True` against the reference's
scale_img / _clip_augmented arithmetic, and the oracle's clip against slicing off whole pyramid levels."""
import math

import pytest
import torch

# (h, w) -> per pass (content (h, w), canvas (H, W), anchors, kept anchors), merged anchors
TABLE = {
    (640, 640): ([((640, 640), (640, 640), 8400, 8000), ((531, 531), (544, 544), 6069, 6069),
                  ((428, 428), (448, 448), 4116, 980)], 15049),
    (384, 640): ([((384, 640), (384, 640), 5040, 4800), ((318, 531), (320, 544), 3570, 3570),
                  ((257, 428), (288, 448), 2646, 630)], 9000),
}
EXTRA = [(32, 32), (64, 96), (1280, 736)]


def _levels(H, W, strides=(8, 16, 32)):
    return [(H // s) * (W // s) for s in strides]


@pytest.mark.parametrize("hw", list(TABLE))
def test_geometry_matches_the_table(hw):
    from yololite.nn.tasks import tta_geometry

    passes, merged = TABLE[hw]
    geo = tta_geometry(*hw)
    assert [p.scale for p in geo] == [1, 0.83, 0.67] and [p.flip for p in geo] == [None, 3, None]
    for p, (content, canvas, A, kept) in zip(geo, passes):
        assert ((p.h, p.w), (p.H, p.W), p.A, p.n) == (content, canvas, A, kept)
    assert sum(p.n for p in geo) == merged
    assert geo[0].a0 == 0 and geo[1].a0 == 0 and geo[2].a0 + geo[2].n == geo[2].A


@pytest.mark.parametrize("hw", list(TABLE) + EXTRA)
def test_kept_anchors_drop_exactly_p5_of_pass0_and_p3_of_pass2(hw):
    from yololite.nn.tasks import tta_geometry

    h, w = hw
    geo = tta_geometry(h, w)
    for p in geo[1:]:
        assert (p.h, p.w) == (int(h * p.scale), int(w * p.scale))
        assert (p.H, p.W) == (math.ceil(h * p.scale / 32) * 32, math.ceil(w * p.scale / 32) * 32)
    for p in geo:
        assert p.A == sum(_levels(p.H, p.W)) and p.H % 32 == 0 and p.W % 32 == 0
    assert geo[0].A - geo[0].n == _levels(geo[0].H, geo[0].W)[2]        # P5 of scale 1
    assert geo[2].a0 == _levels(geo[2].H, geo[2].W)[0]                 # P3 of scale 0.67
    assert geo[1].n == geo[1].A


@pytest.mark.parametrize("hw", list(TABLE) + EXTRA)
def test_oracle_clip_equals_slicing_off_levels(hw):
    from oracle import tta_ref
    from yololite.nn.tasks import tta_geometry

    geo = tta_geometry(*hw)
    g = torch.Generator().manual_seed(0)
    ys = [torch.rand(2, 7, p.A, generator=g) for p in geo]
    clipped = tta_ref.clip_augmented(list(ys))
    p5 = _levels(geo[0].H, geo[0].W)[2]
    p3 = _levels(geo[2].H, geo[2].W)[0]
    assert torch.equal(clipped[0], ys[0][..., : geo[0].A - p5])
    assert torch.equal(clipped[1], ys[1])
    assert torch.equal(clipped[2], ys[2][..., p3:])
    for c, p in zip(clipped, geo):
        assert torch.equal(c, ys[geo.index(p)][..., p.a0: p.a0 + p.n])


def test_oracle_scale_img_and_descale_pred():
    """scale_img pads with 0.447 to a multiple of gs; _descale_pred divides the box rows and mirrors x."""
    from oracle import tta_ref

    x = torch.rand(1, 3, 64, 96, generator=torch.Generator().manual_seed(1))
    y = tta_ref.scale_img(x, 0.67)
    assert y.shape == (1, 3, 64, 96)
    assert bool((y[..., 42:, :] == torch.tensor(0.447)).all()) and bool((y[..., :, 64:] == torch.tensor(0.447)).all())
    assert tta_ref.scale_img(x, 1.0) is x
    p = torch.tensor([[[10.0], [20.0], [4.0], [6.0], [0.5]]])
    d = tta_ref.descale_pred(p.clone(), 3, 0.5, (64, 96))
    assert d[0, :, 0].tolist() == [96 - 20.0, 40.0, 8.0, 12.0, 0.5]
