"""Test-time augmentation (`augment=True`) on the B200 path: the two TTA kernels against torch on the same CUDA tensors,
the model against the fp32 oracle (oracle/tta_ref.py), NMS on the merged prediction, narrow ingest dtypes, graph mode,
and the predictor / validator wiring."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import model_state_dict

pytestmark = pytest.mark.gpu

BOX_TOL_PX = 0.5
SCORE_TOL = 1e-2


@pytest.fixture(scope="module")
def n_model(golden):
    """yolo11n with the golden weights on the GPU, and its state_dict for the oracle."""
    from yololite.nn.tasks import DetectionModel

    sd = model_state_dict(golden("model_yolo11n.npz"))
    m = DetectionModel("yolo11n.yaml", verbose=False)
    m.load_state_dict(sd)
    return m.cuda().eval(), sd


@pytest.fixture
def chunk_small_batches(monkeypatch):
    """Let the small test batches take the chunk-pipelined ingest (by default only >= 48 MB chunks are split off)."""
    from yololite.engine.predictor import DetectionPredictor

    monkeypatch.setattr(DetectionPredictor, "pipeline_min_chunk_bytes", 0)


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.uint8])
@pytest.mark.parametrize("shape", [(1, 640, 640), (3, 384, 640), (2, 32, 32), (64, 640, 640)])
def test_scale_img_matches_torch(shape, dtype):
    from yololite import _ops
    from yololite.nn.tasks import tta_geometry

    B, H, W = shape
    g = torch.Generator(device="cuda").manual_seed(B * H + W)
    if dtype is torch.uint8:
        x = torch.randint(0, 256, (B, 3, H, W), dtype=torch.uint8, device="cuda", generator=g)
        xf = x.float() / 255
    else:
        x = torch.rand(B, 3, H, W, device="cuda", generator=g).to(dtype)
        xf = x.float()
    geo = tta_geometry(H, W)[1:]
    outs = [torch.full((B, 3, p.H, p.W), float("nan"), device="cuda") for p in geo]
    _ops.tta_scale_img(x, [(o, (p.h, p.w), p.flip) for o, p in zip(outs, geo)])
    for o, p in zip(outs, geo):
        ref = F.pad(F.interpolate(xf.flip(3) if p.flip else xf, size=(p.h, p.w), mode="bilinear", align_corners=False),
                    [0, p.W - p.w, 0, p.H - p.h], value=0.447)
        assert ref.shape == o.shape
        torch.testing.assert_close(o[..., :p.h, :p.w], ref[..., :p.h, :p.w], rtol=0, atol=1e-6)
        pad = torch.ones(p.H, p.W, dtype=torch.bool, device="cuda")
        pad[:p.h, :p.w] = False
        assert bool((o[..., pad] == torch.tensor(0.447, dtype=torch.float32)).all())


@pytest.mark.parametrize("nc", [80, 3])
@pytest.mark.parametrize("hw", [(640, 640), (384, 640)])
def test_merge_is_bit_identical_to_torch(hw, nc):
    from oracle import tta_ref
    from yololite import _ops
    from yololite.nn.tasks import tta_geometry

    geo = tta_geometry(*hw)
    g = torch.Generator(device="cuda").manual_seed(nc)
    preds = []
    for p in geo:
        t = torch.rand(2, 4 + nc, p.A, device="cuda", generator=g)
        t[:, :4] *= 700
        preds.append(t)
    ref = torch.cat(tta_ref.clip_augmented([tta_ref.descale_pred(t.clone(), p.flip, p.scale, hw)
                                            for t, p in zip(preds, geo)]), -1)
    out = torch.full((2, 4 + nc, sum(p.n for p in geo)), float("nan"), device="cuda")
    _ops.tta_merge([(t, p.a0, p.n, p.scale, p.flip) for t, p in zip(preds, geo)], hw[1], out)
    assert out.shape == ref.shape
    assert torch.equal(out, ref)


# ------------------------------------------------------------------------------------------------ model
@pytest.mark.parametrize("hw", [(640, 640), (384, 640)])
def test_model_augment_matches_oracle(n_model, hw):
    from oracle import tta_ref
    from yololite.nn.tasks import tta_geometry

    m, sd = n_model
    geo = tta_geometry(*hw)
    x = torch.rand(2, 3, *hw, generator=torch.Generator().manual_seed(hw[0]))
    y, none = m(x.cuda(), augment=True)
    assert none is None and tuple(y.shape) == (2, 84, sum(p.n for p in geo)) == (2, 84, {640: 15049, 384: 9000}[hw[0]])
    yr = tta_ref.predict_augment(sd, x).numpy()
    yc = y.cpu().numpy()
    off = 0
    for p in geo:
        seg = slice(off, off + p.n)
        assert np.abs(yc[:, :4, seg] - yr[:, :4, seg]).max() <= BOX_TOL_PX / p.scale, p
        assert np.abs(yc[:, 4:, seg] - yr[:, 4:, seg]).max() <= SCORE_TOL, p
        off += p.n
    plain = m.infer(x.cuda())[0]
    assert torch.equal(y[..., :geo[0].n], plain[..., :geo[0].n])


@pytest.mark.parametrize("kw", [dict(conf=0.25, iou=0.7), dict(conf=0.001, iou=0.7, multi_label=True)])
def test_infer_nms_augment_equals_nms_of_merged(n_model, kw):
    from oracle import nms_ref
    from yololite.utils import ops

    m, _ = n_model
    x = torch.rand(2, 3, 384, 640, generator=torch.Generator().manual_seed(9)).cuda()
    merged = m.infer(x, augment=True)[0].clone()
    d0, c0 = ops.nms_padded(merged.clone(), kw["conf"], kw["iou"], None, False, kw.get("multi_label", False), 300)
    d1, c1 = m.infer_nms(x, augment=True, **kw)
    torch.cuda.synchronize()
    assert torch.equal(c0, c1)
    ref = nms_ref.non_max_suppression(merged.cpu().numpy(), conf_thres=kw["conf"], iou_thres=kw["iou"],
                                      multi_label=kw.get("multi_label", False))
    n = c1.tolist()
    assert n == [len(r) for r in ref]
    for i in range(2):
        np.testing.assert_array_equal(d0[i, :n[i]].cpu().numpy(), d1[i, :n[i]].cpu().numpy())
        np.testing.assert_array_equal(d1[i, :n[i]].cpu().numpy(), ref[i])
    # a class list takes the same path (kept as a device tensor of the TTA state)
    d2, c2 = m.infer_nms(x, augment=True, classes=[0, 5], **kw)
    d3, c3 = ops.nms_padded(merged.clone(), kw["conf"], kw["iou"], [0, 5], False, kw.get("multi_label", False), 300)
    torch.cuda.synchronize()
    assert torch.equal(c2, c3)
    for i in range(2):
        assert torch.equal(d2[i, :int(c2[i])], d3[i, :int(c3[i])])


@pytest.mark.parametrize("hw", [(640, 640), (64, 96)])
def test_augment_narrow_ingest_and_graph_mode_are_bit_identical(n_model, hw):
    """uint8 (bytes / 255) and fp16 batches equal the widened fp32 batch; eager launches equal the CUDA graph.  At 64x96
    all three passes have the same canvas shape (their plans must still be distinct).

    The widening divides by 255 (true division, as the ingest kernels do): torch's `x / 255` multiplies by the fp32
    reciprocal instead, which is 1 ulp off for some bytes, and the rescaled canvases keep that difference in fp32."""
    m, _ = n_model
    xu = torch.randint(0, 256, (2, 3, *hw), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).cuda()
    xf = xu.float() / torch.tensor(255.0, device="cuda")
    y_ref = m.infer(xf, augment=True)[0].clone()
    assert torch.equal(m.infer(xu, augment=True)[0], y_ref)
    xh = xf.half()
    y_h = m.infer(xh, augment=True)[0].clone()
    assert torch.equal(y_h, m.infer(xh.float(), augment=True)[0])
    m.use_cuda_graph = False
    try:
        assert torch.equal(m.infer(xf, augment=True)[0], y_ref)
    finally:
        m.use_cuda_graph = True


# ------------------------------------------------------------------------------------------------ engine
def _expected(model, x_dev, img_shape, orig_shapes, **kw):
    """infer_nms(augment=True) + the rescale kernel to the original images: what the predictor must return."""
    from yololite import _C
    from yololite.utils import ops

    d, c = model.infer_nms(x_dev, augment=True, max_det=300, **kw)
    d, c = d.clone(), c.clone()
    rows = []
    for s0 in orig_shapes:
        gain, pad = ops.letterbox_params(tuple(img_shape), tuple(s0))
        rows.append([gain, pad[0], pad[1], s0[1], s0[0]])
    prm = torch.tensor(rows, dtype=torch.float32).cuda()
    _C.check(_C.load().yl_scale_boxes(d.data_ptr(), c.data_ptr(), d.shape[0], d.shape[1], prm.data_ptr(),
                                      _C.stream_ptr()), "yl_scale_boxes")
    n = c.tolist()
    return [d[i, :n[i]].cpu().numpy() for i in range(len(n))]


def _boxes(results):
    return [r.boxes.data.cpu().numpy() for r in results]


def _same(got, want):
    assert len(got) == len(want)
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a, b)


def test_predictor_augment_host_tensors(n_model, chunk_small_batches):
    from yololite import YOLOLite

    m, sd = n_model
    yl = YOLOLite("yolo11n.yaml")
    yl.model.load_state_dict(sd)
    gen = torch.Generator().manual_seed(6)
    x = torch.rand(64, 3, 64, 64, generator=gen)
    kw = dict(imgsz=64, conf=0.05, iou=0.7, verbose=False, device=0, batch=64)
    b1 = _boxes(yl.predict(x.pin_memory(), augment=True, **kw))
    assert yl.predictor._chunking(x) == 4 and yl.predictor.in_flight == 2     # two lanes / plan slots
    want = _expected(yl.model, x.cuda(), (64, 64), [(64, 64)] * 64, conf=0.05, iou=0.7)
    _same(b1, want)
    _same(_boxes(yl.predict(x.pin_memory(), augment=True, **kw)), want)         # a second call: same result
    plain = _boxes(yl.predict(x.pin_memory(), **kw))
    assert any(len(a) != len(b) or not np.array_equal(a, b) for a, b in zip(plain, want))
    for _ in range(2):                                                          # alternating plain / TTA
        _same(_boxes(yl.predict(x.pin_memory(), augment=True, **kw)), want)
        _same(_boxes(yl.predict(x.pin_memory(), **kw)), plain)
    xu = torch.randint(0, 256, (32, 3, 64, 64), dtype=torch.uint8, generator=gen)
    b8 = _boxes(yl.predict(xu.pin_memory(), augment=True, **dict(kw, batch=32)))
    _same(b8, _expected(yl.model, xu.cuda(), (64, 64), [(64, 64)] * 32, conf=0.05, iou=0.7))


def test_predictor_augment_numpy_images(n_model, golden):
    from test_real_images import _decode
    from yololite import YOLOLite
    from yololite.data import letterbox_batch_cuda

    m, sd = n_model
    real = golden("real_images.npz")
    ims = [_decode(real[f"coco8.jpg{i}"]) for i in range(len(real["coco8.files"]))]
    yl = YOLOLite("yolo11n.yaml")
    yl.model.load_state_dict(sd)
    got = _boxes(yl.predict(ims, augment=True, conf=0.05, iou=0.7, verbose=False, device=0, batch=len(ims)))
    x = letterbox_batch_cuda(ims, (640, 640), auto=False, stride=32)
    _same(got, _expected(yl.model, x, x.shape[2:], [im.shape[:2] for im in ims], conf=0.05, iou=0.7))


def test_validator_augment(n_model, golden):
    from test_real_images import _decode, _raw_labels
    from yololite.data import RectValLoader
    from yololite.engine.validator import DetectionValidator
    from yololite.nn.tasks import tta_geometry

    m, _ = n_model
    real = golden("real_images.npz")
    files = [str(f) for f in real["coco8.files"]]
    ims = [_decode(real[f"coco8.jpg{i}"]) for i in range(len(files))]
    batch = next(iter(RectValLoader(ims, _raw_labels(real), imgsz=640, batch_size=16, stride=32, im_files=files)))
    args = dict(augment=True, device="cuda:0", verbose=False)
    stats = DetectionValidator(dataloader=[dict(batch)], args=args)(model=m)
    v = DetectionValidator(args=args)
    v.device = torch.device("cuda:0")
    v.init_metrics(m)
    b = v.preprocess(dict(batch))
    y, _ = m.infer(b["img"], augment=True)
    assert y.shape[2] == sum(p.n for p in tta_geometry(672, 672))
    v.update_metrics(v.postprocess(y), b)
    assert v.get_stats() == stats


# ------------------------------------------------------------------------------------------------ real images
def test_real_images_augment_agree_with_oracle(golden):
    from oracle import nms_ref, tta_ref
    from test_real_images import _agreement, _decode, _raw_labels, _seeded_model
    from yololite.data import RectValLoader, letterbox_batch_cuda

    real = golden("real_images.npz")
    m, sd = _seeded_model()
    m = m.cuda()
    # boats: the predictor's 384x640 letterbox, conf 0.25
    x = letterbox_batch_cuda([_decode(real["boats.jpg"])], (640, 640), auto=True, stride=32)
    d, c = m.infer_nms(x, conf=0.25, iou=0.7, augment=True)
    mine = d[0, :int(c[0])].cpu().numpy()
    theirs = nms_ref.non_max_suppression(tta_ref.predict_augment(sd, x.cpu()).numpy(), conf_thres=0.25, iou_thres=0.7)[0]
    assert len(theirs) > 0
    f1 = _agreement(theirs[theirs[:, 4] > 0.25 + SCORE_TOL], mine, iou_thr=0.7)
    f2 = _agreement(mine[mine[:, 4] > 0.25 + SCORE_TOL], theirs, iou_thr=0.7)
    assert f1 >= 0.95 and f2 >= 0.95, (f1, f2, len(mine), len(theirs))
    # coco8: the validator's NMS (multi_label, conf 0.001) on the 672x672 rect batch; the oracle side keeps every
    # survivor because the max_det cut falls inside blobs of near-tied scores (see test_real_images)
    files = [str(f) for f in real["coco8.files"]]
    ims = [_decode(real[f"coco8.jpg{i}"]) for i in range(len(files))]
    batch = next(iter(RectValLoader(ims, _raw_labels(real), imgsz=640, batch_size=16, stride=32, im_files=files)))
    x = batch["img"].cuda().float() / 255
    d, c = m.infer_nms(x, conf=0.001, iou=0.7, multi_label=True, augment=True)
    yr = tta_ref.predict_augment(sd, x.cpu()).numpy()
    ref_all = nms_ref.non_max_suppression(yr, conf_thres=0.001, iou_thres=0.7, multi_label=True, max_det=30000)
    for i in range(x.shape[0]):
        f = _agreement(d[i, :int(c[i])].cpu().numpy(), ref_all[i], iou_thr=0.7)
        assert f >= 0.95, (i, f)
