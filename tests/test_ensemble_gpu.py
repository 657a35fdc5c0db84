"""Model ensembles on the B200 path: yl_detect_decode_into against yl_detect_decode, `Ensemble.infer` against its members
and the fp32 oracle (oracle/ensemble_ref.py), `Ensemble.infer_nms` against NMS on the concatenated prediction, narrow
ingest, graph mode and slots, `augment=True`, and the loader / backend / facade / predictor / validator wiring."""
import numpy as np
import pytest
import torch

from conftest import model_state_dict

pytestmark = pytest.mark.gpu

BOX_TOL_PX, SCORE_TOL = 0.5, 1e-2          # the head tolerances of the single-model tests


def _model(cfg, salt=0, nc=None, sd=None):
    """(DetectionModel on the GPU, its fp32 state_dict for the oracle) with name-keyed seeded weights (`salt` reseeds)."""
    from oracle.weights import fill_state_dict_
    from yololite.nn.tasks import DetectionModel

    m = DetectionModel(cfg, nc=nc, verbose=False)
    if sd is None:
        fill_state_dict_(m, salt)
    else:
        m.load_state_dict(sd)
    return m.cuda().eval(), {k: v.detach().float().cpu() for k, v in m.state_dict().items()}


@pytest.fixture(scope="module")
def members(golden):
    """Member pairs: yolo11n + yolo11s (golden weights), yolo11n twice (differently seeded), two nc = 3 yolo11n."""
    n = _model("yolo11n.yaml", sd=model_state_dict(golden("model_yolo11n.npz")))
    s = _model("yolo11s.yaml", sd=model_state_dict(golden("model_yolo11s.npz")))
    n1 = _model("yolo11n.yaml", salt=1)
    c3 = [_model("yolo11n.yaml", salt=k, nc=3) for k in (2, 3)]
    return {"n+s": [n, s], "n*2": [n, n1], "nc3": c3}


def _ensemble(pair):
    from yololite.nn.tasks import Ensemble

    return Ensemble([m for m, _ in pair])


def _cat(ms, x):
    return torch.cat([m.infer(x)[0].clone() for m in ms], 2)


def _same_dets(got, want):
    """Equal padded NMS outputs: the counts and every image's valid rows."""
    (d, c), (rd, rc) = got, want
    assert torch.equal(c, rc)
    for i, k in enumerate(c.tolist()):
        assert torch.equal(d[i, :k], rd[i, :k])


@pytest.fixture
def chunk_small_batches(monkeypatch):
    """Let the small test batches take the chunk-pipelined ingest (by default only >= 48 MB chunks are split off)."""
    from yololite.engine.predictor import DetectionPredictor

    monkeypatch.setattr(DetectionPredictor, "pipeline_min_chunk_bytes", 0)


# ------------------------------------------------------------------------------------------------ kernel
@pytest.mark.parametrize("nc", [80, 3])
def test_decode_into_writes_only_its_window(nc):
    from yololite import _ops
    from yololite._ops import View

    B, no = 2, 64 + nc
    g = torch.Generator(device="cuda").manual_seed(nc)
    levels = [View(torch.randn(B, h, h, no, device="cuda", generator=g) * 3, 0, no) for h in (40, 20, 10)]
    A = sum(v.h * v.w for v in levels)
    ref = torch.full((B, 4 + nc, A), float("nan"), device="cuda")
    _ops.detect_decode(levels, (8, 16, 32), 16, nc, ref)
    assert not bool(ref.isnan().any())
    for base, tail in ((0, 0), (8400, 37), (123, 5)):
        y = torch.full((B, 4 + nc, base + A + tail), float("nan"), device="cuda")
        _ops.detect_decode(levels, (8, 16, 32), 16, nc, y, anchor_base=base)
        assert torch.equal(y[..., base:base + A], ref)
        assert bool(y[..., :base].isnan().all()) and bool(y[..., base + A:].isnan().all())


def test_decode_into_refuses_a_window_outside_y():
    from yololite import _C, _ops
    from yololite._ops import View

    levels = [View(torch.zeros(1, h, h, 144, device="cuda"), 0, 144) for h in (4, 2, 1)]
    y = torch.full((1, 84, 30), float("nan"), device="cuda")
    with pytest.raises(_C.YLError, match="anchor window"):
        _ops.detect_decode(levels, (8, 16, 32), 16, 80, y, anchor_base=10)
    torch.cuda.synchronize()
    assert bool(y.isnan().all())


# ------------------------------------------------------------------------------------------------ model
@pytest.mark.parametrize("pair", ["n+s", "n*2", "nc3"])
def test_infer_is_the_concatenation_of_the_members(members, pair):
    ms = [m for m, _ in members[pair]]
    e = _ensemble(members[pair])
    for B, hw in ((2, (640, 640)), (3, (384, 640))):
        x = torch.rand(B, 3, *hw, device="cuda", generator=torch.Generator(device="cuda").manual_seed(B))
        y, raws = e.infer(x)
        assert raws == [] and y.shape[2] == sum(m.infer(x)[0].shape[2] for m in ms)
        assert torch.equal(y, _cat(ms, x))
        y2, none = e(x)                                  # module-level API: a fresh tensor, like the reference
        assert none is None and torch.equal(y2, y) and y2.data_ptr() != y.data_ptr()


@pytest.mark.parametrize("pair", ["n+s", "nc3"])
def test_infer_matches_the_oracle(members, pair):
    from oracle import ensemble_ref

    e = _ensemble(members[pair])
    x = torch.rand(2, 3, 320, 320, generator=torch.Generator().manual_seed(11))
    y = e.infer(x.cuda())[0].cpu()
    ref, _ = ensemble_ref.forward([sd for _, sd in members[pair]], x)
    assert y.shape == ref.shape
    assert float((y[:, :4] - ref[:, :4]).abs().max()) <= BOX_TOL_PX
    assert float((y[:, 4:] - ref[:, 4:]).abs().max()) <= SCORE_TOL


NMS_ARGS = [dict(conf=0.1, iou=0.7), dict(conf=0.05, iou=0.45, multi_label=True), dict(conf=0.1, iou=0.6, classes="best"),
            dict(conf=0.1, iou=0.6, agnostic=True)]


@pytest.mark.parametrize("kw", NMS_ARGS)
@pytest.mark.parametrize("pair", ["n+s", "n*2", "nc3"])
def test_infer_nms_is_nms_of_the_concatenation(members, pair, kw):
    from yololite.nn.tasks import _nms_key
    from yololite.utils import ops

    ms = [m for m, _ in members[pair]]
    e = _ensemble(members[pair])
    x = torch.rand(4, 3, 640, 640, device="cuda", generator=torch.Generator(device="cuda").manual_seed(5))
    if kw.get("classes") == "best":          # class 0 and the class of the highest score of image 0
        y = _cat(ms, x)
        kw = dict(kw, classes=sorted({0, int(y[0, 4:].flatten().argmax()) // y.shape[2]}))
    d, c = e.infer_nms(x, **kw)
    rd, rc = ops.nms_padded(_cat(ms, x), kw["conf"], kw["iou"], kw.get("classes"), kw.get("agnostic", False),
                            kw.get("multi_label", False), 300)
    _same_dets((d, c), (rd, rc))
    assert int(c.sum()) > 0
    key = _nms_key(kw["conf"], kw["iou"], kw.get("classes"), kw.get("agnostic", False), kw.get("multi_label", False), 300,
                   30000, 7680.0)
    plan = e._get_plan(x.shape, x.device, 0, key)[0]
    kinds = [md["kind"] for md in plan.meta]
    fused = pair != "nc3" and not kw.get("multi_label") and "classes" not in kw
    assert ("nms_select" in kinds) == fused and ("nms" in kinds) == (not fused)
    assert kinds.count("nms_begin") == int(fused)
    # one plan: every member's ingest leads (eager), everything else is one graph
    assert plan.n_ingest == 2 and all(k in ("stem_fused", "stem_conv", "ingest_nchw_to_nhwc") for k in kinds[:2])


@pytest.mark.parametrize("pair", ["n*2", "n+s"])
def test_narrow_ingest_graph_mode_and_slots(members, pair):
    """uint8 (bytes / 255) and fp16 batches equal the widened fp32 batch; eager launches equal the CUDA graph; two
    slots are independent plans with the same result.  yolo11n's fused stem reads all three dtypes; yolo11s's stem
    conv reads fp32 only, so with it in the ensemble narrow batches are widened once into the shared input."""
    from yololite import _C

    e = _ensemble(members[pair])
    xu = torch.randint(0, 256, (2, 3, 640, 640), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).cuda()
    xf = xu.float() / torch.tensor(255.0, device="cuda")
    y_ref = e.infer(xf)[0].clone()
    native = {_C.YL_F32, _C.YL_F16, _C.YL_U8} if pair == "n*2" else {_C.YL_F32}
    assert set(e._get_plan(xf.shape, xf.device)[0].native_ingest) == native
    assert torch.equal(e.infer(xu)[0], y_ref)
    xh = xf.half()
    assert torch.equal(e.infer(xh)[0].clone(), e.infer(xh.float())[0])
    ref = tuple(t.clone() for t in e.infer_nms(xu, conf=0.25, iou=0.7))
    _same_dets(e.infer_nms(xf, conf=0.25, iou=0.7, slot=1), ref)
    assert e.infer(xf, slot=1)[0].data_ptr() != e.infer(xf, slot=0)[0].data_ptr()
    e.use_cuda_graph = False
    try:
        assert torch.equal(e.infer(xf)[0], y_ref)
        _same_dets(e.infer_nms(xu, conf=0.25, iou=0.7), ref)
    finally:
        e.use_cuda_graph = True


def test_augment_warns_and_predicts_single_scale(members, monkeypatch):
    from yololite.nn import tasks

    e = _ensemble(members["n*2"])
    x = torch.rand(2, 3, 640, 640, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    plain = e.infer(x)[0].clone()
    seen = []
    monkeypatch.setattr(tasks.LOGGER, "warning", lambda msg, *a, **k: seen.append(msg))
    y, none = e(x, augment=True)
    assert none is None and torch.equal(y, plain)
    assert len(seen) == 1 and "not applied to model ensembles" in seen[0]
    ref = tuple(t.clone() for t in e.infer_nms(x))
    _same_dets(e.infer_nms(x, augment=True), ref)


def test_plan_lru_is_bounded(members):
    e = _ensemble(members["n*2"])
    e.max_plans = 2
    for h in (64, 96, 128):
        e.infer(torch.rand(1, 3, h, 64, device="cuda"))
    assert len(e._yl_plans) == 2


# ------------------------------------------------------------------------------------------------ public surface
@pytest.fixture(scope="module")
def ckpts(tmp_path_factory):
    """The members of members["n*2"] (yolo11n, seeds 0 and 1) as reference-layout checkpoints."""
    from oracle.weights import fill_state_dict_
    from yololite.nn.tasks import DetectionModel

    d = tmp_path_factory.mktemp("ens")
    paths = []
    for k in range(2):
        p = d / f"m{k}.pt"
        torch.save({"model": fill_state_dict_(DetectionModel("yolo11n.yaml", verbose=False), k), "train_args": {"imgsz": 64}}, p)
        paths.append(str(p))
    return paths


def _expected(ms, x_dev, orig_shapes, **kw):
    """NMS on the concatenated member predictions + the rescale kernel: what the predictor must return."""
    from yololite import _C
    from yololite.utils import ops

    d, c = ops.nms_padded(_cat(ms, x_dev), kw["conf"], kw["iou"], None, False, False, 300)
    rows = []
    for s0 in orig_shapes:
        gain, pad = ops.letterbox_params(tuple(x_dev.shape[2:]), tuple(s0))
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


def test_autobackend_keeps_every_member(members, ckpts):
    """A list of checkpoints is one ensemble: the prediction has the anchors of both members (not only the first's)."""
    from yololite.nn.autobackend import AutoBackend
    from yololite.nn.tasks import Ensemble

    ms = [m for m, _ in members["n*2"]]
    be = AutoBackend(weights=ckpts, device=torch.device("cuda:0"))
    assert type(be.model) is Ensemble and len(be.model) == 2 and be.stride == 32
    x = torch.rand(2, 3, 640, 640, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1))
    y, raws = be(x)
    assert y.shape == (2, 84, 2 * 8400)
    assert torch.equal(y, _cat(ms, x))
    assert AutoBackend(weights=be.model, device=torch.device("cuda:0")).model is be.model
    with pytest.raises(TypeError, match="ensemble"):
        be(x, embed=[22])


def test_predictor_plain_and_pipelined(members, ckpts, chunk_small_batches):
    from yololite import YOLOLite

    ms = [m for m, _ in members["n*2"]]
    yl = YOLOLite(ckpts)
    kw = dict(imgsz=64, conf=0.05, iou=0.7, verbose=False, device=0)
    gen = torch.Generator().manual_seed(6)
    x = torch.rand(64, 3, 64, 64, generator=gen)
    want = _expected(ms, x.cuda(), [(64, 64)] * 64, conf=0.05, iou=0.7)
    _same(_boxes(yl.predict(x.pin_memory(), batch=64, **kw)), want)       # host tensor: chunk-pipelined, two slots
    assert yl.predictor._chunking(x) == 4 and yl.predictor.in_flight == 2
    _same(_boxes(yl.predict(x.pin_memory(), batch=64, **kw)), want)
    _same(_boxes(yl.predict(x.cuda(), batch=64, **kw)), want)             # device tensor: the plain path
    xu = torch.randint(0, 256, (32, 3, 64, 64), dtype=torch.uint8, generator=gen)
    _same(_boxes(yl.predict(xu.pin_memory(), batch=32, **kw)),
          _expected(ms, xu.cuda().float() / torch.tensor(255.0, device="cuda"), [(64, 64)] * 32, conf=0.05, iou=0.7))
    with pytest.raises(TypeError, match="ensemble"):
        yl.predict(x.cuda(), embed=[22], **kw)


def test_predictor_numpy_images(members, ckpts, golden):
    from test_real_images import _decode
    from yololite import YOLOLite
    from yololite.data import letterbox_batch_cuda

    ms = [m for m, _ in members["n*2"]]
    real = golden("real_images.npz")
    ims = [_decode(real[f"coco8.jpg{i}"]) for i in range(len(real["coco8.files"]))]
    got = _boxes(YOLOLite(ckpts).predict(ims, imgsz=640, conf=0.05, iou=0.7, verbose=False, device=0, batch=len(ims)))
    x = letterbox_batch_cuda(ims, (640, 640), auto=False, stride=32)
    _same(got, _expected(ms, x, [im.shape[:2] for im in ims], conf=0.05, iou=0.7))


def test_validator(members, golden):
    from test_real_images import _decode, _raw_labels
    from yololite.data import RectValLoader
    from yololite.engine.validator import DetectionValidator

    ms = [m for m, _ in members["n+s"]]
    e = _ensemble(members["n+s"])
    real = golden("real_images.npz")
    files = [str(f) for f in real["coco8.files"]]
    ims = [_decode(real[f"coco8.jpg{i}"]) for i in range(len(files))]
    batch = next(iter(RectValLoader(ims, _raw_labels(real), imgsz=640, batch_size=16, stride=32, im_files=files)))
    args = dict(device="cuda:0", verbose=False)
    stats = DetectionValidator(dataloader=[dict(batch)], args=args)(model=e)
    v = DetectionValidator(args=args)
    v.device = torch.device("cuda:0")
    v.init_metrics(e)
    b = v.preprocess(dict(batch))
    v.update_metrics(v.postprocess(_cat(ms, b["img"])), b)
    assert v.get_stats() == stats
