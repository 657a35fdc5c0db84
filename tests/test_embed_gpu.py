"""Feature embeddings (`embed=[...]`) on the B200 path: yl_embed_pool against torch on the same bf16 buffers, its
determinism and argument checks, the model against the fp32 oracle (oracle/embed_ref.py), the truncated plans, narrow
ingest and graph mode, and the predictor / backend / facade wiring."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import model_state_dict

pytestmark = pytest.mark.gpu

ATOL, RTOL = 4e-2, 2e-2          # bf16 feature maps (DESIGN.md §4)
SETS = [[22], [0], [11, 12], [4, 6, 10, 16, 19, 22]]


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


# ------------------------------------------------------------------------------------------------ kernel
def _taps(B, seed):
    """Whole buffers and concat slices (coff > 0, cstride > c) of 160², 80², 40² and 20² maps."""
    from yololite._ops import View

    g = torch.Generator(device="cuda").manual_seed(seed)

    def buf(h, w, cstride):
        return torch.randn(B, h, w, cstride, device="cuda", generator=g).to(torch.bfloat16)

    return [View(buf(160, 160, 64), 0, 64), View(buf(80, 80, 192), 128, 64), View(buf(20, 20, 384), 0, 256),
            View(buf(40, 40, 24), 8, 8), View(buf(20, 20, 512), 64, 448)]


@pytest.mark.parametrize("B", [1, 3, 64])
def test_pool_matches_torch_and_is_deterministic(B):
    from yololite import _ops

    views = _taps(B, B)
    D = sum(v.c for v in views)
    out = torch.full((B, D), float("nan"), device="cuda")
    _ops.embed_pool(views, out)
    ref = torch.cat([v.torch_nhwc().float().mean((1, 2)) for v in views], 1)
    torch.testing.assert_close(out, ref, rtol=1e-5, atol=1e-5)
    again = torch.full_like(out, float("nan"))
    _ops.embed_pool(views, again)
    assert torch.equal(out, again)
    # one tap alone lands in the same columns' values
    solo = torch.empty((B, views[2].c), device="cuda")
    _ops.embed_pool([views[2]], solo)
    assert torch.equal(solo, out[:, 128:384])


def test_misaligned_tap_is_refused():
    from yololite import _C

    lib = _C.init(0)
    buf = torch.zeros(2, 20, 20, 64, dtype=torch.bfloat16, device="cuda")
    out = torch.full((2, 32), float("nan"), device="cuda")
    ws = torch.zeros(1 << 16, dtype=torch.uint8, device="cuda")
    arr = (_C.EmbedTap * 1)(_C.EmbedTap(_C.Tensor(buf.data_ptr(), 2, 20, 20, 32, 64, 4, _C.YL_BF16, 0), 0, 0))
    cap = ctypes.c_size_t(ws.numel())
    rc = lib.yl_embed_pool(arr, 1, 2, 32, out.data_ptr(), ws.data_ptr(), ctypes.byref(cap), _C.stream_ptr())
    assert rc == -1 and b"multiples of 8" in lib.yl_last_error_string()
    torch.cuda.synchronize()
    assert bool(out.isnan().all())


# ------------------------------------------------------------------------------------------------ model
def _check(got, ref):
    got, ref = got.cpu().double(), ref.double()
    assert got.shape == ref.shape
    excess = (got - ref).abs() - (ATOL + RTOL * ref.abs())
    assert float(excess.max()) <= 0, float(excess.max())
    cos = torch.nn.functional.cosine_similarity(got, ref, dim=1)
    assert float(cos.min()) >= 0.999, cos.tolist()


def test_model_matches_oracle(n_model):
    from oracle import embed_ref, yolo11_ref

    m, sd = n_model
    x = torch.rand(2, 3, 640, 640, generator=torch.Generator().manual_seed(7))
    _, _, ys = yolo11_ref.forward(sd, x, return_features=True)
    for idx in SETS:
        _check(m.infer_embed(x.cuda(), idx), embed_ref.from_features(ys, idx))


def test_yolo11m_matches_oracle(golden):
    from oracle import embed_ref
    from yololite.nn.tasks import DetectionModel

    sd = model_state_dict(golden("model_yolo11m.npz"))
    m = DetectionModel("yolo11m.yaml", verbose=False)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    x = torch.rand(2, 3, 640, 640, generator=torch.Generator().manual_seed(8))
    got = m.infer_embed(x.cuda(), [22])
    assert got.shape == (2, 512)
    _check(got, embed_ref.embed(sd, x, [22]))


def test_plan_structure(n_model):
    m, _ = n_model
    x = torch.rand(2, 3, 640, 640, device="cuda")
    m.infer_embed(x, [22])
    m.infer_embed(x, [4])
    m.infer_embed(x, [0])
    plans = {k[-1]: v[0] for k, v in m.__dict__["_yl_plans"].items() if k[0] == (2, 3, 640, 640) and k[-1] is not None}
    meta = plans[(22,)].meta
    assert [md["kind"] for md in meta].count("embed_pool") == 1 and meta[-1]["kind"] == "embed_pool"
    assert not any(md["kind"] in ("detect_decode", "nms", "nms_begin", "nms_select") or "+decode" in md["desc"]
                   or "+filter" in md["desc"] for md in meta)
    assert max(md["layer"] for md in meta) == 22
    layers4 = {md["layer"] for md in plans[(4,)].meta}
    assert max(layers4) == 4 and layers4 <= {0, 1, 2, 3, 4}
    assert plans[(4,)].n_launches < plans[(22,)].n_launches
    assert plans[(0,)].calls[0][0].__name__ != "yl_stem_fused"
    assert [md["kind"] for md in plans[(0,)].meta][-1] == "embed_pool"
    assert {md["layer"] for md in plans[(0,)].meta} == {0}


@pytest.mark.parametrize("idx", [[22], [0]])
def test_narrow_ingest_and_graph_mode_are_bit_identical(n_model, idx):
    m, _ = n_model
    xu = torch.randint(0, 256, (3, 3, 640, 640), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).cuda()
    xf = xu.float() / torch.tensor(255.0, device="cuda")
    ref = m.infer_embed(xf, idx).clone()
    assert torch.equal(m.infer_embed(xu, idx), ref)
    xh = xf.half()
    assert torch.equal(m.infer_embed(xh, idx).clone(), m.infer_embed(xh.float(), idx))
    m.use_cuda_graph = False
    try:
        assert torch.equal(m.infer_embed(xf, idx), ref)
    finally:
        m.use_cuda_graph = True


# ------------------------------------------------------------------------------------------------ API
def test_module_and_backend_api(n_model):
    from yololite.nn.autobackend import AutoBackend

    m, _ = n_model
    x = torch.rand(3, 3, 320, 320, device="cuda")
    e = m.infer_embed(x, [22]).clone()
    out = m.predict(x, embed=[22])
    assert isinstance(out, tuple) and len(out) == 3 and all(t.shape == (256,) for t in out)
    assert torch.equal(torch.stack(out), e)
    assert m(x, embed=[22])[0].data_ptr() != m.infer_embed(x, [22]).data_ptr()           # forward returns copies
    y, _ = m.predict(x, augment=True, embed=[22])                                         # augment wins
    assert y.shape[1] == 84
    with pytest.raises(ValueError):
        m.predict(x, embed=[23])
    ab = AutoBackend(m, device=torch.device("cuda:0"), verbose=False)
    one = ab(x[:1], embed=[22])
    assert isinstance(one, torch.Tensor) and one.shape == (256,)
    assert torch.equal(one, m.infer_embed(x[:1], [22])[0])
    many = ab(x, embed=[4, 22])
    assert isinstance(many, list) and len(many) == 3 and all(t.shape == (128 + 256,) for t in many)
    assert isinstance(ab(x)[0], torch.Tensor) and ab(x)[0].dim() == 3                    # embed unset: detections


def _rows(out):
    assert all(isinstance(t, torch.Tensor) and t.dim() == 1 for t in out)
    return torch.stack(list(out))


def test_predict_and_embed_yield_feature_vectors(n_model, golden, chunk_small_batches):
    from test_real_images import _decode
    from yololite import YOLOLite
    from yololite.data import letterbox_batch_cuda

    m, sd = n_model
    yl = YOLOLite("yolo11n.yaml")
    yl.model.load_state_dict(sd)
    kw = dict(imgsz=64, verbose=False, device=0)
    # a device tensor
    x = torch.rand(4, 3, 64, 64, generator=torch.Generator().manual_seed(1)).cuda()
    got = _rows(yl.predict(x, embed=[22], batch=4, **kw))
    want = yl.model.infer_embed(x, [22]).clone()
    assert torch.equal(got, want) and got.shape == (4, 256)
    assert torch.equal(_rows(yl.embed(x, batch=4, **kw)), want)
    assert torch.equal(_rows(list(yl.embed(x, stream=True, batch=4, **kw))), want)
    # a host tensor through the chunk pipeline (4 chunks, two lanes), twice, and the uint8 path
    xh = torch.rand(32, 3, 64, 64, generator=torch.Generator().manual_seed(2))
    want = yl.model.infer_embed(xh.cuda(), [4, 22]).clone()
    for _ in range(2):
        got = _rows(yl.predict(xh.pin_memory(), embed=[4, 22], batch=32, **kw))
        assert yl.predictor._chunking(xh) == 4
        assert torch.equal(got, want)
    xu = torch.randint(0, 256, (32, 3, 64, 64), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    assert torch.equal(_rows(yl.embed(xu.pin_memory(), batch=32, **kw)), yl.model.infer_embed(xu.cuda(), [22]))
    # a list of numpy images (GPU letterbox)
    real = golden("real_images.npz")
    ims = [_decode(real[f"coco8.jpg{i}"]) for i in range(len(real["coco8.files"]))]
    got = _rows(yl.embed(ims, batch=len(ims), verbose=False, device=0))
    xl = letterbox_batch_cuda(ims, (640, 640), auto=False, stride=32)
    assert torch.equal(got, yl.model.infer_embed(xl, [22]))


def _boxes(results):
    return [r.boxes.data.cpu().numpy() for r in results]


def test_detection_path_unchanged_after_embed(n_model, chunk_small_batches):
    from yololite import YOLOLite

    m, sd = n_model
    yl = YOLOLite("yolo11n.yaml")
    yl.model.load_state_dict(sd)
    kw = dict(imgsz=64, conf=0.05, iou=0.7, verbose=False, device=0, batch=32)
    x = torch.rand(32, 3, 64, 64, generator=torch.Generator().manual_seed(4))
    for src in (x.cuda(), x.pin_memory()):
        before = _boxes(yl.predict(src, **kw))
        d0, c0 = (t.clone() for t in yl.model.infer_nms(x.cuda(), 0.05, 0.7))
        yl.predict(src, embed=[22], **kw)
        after = _boxes(yl.predict(src, **kw))
        assert len(before) == len(after) == 32 and sum(len(b) for b in before) > 0
        for a, b in zip(before, after):
            np.testing.assert_array_equal(a, b)
        d1, c1 = yl.model.infer_nms(x.cuda(), 0.05, 0.7)
        assert torch.equal(c0, c1)
        for i in range(32):
            assert torch.equal(d0[i, :int(c0[i])], d1[i, :int(c1[i])])
