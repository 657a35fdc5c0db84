"""GPU parity of the drop-in nn modules and full models against fixtures produced by the reference itself
(tests/golden, oracle/gen_golden.py) and against the oracle at BASELINE sizes.

Tolerances (bf16 storage, fp32 accumulation) are the north star's: box coordinates <= 0.5 px, class scores
<= 1e-2 absolute; intermediate feature maps: |d| <= 4e-2 + 2e-2*|ref| (bf16 has 8 mantissa bits)."""
import numpy as np
import pytest
import torch

from conftest import model_state_dict

pytestmark = pytest.mark.gpu

BOX_TOL_PX = 0.5
SCORE_TOL = 1e-2


def feat_close(got, ref, tag):
    np.testing.assert_allclose(np.asarray(got), np.asarray(ref), rtol=2e-2, atol=4e-2, err_msg=tag)


def _mk(tag):
    from yololite.nn.modules import C2PSA, C3k, C3k2, SPPF, Attention, Bottleneck, Conv, DWConv, PSABlock

    return {
        "conv_k3s2": lambda: Conv(16, 32, 3, 2), "conv_k1": lambda: Conv(48, 64, 1, 1),
        "conv_k3s1_noact": lambda: Conv(32, 16, 3, 1, act=False), "conv_stem": lambda: Conv(3, 16, 3, 2),
        "dwconv": lambda: DWConv(64, 64, 3), "bottleneck": lambda: Bottleneck(32, 32, True),
        "c3k": lambda: C3k(64, 64, 2), "c3k2_plain": lambda: C3k2(64, 128, 1, False, 0.25),
        "c3k2_c3k": lambda: C3k2(128, 128, 1, True), "sppf": lambda: SPPF(128, 128, 5),
        "attention": lambda: Attention(128, num_heads=2, attn_ratio=0.5), "psablock": lambda: PSABlock(128, 0.5, 2),
        "c2psa": lambda: C2PSA(256, 256, 1),
    }[tag]()


MODULE_TAGS = ["conv_k3s2", "conv_k1", "conv_k3s1_noact", "conv_stem", "dwconv", "bottleneck", "c3k", "c3k2_plain",
               "c3k2_c3k", "sppf", "attention", "psablock", "c2psa"]


@pytest.mark.parametrize("tag", MODULE_TAGS)
def test_module_matches_reference(golden, tag):
    from oracle.weights import fill_state_dict_

    g = golden("modules.npz")
    m = fill_state_dict_(_mk(tag)).cuda().eval()
    x = torch.from_numpy(g[f"{tag}.x"]).cuda()
    y = m(x)
    assert y.dtype == torch.float32 and tuple(y.shape) == g[f"{tag}.y"].shape
    feat_close(y.cpu().numpy(), g[f"{tag}.y"], tag)
    y2 = m(x)                                            # cached plan replay gives identical results
    assert torch.equal(y, y2)


def test_dfl_and_detect_match_reference(golden):
    from oracle.weights import fill_state_dict_
    from yololite.nn.modules import DFL, Detect

    g = golden("modules.npz")
    d = DFL(16).cuda()
    np.testing.assert_allclose(d(torch.from_numpy(g["dfl.x"]).cuda()).cpu().numpy(), g["dfl.y"], rtol=1e-5, atol=1e-5)
    det = Detect(80, (64, 128, 256))
    det.stride = torch.tensor([8.0, 16.0, 32.0])
    fill_state_dict_(det).cuda().eval()
    y, raw = det([torch.from_numpy(g[f"detect.x{i}"]).cuda() for i in range(3)])
    for i in range(3):
        assert tuple(raw[i].shape) == g[f"detect.raw{i}"].shape
        feat_close(raw[i].cpu().numpy(), g[f"detect.raw{i}"], f"raw{i}")
    y = y.cpu().numpy()
    assert np.abs(y[:, :4] - g["detect.y"][:, :4]).max() <= BOX_TOL_PX
    assert np.abs(y[:, 4:] - g["detect.y"][:, 4:]).max() <= SCORE_TOL


@pytest.mark.parametrize("scale", ["n", "s", "m"])
@pytest.mark.parametrize("graph", [True, False])
def test_model_matches_reference_golden(golden, scale, graph):
    from yololite.nn.tasks import DetectionModel

    g = golden(f"model_yolo11{scale}.npz")
    m = DetectionModel(f"yolo11{scale}.yaml", verbose=False)
    m.use_cuda_graph = graph
    m.load_state_dict(model_state_dict(g))
    m = m.cuda().eval()
    y, raw = m(torch.from_numpy(g["x"]).cuda())
    assert tuple(y.shape) == g["y"].shape and y.dtype == torch.float32
    for i in range(3):
        assert tuple(raw[i].shape) == g[f"raw{i}"].shape
        feat_close(raw[i].cpu().numpy(), g[f"raw{i}"], f"raw{i}")
    y = y.cpu().numpy()
    assert np.abs(y[:, :4] - g["y"][:, :4]).max() <= BOX_TOL_PX
    assert np.abs(y[:, 4:] - g["y"][:, 4:]).max() <= SCORE_TOL


def test_model_640_matches_oracle_and_nms_end_to_end(golden):
    """BASELINE config 3 shape (yolo11n, 640x640): head output within tolerance of the fp32 oracle; NMS on the
    GPU's own pre-NMS tensor is bit-exact against the oracle NMS on the same tensor."""
    from oracle import nms_ref, yolo11_ref
    from yololite.nn.tasks import DetectionModel
    from yololite.utils import ops

    g = golden("model_yolo11n.npz")
    sd = model_state_dict(g)
    m = DetectionModel("yolo11n.yaml", verbose=False)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    x = torch.rand(4, 3, 640, 640, generator=torch.Generator().manual_seed(0))
    yr, _ = yolo11_ref.forward(sd, x)
    y, _ = m(x.cuda())
    assert tuple(y.shape) == (4, 84, 8400)
    yc = y.cpu().numpy()
    assert np.abs(yc[:, :4] - yr.numpy()[:, :4]).max() <= BOX_TOL_PX
    assert np.abs(yc[:, 4:] - yr.numpy()[:, 4:]).max() <= SCORE_TOL
    for kw in (dict(conf_thres=0.25, iou_thres=0.7), dict(conf_thres=0.001, iou_thres=0.7, multi_label=True)):
        got = ops.non_max_suppression(y.clone(), **kw)
        ref = nms_ref.non_max_suppression(yc, **kw)
        assert [len(a) for a in got] == [len(b) for b in ref]
        for a, b in zip(got, ref):
            np.testing.assert_array_equal(a.cpu().numpy(), b)


def test_nms_in_place_side_effect_and_list_layout():
    from yololite.utils import ops

    p = torch.rand(2, 84, 256, device="cuda")
    p[:, :4] *= 100
    before = p.clone()
    out = ops.non_max_suppression(p, 0.5, 0.5)
    assert isinstance(out, list) and len(out) == 2 and all(o.shape[1] == 6 and o.dtype == torch.float32 for o in out)
    torch.testing.assert_close(p[:, :4].transpose(1, 2), ops.xywh2xyxy(before[:, :4].transpose(1, 2)))
    torch.testing.assert_close(p[:, 4:], before[:, 4:])
    out2 = ops.non_max_suppression((before.clone(), None), 0.5, 0.5, in_place=False)   # tuple input accepted
    for a, b in zip(out, out2):
        assert torch.equal(a, b)
    with pytest.raises(AssertionError):
        ops.non_max_suppression(before, conf_thres=1.5)
    empty = ops.non_max_suppression(torch.zeros(1, 84, 64, device="cuda"), 0.25, 0.45)
    assert empty[0].shape == (0, 6)


def test_yololite_predict_tensor_and_numpy(golden):
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    x = torch.rand(2, 3, 640, 640, generator=torch.Generator().manual_seed(1))
    res = yl.predict(x, conf=0.05, verbose=False)
    assert len(res) == 2
    for r in res:
        b = r.boxes
        assert b.data.shape[1] == 6 and r.orig_shape == (640, 640)
        if len(b):
            assert float(b.conf.min()) > 0.05 and bool((b.conf[:-1] >= b.conf[1:]).all())
            assert float(b.xyxy.min()) >= 0 and float(b.xyxy.max()) <= 640
        assert set(r.speed) == {"preprocess", "inference", "postprocess"}
    # numpy HWC BGR image, letterboxed 1080x1920 -> 384x640 like the reference predictor
    im = (np.random.default_rng(0).uniform(0, 255, (1080, 1920, 3))).astype(np.uint8)
    r2 = yl(im, conf=0.05, verbose=False)
    assert len(r2) == 1 and r2[0].orig_shape == (1080, 1920)
    if len(r2[0].boxes):
        assert float(r2[0].boxes.xyxy[:, [0, 2]].max()) <= 1920 and float(r2[0].boxes.xyxy[:, [1, 3]].max()) <= 1080


def test_checkpoint_roundtrip_pt(tmp_path, golden):
    """A reference-format checkpoint ({'model': module}) loads through YOLOLite('x.pt') and predicts identically."""
    from yololite import YOLOLite
    from yololite.nn.tasks import DetectionModel

    g = golden("model_yolo11n.npz")
    m = DetectionModel("yolo11n.yaml", verbose=False)
    m.load_state_dict(model_state_dict(g))
    p = tmp_path / "tiny.pt"
    torch.save({"model": m.half(), "train_args": {}}, p)
    yl = YOLOLite(str(p))
    x = torch.from_numpy(g["x"])
    y, _ = yl.model.cuda().eval()(x.cuda())
    assert np.abs(y.cpu().numpy()[:, 4:] - g["y"][:, 4:]).max() <= SCORE_TOL


def test_fused_decode_matches_decode_kernel_and_engine_path(golden):
    """The Detect decode fused into the head convs' epilogue (a) equals the standalone decode kernel fed by the
    raw maps within fp32 rounding of the fast exp, (b) is identical with and without materialising the raw maps
    (engine path `infer(want_raw=False)`), also for a batch that leaves the last 128-pixel tile ragged."""
    _check_fused_decode(golden, "yolo11n", 80)


@pytest.mark.parametrize("cfg,nc", [("yolo11n", 64), ("yolo11s", 256)])
def test_fused_decode_matches_decode_kernel_and_engine_path_class_counts(golden, cfg, nc):
    """The same parity for class counts at which a plain conv of these small class maps would be split into N tiles
    (nc % 64 == 0): the fused class decode addresses its rows by the chunk index inside one N tile, so those convs must
    run unsplit (nc = 256 on yolo11s: yolo11n's class branch would be 100 channels wide, which the fused decode does not
    take)."""
    _check_fused_decode(golden, cfg, nc)


def _check_fused_decode(golden, cfg, nc):
    from oracle.weights import tensor_for
    from yololite.nn.modules import Detect
    from yololite.nn.tasks import DetectionModel

    g = golden("model_yolo11n.npz")
    sd = model_state_dict(g)
    if nc != 80:
        shapes = DetectionModel(f"{cfg}.yaml", nc=nc, verbose=False).state_dict()
        sd = {k: tensor_for(k, tuple(v.shape)) for k, v in shapes.items()}
    x = torch.rand(3, 3, 96, 160, generator=torch.Generator().manual_seed(5)).cuda()   # P5 map: 3*3*5 = 45 pixels
    outs = {}
    for fuse in (True, False):
        Detect.fuse_decode = fuse
        try:
            m = DetectionModel(f"{cfg}.yaml", nc=nc, verbose=False)
            m.load_state_dict(sd)
            m = m.cuda().eval()
            assert m.model[-1]._fuses_decode() == fuse
            y, raw = m(x)
            outs[fuse] = (y.cpu().numpy(), [r.cpu().numpy() for r in raw])
            if fuse:
                y_engine, no_raw = m.infer(x)           # want_raw=False: separate plan, no raw maps written
                assert no_raw == []
                np.testing.assert_array_equal(y_engine.cpu().numpy(), outs[True][0])
        finally:
            Detect.fuse_decode = True
    (yf, rf), (yk, rk) = outs[True], outs[False]
    for a, b in zip(rf, rk):
        np.testing.assert_array_equal(a, b)              # same conv, same raw logits
    assert np.abs(yf[:, :4] - yk[:, :4]).max() <= 2e-3   # box px: __expf / __fdividef vs expf / div
    assert np.abs(yf[:, 4:] - yk[:, 4:]).max() <= 1e-5


@pytest.fixture
def chunk_small_batches(monkeypatch):
    """Let the small test batches take the chunk-pipelined ingest (by default only >= 48 MB chunks are split off)."""
    from yololite.engine.predictor import DetectionPredictor

    monkeypatch.setattr(DetectionPredictor, "pipeline_min_chunk_bytes", 0)


def test_predict_pipelined_host_batch_equals_device_batch(golden, chunk_small_batches):
    """A pinned HOST batch goes through the chunk-pipelined ingest (4 chunks of 8); the detections must be the
    same as for the same batch already resident on the device (single plan, no chunking)."""
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    x = torch.rand(32, 3, 64, 96, generator=torch.Generator().manual_seed(2))
    r_host = yl.predict(x.pin_memory(), conf=0.05, verbose=False)
    assert yl.predictor._chunking(x) == 4
    r_dev = yl.predict(x.cuda(), conf=0.05, verbose=False)
    assert len(r_host) == len(r_dev) == 32
    for a, b in zip(r_host, r_dev):
        assert torch.equal(a.boxes.data, b.boxes.data)


def test_predict_fp16_host_tensor_matches_fp32_path():
    """An fp16 host batch (half the upload) is widened on the device and gives the detections of the same values
    fed as fp32 (the reference applies `.float()` on the device, engine/predictor.py:83)."""
    import numpy as np
    import torch

    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    x16 = torch.rand(16, 3, 64, 64, generator=torch.Generator().manual_seed(4)).half().pin_memory()
    r16 = yl.predict(x16, imgsz=64, conf=0.001, verbose=False, device=0, batch=16)
    r32 = yl.predict(x16.float().pin_memory(), imgsz=64, conf=0.001, verbose=False, device=0, batch=16)
    assert len(r16) == len(r32) == 16
    for a, b in zip(r16, r32):
        assert np.array_equal(a.boxes.data.cpu().numpy(), b.boxes.data.cpu().numpy())


def test_async_host_predict_then_device_predict_do_not_race():
    """A device-tensor predict (plain path, caller's stream) right after an asynchronous host-tensor predict shares
    the plan slots with it: both must still produce the detections of their own batch."""
    import numpy as np
    import torch

    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    g = torch.Generator().manual_seed(8)
    xa = torch.rand(16, 3, 64, 64, generator=g).pin_memory()
    xb = torch.rand(16, 3, 64, 64, generator=g)
    kw = dict(imgsz=64, conf=0.001, verbose=False, device=0, batch=16)
    ref_a = [r.boxes.data.cpu().numpy() for r in yl.predict(xa, **kw)]
    ref_b = [r.boxes.data.cpu().numpy() for r in yl.predict(xb.cuda(), **kw)]
    for _ in range(5):
        ra = yl.predict(xa, **kw)                 # asynchronous: only enqueued
        rb = yl.predict(xb.cuda(), **kw)          # plain path, immediately behind it
        for r, want in zip(ra, ref_a):
            assert np.array_equal(r.boxes.data.cpu().numpy(), want)
        for r, want in zip(rb, ref_b):
            assert np.array_equal(r.boxes.data.cpu().numpy(), want)


def test_infer_nms_equals_infer_then_nms():
    """The in-plan NMS (one CUDA graph per step) returns exactly what infer() + ops.nms_padded() return."""
    import numpy as np
    import torch

    from oracle.weights import fill_state_dict_
    from yololite.nn.tasks import DetectionModel
    from yololite.utils import ops

    m = fill_state_dict_(DetectionModel("yolo11n.yaml", verbose=False)).eval().cuda()
    x = torch.rand(3, 3, 96, 64, generator=torch.Generator().manual_seed(3)).cuda()
    for kw in (dict(conf=0.001, iou=0.7), dict(conf=0.05, iou=0.45, classes=[0, 3, 7], max_det=50),
               dict(conf=0.001, iou=0.6, agnostic=True, multi_label=True)):
        y, _ = m.infer(x)
        d0, c0 = ops.nms_padded(y.clone(), kw.get("conf"), kw.get("iou"), kw.get("classes"), kw.get("agnostic", False),
                                kw.get("multi_label", False), kw.get("max_det", 300))
        d1, c1 = m.infer_nms(x, **kw)
        torch.cuda.synchronize()
        assert torch.equal(c0, c1), kw
        # single-label without a class list: the confidence filter runs inside the head convs (no filter kernel, no
        # class-score rows); everything else takes the two-kernel NMS on the full prediction
        key = (float(kw["conf"]), float(kw["iou"]), None if kw.get("classes") is None else tuple(kw["classes"]),
               bool(kw.get("agnostic", False)), bool(kw.get("multi_label", False)), int(kw.get("max_det", 300)), 30000, 7680.0)
        kinds = [md["kind"] for md in m._get_plan(x.shape, x.device, False, 0, key)[0].meta]
        fused = not kw.get("multi_label", False) and kw.get("classes") is None
        assert ("nms_select" in kinds and "nms_begin" in kinds and "nms" not in kinds) == fused, (kw, kinds[-4:])
        n = c0.tolist()
        for i in range(3):
            assert np.array_equal(d0[i, : n[i]].cpu().numpy(), d1[i, : n[i]].cpu().numpy()), (kw, i)
        # a second call with the same arguments replays the same plan (and must not depend on stale scratch)
        d2, c2 = m.infer_nms(x, **kw)
        torch.cuda.synchronize()
        assert torch.equal(c1, c2)


def test_fused_class_filter_tie_rules_match_the_score_path():
    """The class filter in the head-conv epilogue picks the best class from the LOGITS (one sigmoid per pixel); the
    reference's rule is `scores.max(1)` = the FIRST class whose SCORE is maximal.  Crafted class weights put exact ties
    (identical rows), near ties (rows whose logits differ by 1e-7 .. 1e-3: some round to the same score, some do not),
    saturated scores (logits > 5 and > 17, where all scores are 1.0) and far-negative logits into every pixel: the fused
    path must still equal `infer()` + `nms_padded()` (which reads the stored scores) bit for bit."""
    import numpy as np
    import torch

    from oracle.weights import fill_state_dict_
    from yololite.nn.tasks import DetectionModel
    from yololite.utils import ops

    m = fill_state_dict_(DetectionModel("yolo11n.yaml", verbose=False)).eval()
    det = m.model[-1]
    g = torch.Generator().manual_seed(11)
    with torch.no_grad():
        for lvl, seq in enumerate(det.cv3):
            w, b = seq[-1].weight, seq[-1].bias            # (nc, c3, 1, 1), (nc,)
            b.copy_(torch.randn(b.shape, generator=g) * 1.0 - 3.0)
            w[40], b[40] = w[12], b[12]                    # exact tie: class 12 must win over 40
            w[41], b[41] = w[12], b[12] + 1e-7             # near ties around the rounding width of the score
            w[42], b[42] = w[12], b[12] + 1e-6
            w[43], b[43] = w[12], b[12] + 1e-5
            w[5], b[5] = w[12], b[12] + 1e-4               # ... with the LARGER logit at the LOWER index as well
            w[44], b[44] = w[12], b[12] + 1e-3
            if lvl == 1:                                   # saturation: sigmoid(v) == 1.0f for both, first index wins
                b[20] = 30.0
                b[60] = 40.0
            if lvl == 2:                                   # scores in (sigmoid(5), 1): the slow path by rule
                b[33] = 9.0
                w[34], b[34] = w[33], b[33] + 2e-6
                b[70] = -120.0                             # e^-v overflows: score 0
    m = m.cuda()
    x = torch.rand(4, 3, 160, 96, generator=torch.Generator().manual_seed(5)).cuda()
    for conf in (0.001, 0.25, 0.9):
        y, _ = m.infer(x)
        d0, c0 = ops.nms_padded(y.clone(), conf, 0.7, None, False, False, 300)
        d1, c1 = m.infer_nms(x, conf=conf, iou=0.7)
        torch.cuda.synchronize()
        assert torch.equal(c0, c1), (conf, c0.tolist(), c1.tolist())
        assert int(c0.sum()) > 0
        for i, n in enumerate(c0.tolist()):
            assert np.array_equal(d0[i, :n].cpu().numpy(), d1[i, :n].cpu().numpy()), (conf, i)
    # the crafted classes are really what the detections carry (the test would be vacuous otherwise)
    cls = set(d1[..., 5].flatten().tolist())
    assert 12.0 in cls or 5.0 in cls or 20.0 in cls or 33.0 in cls, sorted(cls)[:10]


# ------------------------------------------------------------------------------------------------ benchmark shapes
def _oracle_forward_chunked(sd, x, chunk=16):
    from oracle import yolo11_ref

    return torch.cat([yolo11_ref.forward(sd, x[i:i + chunk])[0] for i in range(0, x.shape[0], chunk)], 0)


def test_model_bs64_matches_oracle_with_batch_dependent_dispatch(golden):
    """The benchmark's own shape (BASELINE config 3: yolo11n, 640x640, bs=64): conv dispatch that depends on the batch
    size — image-stacked 128-row tiles on the 20x20 maps, the wave-quantisation N split (148 < m_tiles <= 296), the halo-patch
    and resident-weight modes — is asserted to be taken, the head output is within tolerance of the fp32 oracle on all
    64 images and the NMS (both label modes) is bit-exact against the oracle on the same pre-NMS tensor."""
    from oracle import nms_ref
    from yololite.nn.tasks import DetectionModel

    g = golden("model_yolo11n.npz")
    sd = model_state_dict(g)
    m = DetectionModel("yolo11n.yaml", verbose=False)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    x = torch.rand(64, 3, 640, 640, generator=torch.Generator().manual_seed(3))
    xc = x.cuda()
    y, _ = m.infer(xc)
    assert tuple(y.shape) == (64, 84, 8400)
    plan = m._get_plan(xc.shape, xc.device)[0]
    disp = plan.conv_dispatch()
    assert len(disp) >= 40
    stacked = [d for d, i in disp if i.tile_n > 1]
    nsplit = [(d, i.m_tiles) for d, i in disp if i.n_tiles == 2 and i.co_tile <= 128]
    patch = [d for d, i in disp if i.patch]
    wres = [d for d, i in disp if i.wres]
    assert any("20x20" in d for d in stacked), "image-stacked tiles were not used on the 20x20 maps"
    assert len(nsplit) >= 8 and all(148 < mt <= 296 for _, mt in nsplit), f"N split not taken at bs=64: {nsplit}"
    assert patch and wres, (patch, wres)
    yr = _oracle_forward_chunked(sd, x).numpy()
    yc = y.cpu().numpy()
    assert np.abs(yc[:, :4] - yr[:, :4]).max() <= BOX_TOL_PX
    assert np.abs(yc[:, 4:] - yr[:, 4:]).max() <= SCORE_TOL
    # the whole step as the bench runs it (model + NMS in one plan / CUDA graph), against the oracle NMS on the SAME tensor
    for kw, multi in ((dict(conf_thres=0.25, iou_thres=0.7), False), (dict(conf_thres=0.001, iou_thres=0.7, multi_label=True), True)):
        dets, counts = m.infer_nms(xc, kw["conf_thres"], kw["iou_thres"], None, False, multi, 300)
        dets, counts = dets.cpu().numpy(), counts.cpu().numpy()
        ref = nms_ref.non_max_suppression(yc, max_det=300, **kw)
        assert list(counts) == [len(r) for r in ref]
        for i, r in enumerate(ref):
            np.testing.assert_array_equal(dets[i, : counts[i]], r, err_msg=f"image {i} multi={multi}")


@pytest.mark.parametrize("scale", ["s", "m"])
def test_model_s_m_640_match_oracle(golden, scale):
    """yolo11s / yolo11m at the benchmark resolution (640x640: K up to 4608, two N tiles, M = 1600 / 6400 per image),
    B = 2: head output within tolerance of the fp32 oracle, NMS bit-exact on the same tensor."""
    from oracle import nms_ref, yolo11_ref
    from yololite.nn.tasks import DetectionModel
    from yololite.utils import ops

    g = golden(f"model_yolo11{scale}.npz")
    sd = model_state_dict(g)
    m = DetectionModel(f"yolo11{scale}.yaml", verbose=False)
    m.load_state_dict(sd)
    m = m.cuda().eval()
    x = torch.rand(2, 3, 640, 640, generator=torch.Generator().manual_seed(5))
    yr, _ = yolo11_ref.forward(sd, x)
    y, _ = m.infer(x.cuda())
    yc = y.cpu().numpy()
    assert np.abs(yc[:, :4] - yr.numpy()[:, :4]).max() <= BOX_TOL_PX
    assert np.abs(yc[:, 4:] - yr.numpy()[:, 4:]).max() <= SCORE_TOL
    got = ops.non_max_suppression(y.clone(), conf_thres=0.05, iou_thres=0.7)
    ref = nms_ref.non_max_suppression(yc, conf_thres=0.05, iou_thres=0.7)
    for a, b in zip(got, ref):
        np.testing.assert_array_equal(a.cpu().numpy(), b)


# ------------------------------------------------------------------------------------------------ narrow ingest
@pytest.mark.parametrize("scale,hw", [("n", (64, 96)), ("n", (640, 640)), ("s", (64, 64))])
def test_uint8_and_fp16_ingest_equal_the_widened_fp32_batch(golden, scale, hw):
    """A uint8 image batch (bytes, /255 on ingest: predictor.py:83-84) and an fp16 batch give bit-identical outputs to
    the same values widened to fp32 first: inside the fused stem for yolo11n (no widened copy ever exists), through
    one conversion launch for the other scales."""
    from yololite import _C
    from yololite.nn.tasks import DetectionModel

    g = golden(f"model_yolo11{scale}.npz")
    m = DetectionModel(f"yolo11{scale}.yaml", verbose=False)
    m.load_state_dict(model_state_dict(g))
    m = m.cuda().eval()
    gen = torch.Generator().manual_seed(11)
    xu = torch.randint(0, 256, (3, 3, *hw), dtype=torch.uint8, generator=gen).cuda()
    y_ref = m.infer(xu.float() / 255)[0].clone()
    y_u8 = m.infer(xu)[0].clone()
    assert torch.equal(y_u8, y_ref)
    plan = m._get_plan(xu.shape, xu.device)[0]
    assert (_C.YL_U8 in plan.native_ingest) == (scale == "n")
    xh = (xu.float() / 255).half()
    assert torch.equal(m.infer(xh)[0], m.infer(xh.float())[0].clone())
    # a non-contiguous / unaligned uint8 batch takes the generic path and still means "bytes / 255"
    xs = torch.randint(0, 256, (3, 3, hw[0], hw[1] + 32), dtype=torch.uint8, generator=gen).cuda()[..., 16:16 + hw[1]]
    assert not xs.is_contiguous()
    assert torch.equal(m.infer(xs)[0].clone(), m.infer(xs.contiguous().float() / 255)[0])


def test_predict_uint8_host_tensor_matches_fp32_path(chunk_small_batches):
    """A pinned uint8 host batch (a quarter of the fp32 upload) through the chunk-pipelined predictor gives exactly the
    detections of the same images fed as fp32 / 255."""
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    xu = torch.randint(0, 256, (32, 3, 64, 64), dtype=torch.uint8, generator=torch.Generator().manual_seed(4)).pin_memory()
    kw = dict(imgsz=64, conf=0.001, verbose=False, device=0, batch=32)
    r8 = yl.predict(xu, **kw)
    assert yl.predictor._chunking(xu) == 4
    r32 = yl.predict((xu.float() / 255).pin_memory(), **kw)
    assert len(r8) == len(r32) == 32
    for a, b in zip(r8, r32):
        assert np.array_equal(a.boxes.data.cpu().numpy(), b.boxes.data.cpu().numpy())
    assert np.asarray(r8[0].orig_img).dtype == np.uint8 and np.asarray(r8[0].orig_img).shape == (64, 64, 3)


def test_predict_single_chunk_async_calls_alternate_lanes():
    """Small uploads are not chunked: every predict() is one asynchronous chunk and successive calls alternate between
    the two lanes / plan slots (two batches in flight); results read one call behind stay those of their own batch."""
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    g = torch.Generator().manual_seed(21)
    xs = [torch.randint(0, 256, (16, 3, 64, 64), dtype=torch.uint8, generator=g).pin_memory() for _ in range(3)]
    kw = dict(imgsz=64, conf=0.001, verbose=False, device=0, batch=16)
    want = [[r.boxes.data.cpu().numpy() for r in yl.predict(x.cuda(), **kw)] for x in xs]
    assert yl.predictor._chunking(xs[0]) == -1
    prev = None
    for it in range(7):
        res = yl.predict(xs[it % 3], **kw)
        if prev is not None:
            for r, w in zip(prev[1], want[prev[0]]):
                assert np.array_equal(r.boxes.data.cpu().numpy(), w)
        prev = (it % 3, res)
    assert yl.predictor.model.__dict__["_yl_pipe"]["next_lane"] in (0, 1)


def test_predict_alternating_batch_shapes_and_plan_cache_bound(chunk_small_batches):
    """ADVICE r1: (a) a full host batch followed by a partial one (and back) must not corrupt the earlier, still
    unread Results: staging states are kept per shape and side streams are drained before anything is freed;
    (b) the per-model plan cache is bounded (LRU) however many shapes / NMS settings stream through."""
    from oracle.weights import fill_state_dict_
    from yololite import YOLOLite

    yl = YOLOLite("yolo11n.yaml")
    fill_state_dict_(yl.model)
    g = torch.Generator().manual_seed(9)
    full = torch.rand(32, 3, 64, 64, generator=g).pin_memory()
    part = torch.rand(16, 3, 64, 64, generator=g).pin_memory()
    odd = torch.rand(16, 3, 96, 64, generator=g).pin_memory()
    kw = dict(imgsz=64, conf=0.001, verbose=False, device=0)
    want = {id(t): [r.boxes.data.cpu().numpy() for r in yl.predict(t, batch=len(t), **kw)] for t in (full, part)}
    want[id(odd)] = [r.boxes.data.cpu().numpy() for r in yl.predict(odd, batch=16, imgsz=(96, 64), conf=0.001, verbose=False, device=0)]
    for _ in range(3):
        pending = []
        for t in (full, part, odd, part, full):     # more shapes than pipeline_states slots would keep at 2
            kk = dict(kw, imgsz=(96, 64)) if t is odd else kw
            pending.append((t, yl.predict(t, batch=len(t), **kk)))      # asynchronous; read only afterwards
        for t, res in pending[-2:]:                  # the documented pattern: batch k-1 is read after submitting k
            for r, w in zip(res, want[id(t)]):
                assert np.array_equal(r.boxes.data.cpu().numpy(), w)
    model = yl.model
    model.max_plans = 4
    x = torch.rand(1, 3, 64, 64).cuda()
    for i in range(12):
        model.infer_nms(x, conf=0.01 + 0.01 * i, iou=0.7)
    assert len(model.__dict__["_yl_plans"]) <= 4
    d, c = model.infer_nms(x, conf=0.01, iou=0.7)    # evicted long ago: rebuilt, still correct
    y, _ = model.infer(x)
    from yololite.utils import ops

    d0, c0 = ops.nms_padded(y.clone(), 0.01, 0.7, None, False, False, 300)
    assert torch.equal(c, c0) and torch.equal(d[0, : int(c[0])], d0[0, : int(c0[0])])
    assert len(model.infer_nms(x, conf=0.3, iou=0.5, classes=0)) == 2          # an int `classes` is legal
