"""GPU parity tests of the individual kernels, called through the C-ABI (ctypes) on torch CUDA buffers and
checked against plain PyTorch fp32 CPU restatements / the oracle.  Run with `pytest -m gpu` on a B200."""
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import test_conv_tc_paths_gpu as P

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ops():
    from yololite import _C, _ops

    _C.init(0)
    return _ops


def bf16r(t):
    return t.to(torch.bfloat16).float()


def nhwc(x_nchw, cstride=None, coff=0, dtype=torch.bfloat16):
    """NCHW fp32 CPU -> NHWC cuda buffer with `cstride` channels, data at [coff, coff+c); rest filled with junk."""
    n, c, h, w = x_nchw.shape
    cstride = cstride or c
    buf = torch.full((n, h, w, cstride), 7.5, dtype=dtype, device="cuda")
    buf[..., coff:coff + c] = x_nchw.permute(0, 2, 3, 1).to(dtype).cuda()
    return buf


CONV_CASES = [
    # ci, co, k, s, n, h, w, act, res, up, x_pad, y_pad, f32out, tag
    (64, 64, 1, 1, 2, 16, 16, True, False, False, 0, 0, False, "k1_sw128"),
    (32, 64, 1, 1, 2, 12, 12, True, False, False, 0, 0, False, "k1_sw64"),
    (16, 32, 1, 1, 1, 20, 20, True, False, False, 0, 0, False, "k1_sw32"),
    (48, 64, 1, 1, 2, 12, 12, True, False, False, 16, 64, False, "k1_ci48_slices"),
    (384, 256, 1, 1, 1, 20, 20, True, False, False, 0, 0, False, "k1_ci384_co256"),
    (256, 512, 1, 1, 1, 10, 10, True, False, False, 0, 0, False, "k1_co512_two_ntiles"),
    (64, 80, 1, 1, 1, 20, 20, False, False, False, 0, 64, True, "k1_co80_f32_bias_slice"),
    (128, 128, 1, 1, 1, 20, 20, False, True, False, 0, 0, False, "k1_residual_noact"),
    (64, 64, 3, 1, 2, 16, 16, True, False, False, 0, 0, False, "k3_s1"),
    (16, 8, 3, 1, 1, 24, 24, True, False, False, 0, 0, False, "k3_co8"),
    (8, 16, 3, 1, 1, 24, 24, True, True, False, 0, 16, False, "k3_ci8_res_slice"),
    (32, 32, 3, 1, 2, 20, 20, True, True, False, 32, 0, False, "k3_residual"),
    (128, 128, 3, 1, 1, 21, 21, True, False, False, 0, 0, False, "k3_ragged21"),
    (64, 64, 3, 1, 1, 12, 20, True, False, False, 0, 0, False, "k3_12x20"),
    (16, 32, 3, 2, 2, 32, 32, True, False, False, 0, 0, False, "k3_s2_sw32"),
    (64, 64, 3, 2, 1, 40, 40, True, False, False, 64, 0, False, "k3_s2_slice_in"),
    (128, 256, 3, 2, 1, 24, 40, True, False, False, 0, 128, False, "k3_s2_co256"),
    (256, 128, 1, 1, 1, 10, 10, True, False, True, 0, 128, False, "k1_upsample_into_concat"),
    (64, 64, 3, 1, 1, 8, 8, True, False, True, 0, 0, False, "k3_upsample"),
    (96, 48, 1, 1, 3, 20, 20, True, False, False, 0, 16, False, "k1_co48_chunk_tail"),
    (64, 144, 1, 1, 1, 20, 20, False, False, False, 0, 0, True, "k1_co144_f32_multichunk"),
    (64, 64, 3, 1, 9, 20, 20, True, True, False, 0, 64, False, "k3_20x20_stacked_images_res"),
    (32, 32, 1, 1, 5, 23, 17, True, True, False, 0, 0, False, "k1_flat_ragged_tail_res"),
    (128, 256, 3, 1, 2, 20, 20, True, False, False, 0, 0, False, "k3_co256_long_k"),
]

# the tcgen05 dispatch paths (test_conv_tc_paths_gpu.conv_paths) each case takes on a 148-SM B200
TC_PATHS = {
    "k1_sw128": {"epi0", "flat", "small_split"},
    "k1_sw64": {"epi0", "flat", "small_split"},
    "k1_sw32": {"epi0", "flat", "resident_weights"},
    "k1_ci48_slices": {"epi0", "flat", "small_split"},
    "k1_ci384_co256": {"epi0", "flat", "small_split"},
    "k1_co512_two_ntiles": {"epi0", "flat", "small_split"},
    "k1_co80_f32_bias_slice": {"epi7", "flat", "resident_weights", "f32_out"},
    "k1_residual_noact": {"epi3", "flat", "small_split"},
    "k3_s1": {"epi0", "patch_1cta", "patch_kblk64"},
    "k3_co8": {"cw16", "epi7", "patch_2cta", "patch_kblk16"},
    "k3_ci8_res_slice": {"cw16", "epi7", "patch_2cta", "patch_kblk16"},
    "k3_residual": {"epi1", "image_stack", "resident_weights"},
    "k3_ragged21": {"epi0", "small_split"},
    "k3_12x20": {"epi0", "patch_1cta", "patch_kblk64"},
    "k3_s2_sw32": {"epi0", "image_stack", "resident_weights", "stride2"},
    "k3_s2_slice_in": {"epi0", "small_split", "stride2"},
    "k3_s2_co256": {"epi0", "small_split", "stride2"},
    "k1_upsample_into_concat": {"epi0", "small_split", "upsample"},
    "k3_upsample": {"epi0", "small_split", "upsample"},
    "k1_co48_chunk_tail": {"epi0", "flat", "resident_weights"},
    "k1_co144_f32_multichunk": {"epi7", "flat", "resident_weights", "f32_out"},
    "k3_20x20_stacked_images_res": {"epi1", "image_stack", "small_split"},
    "k1_flat_ragged_tail_res": {"epi1", "flat", "resident_weights"},
    "k3_co256_long_k": {"epi0", "image_stack", "small_split"},
}

DUAL_CASES = [
    # ci, co, k, s, n, h, w, y_pad, up_pad, tag
    (256, 256, 1, 1, 2, 20, 20, 0, 128, "k1_dual_concat"),
    (64, 128, 3, 2, 3, 16, 24, 128, 64, "k3s2_dual_slices"),
    (32, 16, 3, 1, 1, 12, 12, 0, 0, "k3_dual_co16"),
]


@pytest.mark.parametrize("case", DUAL_CASES, ids=[c[-1] for c in DUAL_CASES])
@pytest.mark.parametrize("impl", ["tc", "direct"])
def test_conv_dual_destination(ops, case, impl):
    """y_up: the result is stored at conv resolution AND 2x2-replicated into a second buffer (Upsample fused)."""
    from yololite import _C

    ci, co, k, s, n, h, w, y_pad, up_pad, tag = case
    g = torch.Generator().manual_seed(zlib.crc32(tag.encode()) % 2**31)
    x = torch.randn(n, ci, h, w, generator=g)
    wt = torch.randn(co, ci, k, k, generator=g) * (1.5 / (ci * k * k) ** 0.5)
    bias = torch.randn(co, generator=g) * 0.1
    pc = ops.pack_conv(wt, bn=None, conv_bias=bias)
    ho, wo = (h + 2 * (k // 2) - k) // s + 1, (w + 2 * (k // 2) - k) // s + 1
    ref = F.silu(F.conv2d(bf16r(x), bf16r(wt), bias, s, k // 2))
    xv = ops.View(nhwc(x), 0, ci)
    yb = torch.full((n, ho, wo, co + y_pad), -3.0, dtype=torch.bfloat16, device="cuda")
    ub = torch.full((n, 2 * ho, 2 * wo, co + up_pad), -3.0, dtype=torch.bfloat16, device="cuda")
    yv, uv = ops.View(yb, y_pad // 2, co), ops.View(ub, up_pad // 2, co)
    ops.conv(xv, yv, pc, s, True, None, False, impl=_C.IMPL_TCGEN05 if impl == "tc" else _C.IMPL_DIRECT, y_up=uv)
    torch.cuda.synchronize()
    got = yv.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    got_up = uv.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=2e-2, atol=2e-2)
    np.testing.assert_array_equal(got_up.numpy(), F.interpolate(got, scale_factor=2.0, mode="nearest").numpy())
    for buf, pad in ((yb, y_pad), (ub, up_pad)):
        if pad:
            rest = torch.cat([buf[..., : pad // 2], buf[..., pad // 2 + co:]], -1)
            assert bool((rest == -3.0).all())


@pytest.mark.parametrize("case", CONV_CASES, ids=[c[-1] for c in CONV_CASES])
@pytest.mark.parametrize("impl", ["tc", "direct"])
def test_conv_bn_act(ops, case, impl):
    from yololite import _C

    ci, co, k, s, n, h, w, act, res, up, x_pad, y_pad, f32out, tag = case
    g = torch.Generator().manual_seed(zlib.crc32(tag.encode()) % 2**31)
    x = torch.randn(n, ci, h, w, generator=g)
    wt = torch.randn(co, ci, k, k, generator=g) * (1.5 / (ci * k * k) ** 0.5)
    gamma = torch.rand(co, generator=g) + 0.5
    beta = torch.randn(co, generator=g) * 0.1
    mean = torch.randn(co, generator=g) * 0.1
    var = torch.rand(co, generator=g) + 0.5
    eps = 1e-3
    pc = ops.pack_conv(wt, bn=(gamma, beta, mean, var, eps))
    # expected: folded weights rounded to bf16 exactly as the pack kernel stores them
    scale = gamma / torch.sqrt(var + eps)
    w_f = bf16r(wt * scale.view(-1, 1, 1, 1))
    b_f = beta - mean * scale
    ho, wo = (h + 2 * (k // 2) - k) // s + 1, (w + 2 * (k // 2) - k) // s + 1
    ref = F.conv2d(bf16r(x), w_f, b_f, s, k // 2)
    if act:
        ref = F.silu(ref)
    r_nchw = None
    if res:
        r_nchw = torch.randn(n, co, ho, wo, generator=g)
        ref = ref + bf16r(r_nchw)
    if up:
        ref = F.interpolate(ref, scale_factor=2.0, mode="nearest")

    xb = nhwc(x, ci + x_pad, x_pad // 2)
    xv = ops.View(xb, x_pad // 2, ci)
    u = 2 if up else 1
    ydt = torch.float32 if f32out else torch.bfloat16
    yb = torch.full((n, ho * u, wo * u, co + y_pad), -3.0, dtype=ydt, device="cuda")
    yv = ops.View(yb, y_pad // 2, co)
    rv = None
    if res:
        rb = nhwc(r_nchw, co + 8, 8)
        rv = ops.View(rb, 8, co)
    a = ops.conv_args(xv, yv, pc, s, act, rv, up)
    supported = bool(_C.load().yl_conv_tc_supported(a))
    if impl == "tc":
        assert supported, "case expected to run on the tcgen05 path"
        sms = torch.cuda.get_device_properties(0).multi_processor_count
        reached = P.conv_paths(P.plan_info(a), n, ho, wo, co, sms, res=res, f32=f32out, up=up, stride=s)
        assert sms != 148 or TC_PATHS[tag] <= reached, (tag, sorted(TC_PATHS[tag] - reached))
    ops.conv(xv, yv, pc, s, act, rv, up, impl=_C.IMPL_TCGEN05 if impl == "tc" else _C.IMPL_DIRECT)
    torch.cuda.synchronize()
    got = yv.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    if impl == "tc":
        # fp64 of the operands the kernel reads (packed weights and bias, bf16 input and residual), per-element bound
        w64, b64 = P.unpack_weights(pc)
        res64 = rv.torch_nhwc().cpu().double().permute(0, 3, 1, 2) if res else None
        ref64, pre, sabs = P.conv_reference(xv.torch_nhwc().cpu().double().permute(0, 3, 1, 2), w64, b64, s, act, res64,
                                            up)
        P.assert_within(got.double(), ref64, P.conv_bound(ref64, pre, sabs, not f32out, act), tag)
    else:
        tol = 1e-3 if f32out else 2e-2
        np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=tol, atol=tol)
    # untouched channels of the destination buffer keep their fill value (slice write discipline)
    if y_pad:
        rest = torch.cat([yb[..., : y_pad // 2], yb[..., y_pad // 2 + co:]], -1)
        assert bool((rest == -3.0).all())


def test_conv_stem_direct(ops):
    g = torch.Generator().manual_seed(3)
    x = torch.rand(2, 3, 64, 64, generator=g)
    wt = torch.randn(16, 3, 3, 3, generator=g) * 0.3
    pc = ops.pack_conv(wt, bn=(torch.ones(16), torch.zeros(16), torch.zeros(16), torch.ones(16), 0.0))
    xv = ops.new_buffer(2, 64, 64, 3)
    ops.nchw_to_nhwc(x.cuda(), xv)
    yv = ops.new_buffer(2, 32, 32, 16)
    ops.conv(xv, yv, pc, 2, True)
    torch.cuda.synchronize()
    ref = F.silu(F.conv2d(bf16r(x), bf16r(wt), None, 2, 1))
    got = yv.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("case", [
    # ci, co, n, h, w, act, y_pad, tag
    (3, 16, 2, 64, 64, True, 0, "rgb_co16"),
    (3, 32, 1, 96, 160, True, 32, "rgb_co32_slice_wide"),
    (3, 64, 2, 36, 70, True, 0, "rgb_co64_ragged_w"),
    (2, 16, 1, 34, 38, False, 0, "two_channel_noact"),
    (4, 48, 1, 40, 72, True, 0, "rgba_co48_k36"),
    (3, 16, 1, 35, 67, True, 0, "odd_hw"),
], ids=lambda c: c[-1])
def test_stem_conv_fused_ingest(ops, case):
    """yl_stem_conv (NCHW fp32 in, mma.sync im2col-in-registers) vs fp32 conv on bf16-rounded operands."""
    ci, co, n, h, w, act, y_pad, tag = case
    g = torch.Generator().manual_seed(zlib.crc32(tag.encode()) % 2**31)
    x = torch.rand(n, ci, h, w, generator=g)
    wt = torch.randn(co, ci, 3, 3, generator=g) * 0.4
    bn = (torch.rand(co, generator=g) + 0.5, torch.randn(co, generator=g) * 0.1, torch.randn(co, generator=g) * 0.1,
          torch.rand(co, generator=g) + 0.5, 1e-3)
    pc = ops.pack_conv(wt, bn=bn)
    scale = bn[0] / torch.sqrt(bn[3] + 1e-3)
    ref = F.conv2d(bf16r(x), bf16r(wt * scale.view(-1, 1, 1, 1)), bn[1] - bn[2] * scale, 2, 1)
    if act:
        ref = F.silu(ref)
    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    yb = torch.full((n, ho, wo, co + y_pad), -3.0, dtype=torch.bfloat16, device="cuda")
    yv = ops.View(yb, y_pad // 2, co)
    ops.stem_conv(x.cuda(), yv, pc, act)
    torch.cuda.synchronize()
    got = yv.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=2e-2, atol=2e-2)
    if y_pad:
        rest = torch.cat([yb[..., : y_pad // 2], yb[..., y_pad // 2 + co:]], -1)
        assert bool((rest == -3.0).all())


def test_layout_roundtrip(ops):
    x = torch.randn(2, 144, 9, 13)
    v = ops.new_buffer(2, 9, 13, 160)
    ops.nchw_to_nhwc(x.cuda(), v.slice(8, 144))
    back = ops.nhwc_to_nchw(v.slice(8, 144))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(back.cpu().numpy(), bf16r(x).numpy())


@pytest.mark.parametrize("shape", [(2, 80, 11, 13), (1, 64, 20, 20), (3, 128, 7, 4), (1, 8, 5, 1), (2, 256, 9, 18)],
                         ids=lambda s: "x".join(map(str, s)))
def test_dwconv3x3(ops, shape):
    g = torch.Generator().manual_seed(5)
    n, c, h, w = shape
    x = torch.randn(n, c, h, w, generator=g)
    wt = torch.randn(c, 1, 3, 3, generator=g) * 0.3
    bn = (torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g) * 0.1, torch.randn(c, generator=g) * 0.1,
          torch.rand(c, generator=g) + 0.5, 1e-3)
    pc = ops.pack_conv(wt, bn=bn)
    assert pc.depthwise
    scale = bn[0] / torch.sqrt(bn[3] + 1e-3)
    ref = F.silu(F.conv2d(bf16r(x), bf16r(wt * scale.view(-1, 1, 1, 1)), bn[1] - bn[2] * scale, 1, 1, 1, c))
    xv = ops.View(nhwc(x, c + 16, 8), 8, c)
    yv = ops.new_buffer(n, h, w, c)
    ops.conv(xv, yv, pc, 1, True)
    torch.cuda.synchronize()
    got = yv.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=2e-2, atol=2e-2)


@pytest.mark.parametrize("hw", [(20, 20), (9, 11), (21, 21), (40, 40)])
def test_sppf_pool(ops, hw):
    h, w = hw
    x = torch.randn(2, 64, h, w)
    cat = torch.full((2, h, w, 256), 1.0, dtype=torch.bfloat16, device="cuda")
    cat[..., :64] = x.permute(0, 2, 3, 1).to(torch.bfloat16).cuda()
    v = ops.View(cat, 0, 256)
    ops.sppf_pool(v.slice(0, 64), v.slice(64, 64), v.slice(128, 64), v.slice(192, 64), 5)
    torch.cuda.synchronize()
    y = [bf16r(x)]
    for _ in range(3):
        y.append(F.max_pool2d(y[-1], 5, 1, 2))
    ref = torch.cat(y, 1)
    np.testing.assert_array_equal(cat.float().cpu().permute(0, 3, 1, 2).numpy(), ref.numpy())


def test_upsample_and_copy(ops):
    x = torch.randn(2, 32, 5, 7)
    xv = ops.View(nhwc(x), 0, 32)
    yv = ops.new_buffer(2, 10, 14, 48)
    ops.upsample2x(xv, yv.slice(16, 32))
    cv = ops.new_buffer(2, 5, 7, 40)
    ops.copy_slice(xv, cv.slice(8, 32))
    torch.cuda.synchronize()
    ref = F.interpolate(bf16r(x), scale_factor=2.0, mode="nearest")
    np.testing.assert_array_equal(yv.slice(16, 32).torch_nhwc().float().cpu().permute(0, 3, 1, 2).numpy(), ref.numpy())
    np.testing.assert_array_equal(cv.slice(8, 32).torch_nhwc().float().cpu().permute(0, 3, 1, 2).numpy(), bf16r(x).numpy())


@pytest.mark.parametrize("shape", [(2, 2, 20, 20), (1, 4, 21, 21), (3, 2, 6, 7)])
def test_psa_attention(ops, shape):
    b, heads, h, w = shape
    kd, hd = 32, 64
    n = h * w
    g = torch.Generator().manual_seed(11)
    qkv = torch.randn(b, heads * (2 * kd + hd), h, w, generator=g)
    q, k, v = bf16r(qkv).view(b, heads, 2 * kd + hd, n).split([kd, kd, hd], dim=2)
    attn = ((q.transpose(-2, -1) @ k) * kd ** -0.5).softmax(-1)
    ref = (v @ attn.transpose(-2, -1)).view(b, heads * hd, h, w)
    qv = ops.View(nhwc(qkv), 0, heads * (2 * kd + hd))
    ov = ops.new_buffer(b, h, w, heads * hd)
    ops.attention(qv, ov, heads, kd, hd, kd ** -0.5)
    torch.cuda.synchronize()
    got = ov.torch_nhwc().float().cpu().permute(0, 3, 1, 2)
    np.testing.assert_allclose(got.numpy(), ref.numpy(), rtol=2e-2, atol=2e-2)


def test_detect_decode_matches_reference_fixture(ops, golden):
    from oracle import yolo11_ref

    g = golden("modules.npz")
    raws = [torch.from_numpy(g[f"detect.raw{i}"]) for i in range(3)]
    levels = [ops.View(nhwc(r, dtype=torch.float32), 0, 144) for r in raws]
    b = raws[0].shape[0]
    a = sum(r.shape[2] * r.shape[3] for r in raws)
    y = torch.empty((b, 84, a), dtype=torch.float32, device="cuda")
    ops.detect_decode(levels, (8.0, 16.0, 32.0), 16, 80, y)
    torch.cuda.synchronize()
    np.testing.assert_allclose(y.cpu().numpy(), g["detect.y"], rtol=1e-5, atol=1e-4)
    np.testing.assert_allclose(y.cpu().numpy(), yolo11_ref.decode(raws).numpy(), rtol=1e-5, atol=1e-4)


def test_detect_decode_640(ops):
    from oracle import yolo11_ref

    g = torch.Generator().manual_seed(2)
    raws = [torch.randn(2, 144, s, s, generator=g) * 2 for s in (80, 40, 20)]
    levels = [ops.View(nhwc(r, dtype=torch.float32), 0, 144) for r in raws]
    y = torch.empty((2, 84, 8400), dtype=torch.float32, device="cuda")
    ops.detect_decode(levels, (8.0, 16.0, 32.0), 16, 80, y)
    torch.cuda.synchronize()
    ref = yolo11_ref.decode(raws)
    np.testing.assert_allclose(y.cpu().numpy(), ref.numpy(), rtol=1e-5, atol=2e-4)
