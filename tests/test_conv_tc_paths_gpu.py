"""fp64 parity of every dispatch path of the tcgen05 conv (csrc/conv_tc.cu, plan_conv_tc) and of its Detect epilogues.

Each case names the paths it is for and asserts them through yl_conv_tc_info, so a change of the planner's thresholds
cannot silently move a case onto another path.  The reference takes the operands the kernel reads (the bf16 input as
stored, the packed weights read back and unpacked, the packed fp32 bias), so the GEMM and the epilogue are checked apart
from the BN fold, against a per-element bound derived from the arithmetic (`conv_bound`) rather than a flat tolerance.
`test_bound_rejects_wrong_results` (no GPU) shows that bound catches the errors a wrong tiling would make."""
import ctypes as C
import zlib
from dataclasses import dataclass

import pytest
import torch
import torch.nn.functional as F

FILL = -3.0          # destination channels around the written slice must keep it
SENTINEL = -777.0    # prediction entries a Detect epilogue must not write
Y_PAD = 16           # every destination is a slice [8, 8 + co) of a buffer with co + 16 channels

# Accumulation term of the bound, in units of S = |x| * |w| + |b| (the conv of the absolute values).  The bf16 x bf16
# products are exact in fp32; the tensor core adds them in fp32, one rounding (or truncation) of at most 2^-23 of
# the partial sum per 16-deep MMA step, and every partial sum is bounded by S.  K / 16 steps give at most
# K * 2^-27 * S, which is <= 2^-16 * S for K <= 2048 (every case here asserts that); the fp32 bias add adds 2^-24 * S.
C_ACC = 2.0 ** -16
MAX_K = 2048


def cdiv(a, b):
    return -(-a // b)


# ----------------------------------------------------------------------------------------------------------- reference
def unpack_weights(pc):
    """Packed bf16 [co_pad][k*k][ci_pad] (yl_fold_bn_pack) -> OIHW fp64 [co][ci][k][k], plus the fp64 bias."""
    k = pc.k
    w = pc.w.float().cpu().double().view(pc.co_pad, k, k, pc.ci_pad)[: pc.co, :, :, : pc.ci]
    return w.permute(0, 3, 1, 2).contiguous(), pc.bias.cpu().double()[: pc.co]


def conv_reference(x, w, b, stride, act, res=None, upsample=False):
    """fp64 conv of the operands as the kernel reads them.  Returns (ref, pre, S): the result, the pre-activation and
    S = |x| * |w| + |b|, all NCHW, at the destination's resolution."""
    pad = w.shape[-1] // 2
    pre = F.conv2d(x, w, b, stride, pad)
    s = F.conv2d(x.abs(), w.abs(), b.abs(), stride, pad)
    ref = pre * torch.sigmoid(pre) if act else pre.clone()
    if res is not None:
        ref = ref + res
    if upsample:
        ref, pre, s = (t.repeat_interleave(2, 2).repeat_interleave(2, 3) for t in (ref, pre, s))
    return ref, pre, s


def conv_bound(ref, pre, s, bf16_out, act):
    """Per-element bound on |kernel - ref|:
      - bf16 output: 2^-8 |ref| (rounding to 8 significant bits, including one flip of the last bit); an fp32 output
        keeps 2^-23 |ref| for the rounding of the epilogue arithmetic;
      - SiLU: 2^-11 |pre|.  The kernel computes h + h * tanh.approx(h) with h = pre / 2 (common.cuh), and
        tanh.approx has a relative error below 2^-10.9, so the error is at most |h| * 2^-10.9 <= 2^-11 |pre|;
      - accumulation: C_ACC * S."""
    tol = C_ACC * s + (2.0 ** -8 if bf16_out else 2.0 ** -23) * ref.abs()
    if act:
        tol = tol + 2.0 ** -11 * pre.abs()
    return tol


def bound_violations(got, ref, tol):
    return int(((got.double() - ref).abs() > tol).sum())


def assert_within(got, ref, tol, what):
    err = (got.double() - ref).abs()
    bad = err > tol
    if bool(bad.any()):
        i = tuple(int(v) for v in torch.nonzero(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; first at {i}: "
                             f"got {float(got[i])} ref {float(ref[i])} err {float(err[i]):.3g} "
                             f"bound {float(tol[i]):.3g}")


def test_bound_rejects_wrong_results():
    """The bound accepts the bf16-rounded fp64 result and rejects what a wrong K loop, M tiling or N tiling would make:
    a dropped input channel, a dropped 3x3 tap, a 128-pixel tile replaced by its neighbour, the channels of the second
    N tile shifted."""
    g = torch.Generator().manual_seed(11)
    ci, co, h, w = 64, 256, 16, 16   # 2 M tiles of 128 pixels, 2 N tiles of 128 channels
    x = torch.randn(1, ci, h, w, generator=g).to(torch.bfloat16).double()
    wt = (torch.randn(co, ci, 3, 3, generator=g) * (1.5 / (9 * ci) ** 0.5)).to(torch.bfloat16).double()
    b = (torch.randn(co, generator=g) * 0.1).double()
    ref, pre, s = conv_reference(x, wt, b, 1, True)
    tol = conv_bound(ref, pre, s, True, True)

    def bf16(t):
        return t.to(torch.bfloat16).double()

    assert bound_violations(bf16(ref), ref, tol) == 0
    x_drop = x.clone()
    x_drop[:, 37] = 0
    assert bound_violations(bf16(conv_reference(x_drop, wt, b, 1, True)[0]), ref, tol) > 0, "dropped input channel"
    w_drop = wt.clone()
    w_drop[:, :, 0, 2] = 0
    assert bound_violations(bf16(conv_reference(x, w_drop, b, 1, True)[0]), ref, tol) > 0, "dropped tap"
    px = bf16(ref).permute(0, 2, 3, 1).reshape(-1, co).clone()      # NHWC pixel rows = the M order of the GEMM
    px[128:256] = px[0:128]
    tile_swap = px.view(1, h, w, co).permute(0, 3, 1, 2)
    assert bound_violations(tile_swap, ref, tol) > 0, "M tile replaced by its neighbour"
    shifted = bf16(ref).clone()
    shifted[:, 128:] = torch.roll(shifted[:, 128:], 1, dims=1)
    assert bound_violations(shifted, ref, tol) > 0, "second N tile shifted"


# ---------------------------------------------------------------------------------------------------------- plan info
PLAN_FIELDS = ("flat", "patch", "wres", "tile_w", "tile_h", "tile_n", "m_tiles", "n_tiles", "co_tile", "kblk", "stages",
               "grid", "smem_bytes", "tmem_cols", "cw", "stg_sub", "epi_kind")


def plan_info(args):
    from yololite import _C

    info = _C.ConvTcPlan()
    _C.check(_C.load().yl_conv_tc_info(C.byref(args), C.byref(info)), "yl_conv_tc_info")
    return {k: int(getattr(info, k)) for k in PLAN_FIELDS}


def conv_paths(p, n, ho, wo, co, sms, *, res=False, f32=False, up=False, y_up=False, stride=1):
    """Names of the dispatch paths a plan `p` (plan_info) takes."""
    co16 = cdiv(co, 16) * 16
    m_est = cdiv(n * ho * wo, 128)
    total = p["m_tiles"] * p["n_tiles"]
    nchunks = cdiv(p["co_tile"], p["cw"])
    one_cta = p["tmem_cols"] > 256 or p["smem_bytes"] > 112 * 1024
    wave = p["n_tiles"] == 2 and 128 < co16 <= 256 and sms < m_est <= 2 * sms
    flags = {
        "flat": p["flat"],
        "patch_kblk16": p["patch"] and p["kblk"] == 16,
        "patch_kblk32": p["patch"] and p["kblk"] == 32,
        "patch_kblk64": p["patch"] and p["kblk"] == 64,
        "patch_1cta": p["patch"] and one_cta,
        "patch_2cta": p["patch"] and not one_cta,
        "resident_weights": p["wres"],
        "streamed_weights_one_ntile": not p["wres"] and not p["patch"] and p["n_tiles"] == 1,
        "image_stack": p["tile_n"] > 1 and n % p["tile_n"] == 0,
        "image_stack_ragged": p["tile_n"] > 1 and n % p["tile_n"] != 0,
        "image_stack_ragged_res": p["tile_n"] > 1 and n % p["tile_n"] != 0 and res,
        "wave_split": wave,
        "wave_split_partial_last_tile": wave and p["n_tiles"] * p["co_tile"] > co16,
        "partial_last_ntile": p["n_tiles"] * p["co_tile"] > co16,
        "small_split": p["n_tiles"] > cdiv(co16, 256) and m_est * p["n_tiles"] <= sms,
        "multi_tile_patch": p["patch"] and total >= 3 * p["grid"],
        "multi_tile": not p["patch"] and total >= 3 * p["grid"],
        "co_tile_gt128_bf16_512cols": p["co_tile"] > 128 and p["tmem_cols"] == 512 and p["epi_kind"] in (0, 1, 2, 3),
        "stg_sub2_ntiles": p["stg_sub"] == 2 and p["n_tiles"] > 1,
        "odd_nchunks_ntiles": p["n_tiles"] > 1 and nchunks % 2 == 1 and p["cw"] == 32 and not f32 and p["stg_sub"] == 1,
        "cw16": p["cw"] == 16,
        "f32_out": f32,
        "upsample": up,
        "y_up": y_up,
        "stride2": stride == 2,
    }
    for k in range(8):
        flags[f"epi{k}"] = p["epi_kind"] == k
    return {k for k, v in flags.items() if v}


# ------------------------------------------------------------------------------------------------------- conv cases
@dataclass(frozen=True)
class Case:
    ci: int
    co: int
    k: int
    s: int
    n: int
    h: int
    w: int
    act: bool = True
    res: bool = False
    up: bool = False
    y_up: bool = False
    f32: bool = False
    paths: tuple = ()


def _wave_n(h, w, sms):
    """A batch whose h*w maps make 1.5 waves of 128-pixel tiles (the wave-quantisation N split's range)."""
    return 3 * sms * 128 // (2 * h * w)


# tag -> Case factory of the SM count (the wave-split and multi-tile shapes are sized from it)
CASES = {
    "flat_co256_three_tiles_per_cta": lambda sms: Case(
        64, 256, 1, 1, cdiv(3 * sms * 128, 1600), 40, 40,
        paths=("flat", "multi_tile", "resident_weights", "co_tile_gt128_bf16_512cols", "epi0")),
    "flat_co256_silu_res_512cols": lambda sms: Case(
        128, 256, 1, 1, 8, 40, 40, res=True, paths=("flat", "co_tile_gt128_bf16_512cols", "epi1")),
    "k3s2_co256_res_noact_512cols": lambda sms: Case(
        64, 256, 3, 2, 24, 40, 40, act=False, res=True, paths=("stride2", "co_tile_gt128_bf16_512cols", "epi3")),
    "wave_co256": lambda sms: Case(
        16, 256, 1, 1, _wave_n(20, 20, sms), 20, 20, paths=("flat", "wave_split", "stg_sub2_ntiles", "epi0")),
    "wave_co192_res_odd_chunks": lambda sms: Case(
        64, 192, 1, 1, _wave_n(20, 20, sms), 20, 20, res=True, paths=("wave_split", "odd_nchunks_ntiles", "epi1")),
    "wave_co144_noact_partial_tile": lambda sms: Case(
        64, 144, 1, 1, _wave_n(20, 20, sms), 20, 20, act=False,
        paths=("wave_split", "wave_split_partial_last_tile", "odd_nchunks_ntiles", "epi2")),
    "two_ntiles_co288": lambda sms: Case(
        64, 288, 1, 1, 8, 40, 40, paths=("flat", "partial_last_ntile", "odd_nchunks_ntiles", "epi0")),
    "patch_kblk16": lambda sms: Case(16, 32, 3, 1, 2, 24, 24, paths=("patch_kblk16", "patch_2cta")),
    "patch_kblk32_three_tiles_per_cta_res": lambda sms: Case(
        24, 96, 3, 1, cdiv(3 * sms, 15), 40, 40, res=True,
        paths=("patch_kblk32", "patch_1cta", "multi_tile_patch", "epi1")),
    "patch_kblk64": lambda sms: Case(48, 32, 3, 1, 2, 16, 16, paths=("patch_kblk64", "patch_2cta")),
    "streamed_weights_one_ntile": lambda sms: Case(
        96, 128, 3, 1, 24, 20, 20, paths=("streamed_weights_one_ntile",)),
    "stack_ragged_res": lambda sms: Case(64, 64, 3, 1, 13, 5, 5, res=True, paths=("image_stack_ragged_res",)),
    "stack_ragged_k1s2": lambda sms: Case(64, 64, 1, 2, 13, 10, 10, paths=("image_stack_ragged", "stride2")),
    "stack_even": lambda sms: Case(32, 64, 3, 1, 10, 5, 5, paths=("image_stack",)),
    "small_split_co256": lambda sms: Case(64, 256, 1, 1, 1, 16, 16, paths=("small_split", "flat")),
    "cw16_bf16_generic": lambda sms: Case(32, 16, 3, 1, 2, 12, 12, paths=("cw16", "epi7")),
    "f32_out": lambda sms: Case(64, 80, 1, 1, 1, 20, 20, act=False, f32=True, paths=("f32_out", "epi7")),
    "upsample_into_slice": lambda sms: Case(128, 64, 1, 1, 2, 10, 10, up=True, paths=("upsample",)),
    "y_up_dual": lambda sms: Case(64, 128, 3, 2, 3, 16, 24, y_up=True, paths=("y_up", "stride2")),
}


@pytest.fixture(scope="module")
def ops():
    from yololite import _C, _ops

    _C.init(0)
    return _ops


@pytest.fixture(scope="module")
def sms(ops):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gen(tag):
    return torch.Generator().manual_seed(zlib.crc32(tag.encode()) % 2**31)


def setup_case(ops, tag, c):
    """Inputs, packed conv, destination buffers and the yl_conv_args of case `c` (nothing is launched)."""
    from yololite import _C

    g = _gen(tag)
    x = torch.randn(c.n, c.ci, c.h, c.w, generator=g)
    wt = torch.randn(c.co, c.ci, c.k, c.k, generator=g) * (1.5 / (c.ci * c.k * c.k) ** 0.5)
    bias = torch.randn(c.co, generator=g) * 0.1
    pc = ops.pack_conv(wt, bn=None, conv_bias=bias)
    ho, wo = (c.h + 2 * (c.k // 2) - c.k) // c.s + 1, (c.w + 2 * (c.k // 2) - c.k) // c.s + 1
    xb = torch.full((c.n, c.h, c.w, c.ci + 8), 7.5, dtype=torch.bfloat16, device="cuda")
    xb[..., 8:] = x.permute(0, 2, 3, 1).to(torch.bfloat16).cuda()
    t = dict(pc=pc, ho=ho, wo=wo, xb=xb, xv=ops.View(xb, 8, c.ci))
    u = 2 if c.up else 1
    t["yb"] = torch.full((c.n, ho * u, wo * u, c.co + Y_PAD), FILL, dtype=torch.float32 if c.f32 else torch.bfloat16,
                         device="cuda")
    t["yv"] = ops.View(t["yb"], Y_PAD // 2, c.co)
    t["rv"] = t["uv"] = None
    if c.res:
        t["rb"] = torch.randn(c.n, ho, wo, c.co, generator=g).to(torch.bfloat16).cuda()
        t["rv"] = ops.View(t["rb"], 0, c.co)
    if c.y_up:
        t["ub"] = torch.full((c.n, 2 * ho, 2 * wo, c.co + Y_PAD), FILL, dtype=torch.bfloat16, device="cuda")
        t["uv"] = ops.View(t["ub"], Y_PAD // 2, c.co)
    t["args"] = ops.conv_args(t["xv"], t["yv"], pc, c.s, c.act, t["rv"], c.up, impl=_C.IMPL_TCGEN05, y_up=t["uv"])
    return t


def case_paths(t, c, sms):
    return conv_paths(plan_info(t["args"]), c.n, t["ho"], t["wo"], c.co, sms, res=c.res, f32=c.f32, up=c.up,
                      y_up=c.y_up, stride=c.s)


def check_fill(buf, co, what):
    rest = torch.cat([buf[..., : Y_PAD // 2], buf[..., Y_PAD // 2 + co:]], -1)
    assert bool((rest == FILL).all()), f"{what}: channels around the destination slice were written"


@pytest.mark.gpu
@pytest.mark.parametrize("tag", list(CASES))
def test_conv_tc_path(ops, sms, tag):
    from yololite import _C

    c = CASES[tag](sms)
    assert c.ci * c.k * c.k <= MAX_K
    t = setup_case(ops, tag, c)
    reached = case_paths(t, c, sms)
    missing = set(c.paths) - reached
    assert not missing, f"{tag} no longer takes {sorted(missing)}: plan {plan_info(t['args'])}"
    _C.check(_C.load().yl_conv_bn_act(C.byref(t["args"]), _C.stream_ptr()), "yl_conv_bn_act")
    torch.cuda.synchronize()

    w64, b64 = unpack_weights(t["pc"])
    x64 = t["xv"].torch_nhwc().cpu().double().permute(0, 3, 1, 2)
    res = t["rv"].torch_nhwc().cpu().double().permute(0, 3, 1, 2) if c.res else None
    ref, pre, s = conv_reference(x64, w64, b64, c.s, c.act, res, c.up)
    tol = conv_bound(ref, pre, s, not c.f32, c.act)
    got = t["yv"].torch_nhwc().cpu().double().permute(0, 3, 1, 2)
    assert_within(got, ref, tol, tag)
    check_fill(t["yb"], c.co, tag)
    if c.y_up:
        got_up = t["uv"].torch_nhwc().cpu().double().permute(0, 3, 1, 2)
        assert torch.equal(got_up, got.repeat_interleave(2, 2).repeat_interleave(2, 3)), f"{tag}: y_up"
        check_fill(t["ub"], c.co, f"{tag} y_up")


# ------------------------------------------------------------------------------------- invariance across batch sizes
INV_LAYER = dict(ci=128, co=256, k=3, h=8, w=8)   # 3x3 on thin maps: no halo patch (ci > 64), stacks images


def _inv_batches(sms):
    """batch -> the paths it must take: small N split, image stack + small split, one 256-wide N tile, wave split."""
    return {1: {"small_split"}, 13: {"small_split", "image_stack_ragged"}, 160: {"co_tile_gt128_bf16_512cols"},
            3 * sms * 128 // (2 * 64): {"wave_split"}}


def inv_setup(ops):
    """The layer and five images of the invariance test; run(batch) launches it on images 0..4 repeated to `batch` and
    returns (output, plan), plan(batch) only plans it."""
    from yololite import _C

    L = INV_LAYER
    g = _gen("invariance")
    imgs = torch.randn(5, L["h"], L["w"], L["ci"], generator=g).to(torch.bfloat16).cuda()
    wt = torch.randn(L["co"], L["ci"], 3, 3, generator=g) * (1.5 / (9 * L["ci"]) ** 0.5)
    pc = ops.pack_conv(wt, bn=None, conv_bias=torch.randn(L["co"], generator=g) * 0.1)

    def args(xb):
        yb = torch.full((xb.shape[0], L["h"], L["w"], L["co"]), FILL, dtype=torch.bfloat16, device="cuda")
        a = ops.conv_args(ops.View(xb, 0, L["ci"]), ops.View(yb, 0, L["co"]), pc, 1, True, impl=_C.IMPL_TCGEN05)
        return a, yb

    def plan(batch):
        return plan_info(args(imgs[torch.arange(batch) % 5].contiguous())[0])

    def run(xb):
        a, yb = args(xb)
        launch(a)
        return yb, plan_info(a)

    return imgs, plan, run


@pytest.mark.gpu
def test_conv_tc_batch_invariance(ops, sms):
    """The same layer on the same images gives bitwise the same output at batch sizes that take different paths.  The
    planner changes only the M / N tiling: every output element is still one dot product in the tap-major,
    channel-block-minor K order, with the same epilogue instantiation (asserted), so nothing may differ."""
    L = INV_LAYER
    imgs, _, run = inv_setup(ops)
    single = [run(imgs[i:i + 1].contiguous()) for i in range(5)]    # bs = 1, one launch per image
    p1 = single[0][1]
    for batch, want in _inv_batches(sms).items():
        yb, p = run(imgs[torch.arange(batch) % 5].contiguous()) if batch > 1 else single[0]
        reached = conv_paths(p, batch, L["h"], L["w"], L["co"], sms)
        assert want <= reached, f"bs={batch} no longer takes {sorted(want - reached)}: plan {p}"
        assert p["epi_kind"] == p1["epi_kind"] == 0, (batch, p)
        torch.cuda.synchronize()
        for b in range(batch):
            ref = single[b % 5][0][0]
            if not torch.equal(yb[b], ref):
                raise AssertionError(
                    f"image {b % 5} differs at bs={batch} (n_tiles {p['n_tiles']}, co_tile {p['co_tile']}, tile_n "
                    f"{p['tile_n']}) from bs=1 (n_tiles {p1['n_tiles']}, co_tile {p1['co_tile']}) in "
                    f"{int((yb[b] != ref).sum())} elements: the accumulation of an output element depends on the N "
                    f"tile width or the image stack, which the fixed K order does not allow")


# ------------------------------------------------------------------------------------------------ Detect epilogues
REG_MAX = 16


def det_level(ops, tag, n, h, w, co, ci=64, bias_shift=0.0, zero_images=()):
    """A 1x1 head conv (ci -> co) on an n x h x w map: bf16 input, packed conv, fp64 logits and their S."""
    g = _gen(tag)
    x = torch.randn(n, ci, h, w, generator=g)
    for i in zero_images:
        x[i] = 0
    wt = torch.randn(co, ci, 1, 1, generator=g) * (2.0 / ci ** 0.5)
    bias = torch.randn(co, generator=g) * 0.1 + bias_shift
    pc = ops.pack_conv(wt, bn=None, conv_bias=bias)
    xb = x.permute(0, 2, 3, 1).to(torch.bfloat16).cuda().contiguous()
    w64, b64 = unpack_weights(pc)
    x64 = xb.cpu().double().permute(0, 3, 1, 2)
    logits = F.conv2d(x64, w64, b64)
    s = F.conv2d(x64.abs(), w64.abs(), b64.abs())
    return dict(pc=pc, xb=xb, xv=ops.View(xb, 0, ci), logits=logits, s=s, n=n, h=h, w=w, co=co)


def det_args(ops, lv, pred, mode, nc, anchor0, stride, store, conf=0.0, cand_ws=None):
    from yololite import _C

    n, h, w, co = lv["n"], lv["h"], lv["w"], lv["co"]
    if store:
        lv["yb"] = torch.full((n, h, w, co + Y_PAD), FILL, dtype=torch.float32, device="cuda")
        yv = ops.View(lv["yb"], Y_PAD // 2, co)
    else:
        yv = ops.NoOutput(n, h, w, co)
    det = ops.DetEpilogue(pred, mode, REG_MAX, nc, anchor0, stride, conf=conf, cand_ws=cand_ws)
    lv["yv"] = yv
    return ops.conv_args(lv["xv"], yv, lv["pc"], 1, False, impl=_C.IMPL_TCGEN05, det=det)


def plain_plan_paths(ops, lv, sms):
    """Paths of the same conv without a Detect epilogue (an fp32 NHWC store): the N splits it would take."""
    from yololite import _C

    yb = torch.empty((lv["n"], lv["h"], lv["w"], lv["co"]), dtype=torch.float32, device="cuda")
    args = ops.conv_args(lv["xv"], ops.View(yb, 0, lv["co"]), lv["pc"], 1, False, impl=_C.IMPL_TCGEN05)
    return conv_paths(plan_info(args), lv["n"], lv["h"], lv["w"], lv["co"], sms)


def det_paths(ops, p, lv, sms, mode, store):
    """Paths of a Detect-epilogue plan `p`.  A Detect conv always runs as one N tile (the planner does not split it);
    the `_one_ntile_at_*_shape` names mark shapes where the same conv without the epilogue is split."""
    from yololite import _C

    assert p["n_tiles"] == 1, f"a Detect epilogue must run as one N tile: plan {p}"
    out = {f"det_epi{p['epi_kind']}"}
    names = {_C.DET_BOX: "box", _C.DET_CLS: "cls", _C.DET_CLS_FILTER: "cls_filter"}
    out.add(f"det_{names[mode]}" + ("_raw_stored" if store else ""))
    if p["cw"] == 16:
        out.add(f"det_{names[mode]}_cw16")
    out |= {f"det_{names[mode]}_one_ntile_at_{k}_shape" for k in plain_plan_paths(ops, lv, sms) & {"small_split",
                                                                                                     "wave_split"}}
    return out


def launch(args):
    from yololite import _C

    _C.check(_C.load().yl_conv_bn_act(C.byref(args), _C.stream_ptr()), "yl_conv_bn_act")


def check_raw(lv, store, tag):
    if not store:
        return
    got = lv["yv"].torch_nhwc().cpu().double().permute(0, 3, 1, 2)
    assert_within(got, lv["logits"], conv_bound(lv["logits"], lv["logits"], lv["s"], False, False), f"{tag} raw map")
    check_fill(lv["yb"], lv["co"], f"{tag} raw map")


def check_untouched(pred, rows, a0, a1, what):
    """Only rows `rows` of anchors [a0, a1) may differ from the sentinel."""
    keep = torch.ones(pred.shape[1:], dtype=torch.bool)
    keep[rows, a0:a1] = False
    assert bool((pred[:, keep] == SENTINEL).all()), f"{what}: entries outside the written window changed"


def box_reference(lv, stride):
    """DFL (softmax expectation over 16 bins per side) + dist2bbox around the anchor centre, * stride, in fp64, with a
    per-element px bound.  A side's distance is an expectation over bins 0..15, whose derivative by the logit of bin j
    is p_j (j - d), so a logit error of at most e moves it by at most 15 e; __expf and __fdividef add relative errors of
    a few 2^-22 to the weights and the quotient (at most 2^-17 px of distance).  Each output is a sum / difference of
    two distances (scaled by the stride) plus the fp32 rounding of the anchor arithmetic (2^-20 of the coordinate
    range)."""
    n, h, w = lv["n"], lv["h"], lv["w"]
    lg = lv["logits"].view(n, 4, REG_MAX, h * w)
    e = (C_ACC * lv["s"]).view(n, 4, REG_MAX, h * w).amax(2)
    dist = (torch.softmax(lg, 2) * torch.arange(REG_MAX, dtype=torch.float64).view(1, 1, -1, 1)).sum(2)
    dtol = 15 * e + 2.0 ** -17
    al = torch.arange(h * w)
    ax, ay = (al % w).double() + 0.5, (al // w).double() + 0.5
    x1, y1, x2, y2 = ax - dist[:, 0], ay - dist[:, 1], ax + dist[:, 2], ay + dist[:, 3]
    ref = torch.stack([(x1 + x2) / 2, (y1 + y2) / 2, x2 - x1, y2 - y1], 1) * stride
    tol = torch.stack([(dtol[:, 0] + dtol[:, 2]) / 2, (dtol[:, 1] + dtol[:, 3]) / 2, dtol[:, 0] + dtol[:, 2],
                       dtol[:, 1] + dtol[:, 3]], 1) * stride + 2.0 ** -20 * stride * max(h, w)
    return ref, tol


def sigmoid_bound(lv):
    """sigmoid' <= 1/4 scales the logit error; __expf / __fdividef add at most 2^-19 absolute to a value in (0, 1)."""
    return 0.25 * C_ACC * lv["s"] + 2.0 ** -19


@pytest.mark.gpu
@pytest.mark.parametrize("store", [False, True], ids=["no_raw", "raw_stored"])
def test_det_box_epilogue(ops, sms, store):
    from yololite import _C

    nc, h, w, stride, a0 = 80, 12, 20, 16.0, 37
    lv = det_level(ops, "det_box", 2, h, w, 4 * REG_MAX)
    A = a0 + h * w + 29
    pred = torch.full((2, 4 + nc, A), SENTINEL, dtype=torch.float32, device="cuda")
    args = det_args(ops, lv, pred, _C.DET_BOX, nc, a0, stride, store)
    p = plan_info(args)
    assert {"det_box" + ("_raw_stored" if store else ""), "det_epi7" if store else "det_epi4"} <= \
        det_paths(ops, p, lv, sms, _C.DET_BOX, store), p
    launch(args)
    torch.cuda.synchronize()
    pc = pred.cpu()
    ref, tol = box_reference(lv, stride)
    assert_within(pc[:, :4, a0:a0 + h * w].double(), ref, tol, "box decode")
    check_untouched(pc, slice(0, 4), a0, a0 + h * w, "box decode")
    check_raw(lv, store, "box decode")


DET_NC = [8, 16, 24, 40, 64, 80, 128, 192, 256]


def cls_level(ops, sms, nc, batch):
    """bs = 1 on a 40x40 map (13 tiles: a plain conv takes the small N split for nc % 64 == 0), or a 20x20 map at a
    batch in the wave-split range (a plain conv takes the wave split for 128 < nc <= 256)."""
    if batch == "bs1":
        return det_level(ops, f"cls{nc}_bs1", 1, 40, 40, nc)
    return det_level(ops, f"cls{nc}_wave", _wave_n(20, 20, sms), 20, 20, nc)


@pytest.mark.gpu
@pytest.mark.parametrize("store", [False, True], ids=["no_raw", "raw_stored"])
@pytest.mark.parametrize("batch", ["bs1", "wave"])
@pytest.mark.parametrize("nc", DET_NC)
def test_det_cls_epilogue(ops, sms, nc, batch, store):
    """Sigmoid of the class logits into rows 4 .. 4 + nc of anchors [anchor0, anchor0 + h*w) of a wider prediction, also
    at the shapes where a conv without the epilogue is split into N tiles (the decode addresses rows by the chunk index
    inside its tile, so the class conv must stay one N tile there)."""
    from yololite import _C

    lv = cls_level(ops, sms, nc, batch)
    n, hw, a0 = lv["n"], lv["h"] * lv["w"], 53
    A = a0 + hw + 19
    pred = torch.full((n, 4 + nc, A), SENTINEL, dtype=torch.float32, device="cuda")
    args = det_args(ops, lv, pred, _C.DET_CLS, nc, a0, 8.0, store)
    p = plan_info(args)
    reached = det_paths(ops, p, lv, sms, _C.DET_CLS, store)
    if batch == "bs1" and nc % 64 == 0:
        assert "det_cls_one_ntile_at_small_split_shape" in reached, p
    if batch == "wave" and nc > 128:
        assert "det_cls_one_ntile_at_wave_split_shape" in reached, p
    launch(args)
    torch.cuda.synchronize()
    pc = pred.cpu()
    ref = torch.sigmoid(lv["logits"]).view(n, nc, hw)
    assert_within(pc[:, 4:, a0:a0 + hw].double(), ref, sigmoid_bound(lv).view(n, nc, hw),
                  f"class decode nc={nc} {batch} (plan n_tiles {p['n_tiles']} co_tile {p['co_tile']})")
    check_untouched(pc, slice(4, 4 + nc), a0, a0 + hw, "class decode")
    check_raw(lv, store, f"class decode nc={nc}")


# two levels whose maps are not multiples of 128 pixels (tiles straddle images); image 1 has no candidate
FILTER_LEVELS = ((12, 10, 8.0), (5, 6, 16.0))
FILTER_B, FILTER_NC, FILTER_CONF, FILTER_IOU = 3, 80, 0.25, 0.45


def filter_setup(ops):
    lvs, a0 = [], 0
    for i, (h, w, st) in enumerate(FILTER_LEVELS):
        lv = det_level(ops, f"filter{i}", FILTER_B, h, w, FILTER_NC, bias_shift=-6.0, zero_images=(1,))
        lv["a0"], lv["stride"] = a0, st
        a0 += h * w
        lvs.append(lv)
    return lvs, a0


@pytest.mark.gpu
def test_det_cls_filter_epilogue(ops, sms):
    """yl_nms_begin + the class-filter convs of two levels + yl_nms_select are bit-identical to the class decode of the
    same convs followed by yl_nms_batched(multi_label = 0)."""
    from yololite import _C

    lib = _C.load()
    lvs, A = filter_setup(ops)
    B, nc = FILTER_B, FILTER_NC
    g = _gen("filter_boxes")
    boxes = torch.cat([torch.rand(B, 2, A, generator=g) * 320, torch.rand(B, 2, A, generator=g) * 76 + 4], 1)
    preds = []
    for _ in range(2):
        pr = torch.full((B, 4 + nc, A), SENTINEL, dtype=torch.float32, device="cuda")
        pr[:, :4] = boxes.cuda()
        preds.append(pr)
    ws_bytes = int(lib.yl_nms_workspace_bytes(B, A, nc, 0))
    max_det, max_nms, max_wh, s = 300, 30000, 7680.0, _C.stream_ptr()
    outs = [(torch.zeros((B, max_det, 6), dtype=torch.float32, device="cuda"),
             torch.full((B,), -1, dtype=torch.int32, device="cuda"),
             torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")) for _ in range(2)]
    # class decode + the whole NMS
    for lv in lvs:
        launch(det_args(ops, lv, preds[0], _C.DET_CLS, nc, lv["a0"], lv["stride"], False))
    out, cnt, ws = outs[0]
    _C.check(lib.yl_nms_batched(preds[0].data_ptr(), B, nc, A, FILTER_CONF, FILTER_IOU, None, 0, 0, 0, max_det, max_nms,
                                max_wh, ws.data_ptr(), ws_bytes, out.data_ptr(), cnt.data_ptr(), s), "yl_nms_batched")
    # class filter in the conv epilogue
    out, cnt, ws = outs[1]
    _C.check(lib.yl_nms_begin(ws.data_ptr(), ws_bytes, B, s), "yl_nms_begin")
    for lv in lvs:
        args = det_args(ops, lv, preds[1], _C.DET_CLS_FILTER, nc, lv["a0"], lv["stride"], False, conf=FILTER_CONF,
                        cand_ws=ws)
        p = plan_info(args)
        assert "det_epi6" in det_paths(ops, p, lv, sms, _C.DET_CLS_FILTER, False), p
        launch(args)
    _C.check(lib.yl_nms_select(preds[1].data_ptr(), B, nc, A, FILTER_IOU, 0, max_det, max_nms, max_wh, ws.data_ptr(),
                               ws_bytes, out.data_ptr(), cnt.data_ptr(), s), "yl_nms_select")
    torch.cuda.synchronize()
    (o0, c0, _), (o1, c1, _) = outs
    c0, c1 = c0.cpu(), c1.cpu()
    assert torch.equal(c0, c1), (c0, c1)
    assert int(c0[1]) == 0 and int(c0[0]) > 0 and int(c0[2]) > 0, c0
    for b in range(B):
        assert torch.equal(o0[b, : int(c0[b])].cpu(), o1[b, : int(c1[b])].cpu()), f"image {b}"
    assert bool((preds[1][:, 4:].cpu() == SENTINEL).all()), "the class filter wrote class rows"


# ------------------------------------------------------------------------------------------------------ coverage
ALL_PATHS = {
    "flat", "patch_kblk16", "patch_kblk32", "patch_kblk64", "patch_1cta", "patch_2cta", "resident_weights",
    "streamed_weights_one_ntile", "image_stack", "image_stack_ragged", "image_stack_ragged_res", "wave_split",
    "wave_split_partial_last_tile", "partial_last_ntile", "small_split", "multi_tile_patch", "multi_tile",
    "co_tile_gt128_bf16_512cols", "stg_sub2_ntiles", "odd_nchunks_ntiles", "cw16", "f32_out", "upsample", "y_up",
    "stride2",
    "epi0", "epi1", "epi2", "epi3", "epi7",
    "det_box", "det_box_raw_stored", "det_cls", "det_cls_raw_stored", "det_cls_filter", "det_epi4", "det_epi5",
    "det_epi6", "det_epi7", "det_cls_one_ntile_at_small_split_shape",
    "det_cls_one_ntile_at_wave_split_shape", "det_cls_cw16",
}


@pytest.mark.gpu
def test_conv_tc_path_coverage(ops, sms):
    """Every dispatch path of plan_conv_tc listed in ALL_PATHS is taken by at least one parity case of this file (the
    plans of all cases, collected through yl_conv_tc_info; nothing is launched)."""
    from yololite import _C

    reached = set()
    for tag, make in CASES.items():
        c = make(sms)
        reached |= case_paths(setup_case(ops, tag, c), c, sms) & set(c.paths)
    _, plan, _ = inv_setup(ops)
    for batch in _inv_batches(sms):
        reached |= conv_paths(plan(batch), batch, INV_LAYER["h"], INV_LAYER["w"], INV_LAYER["co"], sms)
    def det(lv, pred, mode, nc, a0, stride, store, **kw):
        p = plan_info(det_args(ops, lv, pred, mode, nc, a0, stride, store, **kw))
        return det_paths(ops, p, lv, sms, mode, store)

    for store in (False, True):
        lv = det_level(ops, "det_box", 2, 12, 20, 4 * REG_MAX)
        pred = torch.empty((2, 4 + 80, 12 * 20 + 66), dtype=torch.float32, device="cuda")
        reached |= det(lv, pred, _C.DET_BOX, 80, 37, 16.0, store)
        for nc in DET_NC:
            for batch in ("bs1", "wave"):
                lv = cls_level(ops, sms, nc, batch)
                pred = torch.empty((lv["n"], 4 + nc, lv["h"] * lv["w"] + 72), dtype=torch.float32, device="cuda")
                reached |= det(lv, pred, _C.DET_CLS, nc, 53, 8.0, store)
    lvs, A = filter_setup(ops)
    pred = torch.empty((FILTER_B, 4 + FILTER_NC, A), dtype=torch.float32, device="cuda")
    ws = torch.empty(int(_C.load().yl_nms_workspace_bytes(FILTER_B, A, FILTER_NC, 0)), dtype=torch.uint8, device="cuda")
    for lv in lvs:
        reached |= det(lv, pred, _C.DET_CLS_FILTER, FILTER_NC, lv["a0"], lv["stride"], False, conf=FILTER_CONF,
                       cand_ws=ws)
    missing = ALL_PATHS - reached
    assert not missing, f"paths no case reaches: {sorted(missing)}"
