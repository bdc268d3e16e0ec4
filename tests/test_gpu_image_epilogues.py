"""Kernel-level checks of the image epilogues of `conv2d_fwd` against float64 references.

Three epilogues write the model's user-visible fp32 results, each from its own store code: EPI_SR (`sr = conv + bilinear(lq)`
in fp32, fp16 or uint8), EPI_CLEAN (the cleaner's fp32 frame updated in place plus its NHWC shadow) and EPI_FLOW (`flow_up +
relu(conv)` for every SPyNet level).  Each launch here is compared with the same operation computed by torch in float64 on
the device, from the same operands (bf16-rounded for the bf16 kernels, the fp32 values for the split-bf16 x3 mode and the
FFMA kernel):

* every mode: max-abs error <= 2e-5 * max(|ref|, 1) (fp32 outputs: only the summation order differs), every launched pixel
  finite (outputs start as NaN), the images before and after the launched batch slice bitwise unchanged;
* EPI_SR: the fp16 and uint8 outputs equal the fp32 output's `.half()` and `mul(255).add(0.5).clamp(0, 255)` bit for bit;
* EPI_CLEAN: the shadow holds bf16(x) (bf16), hi = bf16(x) and lo = bf16(x - hi) (split) or x (fp32) bit for bit, every
  other allocated channel exactly 0, and equals what `nchw_to_nhwc` makes of the new frame;
* EPI_FLOW: the CTA-pair and single-CTA kernels are bit-identical.

The shapes straddle the stacked tile width (30 columns for 3x3, 26 for 7x7) and the 4-row sub-tile, include odd tile counts
(the pair's dummy tile) and few CTAs (each CTA runs many tiles through both twin epilogue warps and the launcher picks two
sub-tiles per tile, the only launches that use the prefetched addend of the second sub-tile).
"""
import math
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

# the kernel selection switches of the conv launcher (VSRB_TC_NO_STACK is read at pack and at launch time)
SWITCHES = ("VSRB_RING_MIN_ROWS", "VSRB_TC_NO_RING", "VSRB_TC_NO_PAIR", "VSRB_TC_NO_STACK", "VSRB_RING_DEBUG",
            "VSRB_TC_DEBUG")
TOL = 2e-5
WORST = {}                                         # (epilogue, variant) -> worst error / bound, printed at the end


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from vsrlab_b200 import load
    load()
    yield torch.device("cuda:0")
    for k in sorted(WORST):
        print(f"worst error / bound {k[0]:6s} {k[1]:14s} {WORST[k]:.3f}")


def env(monkeypatch, **kv):
    """Clear every kernel switch, then set `kv`."""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in kv.items():
        monkeypatch.setenv(k, v)


def seed_of(*key):
    return zlib.crc32(repr(key).encode())


def bf16r(x):
    return x.to(torch.bfloat16).to(x.dtype)


def bits(t):
    """The raw bits of `t` (NaN-safe bitwise comparison)."""
    t = t.contiguous()
    return t.view({1: torch.uint8, 2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()])


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and torch.equal(bits(a), bits(b))


def variant(name):
    """kernel variant -> (activation dtype, kernel switches)"""
    from vsrlab_b200._lib import BF16, BF16X2, F32
    return {
        "bf16": (BF16, {}),                                    # stacked layout; 7x7 16->2: CTA pairs
        "bf16_single": (BF16, {"VSRB_TC_NO_PAIR": "1"}),
        "bf16_classic": (BF16, {"VSRB_TC_NO_STACK": "1"}),
        "x3": (BF16X2, {}),                                    # split-bf16 operands [hi | lo], fp32-accurate
        "ffma": (F32, {}),                                     # conv_f32_kernel
    }[name]


def make_convs(cin, cout, k, groups, gen, dev, bias_shift=0.0, wscale=1.0):
    convs = []
    for _ in range(groups):
        cv = torch.nn.Conv2d(cin, cout, k, 1, k // 2).to(dev)
        with torch.no_grad():
            cv.weight.copy_(torch.randn(cv.weight.shape, generator=gen, device=dev) * (wscale / (cin * k * k) ** 0.5))
            cv.bias.copy_(torch.randn(cv.bias.shape, generator=gen, device=dev) * 0.1 + bias_shift)
        convs.append(cv)
    return convs


def conv_ref(x, convs, dt, n):
    """float64 conv of image group g with convs[g]; bf16 operands for the bf16 kernels."""
    from vsrlab_b200._lib import BF16
    k = convs[0].kernel_size[0]
    outs = []
    for g, cv in enumerate(convs):
        xs, wt = x[g * n:(g + 1) * n], cv.weight.detach()
        if dt == BF16:
            xs, wt = bf16r(xs), bf16r(wt)
        outs.append(F.conv2d(xs.double(), wt.double(), cv.bias.detach().double(), padding=k // 2))
    return torch.cat(outs)


def operand(x, dt):
    """[B, c, h, w] fp32 -> the NHWC activation tensor of dtype `dt` (split-bf16: [hi Cp | lo Cp]) and its channel count."""
    from vsrlab_b200 import functional as VF, ops
    from vsrlab_b200._lib import BF16X2
    B, c, h, w = x.shape
    ca = VF._act_c(c, dt)
    t = torch.zeros(B, h, w, ca, dtype=ops.TORCH_DT[dt], device=x.device)
    v = x.permute(0, 2, 3, 1)
    if dt == BF16X2:
        hi = v.to(torch.bfloat16)
        t[..., :c] = hi
        t[..., ca // 2:ca // 2 + c] = (v - hi.float()).to(torch.bfloat16)
    else:
        t[..., :c] = v.to(t.dtype)
    return t, ca


def taps(out_size, in_size, align_corners, dev):
    """1-D bilinear source taps (i0, i1) and fp32 weight of the far tap, the way the kernels (and ATen's CUDA upsample)
    compute them: fp32 scale; with align_corners=False the source index is one fused multiply-add, rounded once."""
    f32 = lambda v: torch.tensor(v, dtype=torch.float32)
    o = torch.arange(out_size, dtype=torch.float64)
    if align_corners:
        scale = f32(in_size - 1) / f32(out_size - 1) if out_size > 1 else f32(0.0)
        src = (o * scale.double()).float()
    else:
        scale = f32(in_size) / f32(out_size)
        src = ((o + 0.5) * scale.double() - 0.5).float().clamp_min(0.0)
    i0 = src.floor().long().clamp_max(in_size - 1)
    i1 = (i0 + 1).clamp_max(in_size - 1)
    lam = src - i0.float()
    return i0.to(dev), i1.to(dev), lam.to(dev)


def resize_ref(x, H, W, align_corners):
    """Bilinear resize of [..., h, w] to (H, W): fp32 taps and weights, float64 blend."""
    y0, y1, ly = taps(H, x.shape[-2], align_corners, x.device)
    x0, x1, lx = taps(W, x.shape[-1], align_corners, x.device)
    q = x.double()
    hy, hx = (1 - ly).double().view(-1, 1), (1 - lx).double()
    ly, lx = ly.double().view(-1, 1), lx.double()
    rows = q[..., y0, :] * hy + q[..., y1, :] * ly
    return rows[..., x0] * hx + rows[..., x1] * lx


def close(got, ref, key, what):
    """max-abs error <= TOL * max(|ref|, 1), every value finite; records the worst ratio per (epilogue, variant)."""
    got = got.double()
    assert torch.isfinite(got).all().item(), f"{what}: {(~torch.isfinite(got)).sum().item()} values not finite (unwritten?)"
    bound = TOL * max(ref.abs().max().item(), 1.0)
    err = (got - ref).abs().max().item()
    WORST[key] = max(WORST.get(key, 0.0), err / bound)
    assert err <= bound, f"{what}: max err {err:.3g} > {bound:.3g}"


def launch(pc, *args, **kw):
    from vsrlab_b200 import ops
    ops.conv2d_fwd(pc, *args, **kw)
    torch.cuda.synchronize()
    assert ops.debug_status() == 0


# (images per group, h, w): widths around the stacked tile widths (30 / 26 columns), heights around the 4-row sub-tile,
# 1 to 5 images; odd tile counts for both kernel sizes
SMALL = [(1, 1, 1), (2, 4, 25), (3, 5, 26), (1, 9, 27), (5, 4, 30), (2, 9, 31), (3, 5, 61), (4, 1, 30), (1, 9, 61),
         (5, 5, 27)]
# each shape with one CTA per SM and with 1..3 CTAs
SMALL_CASES = [(s, mc) for i, s in enumerate(SMALL) for mc in (0, 1 + i % 3)]


def small_id(c):
    (n, h, w), mc = c
    return f"{n}x{h}x{w}_ctas{mc}"


# ----------------------------------------------------------------------------------------------------------------------
# EPI_SR: conv_last.2 (3x3 64 -> 3) + bilinear(lq), fp32 / fp16 / uint8
# ----------------------------------------------------------------------------------------------------------------------
SR_VARIANTS = ("bf16", "bf16_classic", "x3", "ffma")


def run_sr(monkeypatch, dev, name, n, h, w, aux, groups=1, max_ctas=0):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_NONE, CONV_SR_F16, CONV_SR_U8, EPI_SR
    dt, sw = variant(name)
    env(monkeypatch, **sw)
    gen = torch.Generator(device=dev).manual_seed(seed_of("sr", name, n, h, w, aux, groups, max_ctas))
    B = n * groups
    convs = make_convs(64, 3, 3, groups, gen, dev, wscale=0.5)
    x = torch.randn(B, 64, h, w, generator=gen, device=dev)
    lq_all = torch.rand(B + 2, 3, *aux, generator=gen, device=dev)         # guard images 0 and B + 1
    lq = lq_all[1:B + 1]
    ref = conv_ref(x, convs, dt, n) + resize_ref(lq, h, w, False)
    pc = ops.PackedConv(convs, [(0, 64)], dt)
    xin, ca = operand(x, dt)
    lq_before = lq_all.clone()
    outs = {}
    for kind, flag, tdt, fill in (("f32", 0, torch.float32, math.nan), ("f16", CONV_SR_F16, torch.float16, math.nan),
                                  ("u8", CONV_SR_U8, torch.uint8, 0xAB)):
        sr_all = torch.full((B + 2, 3, h, w), fill, dtype=tdt, device=dev)
        before = sr_all.clone()
        launch(pc, [xin], [ca], B, h, w, act=ACT_NONE, epilogue=EPI_SR, f32_io=sr_all[1:B + 1], f32_in=lq, aux_hw=aux,
               max_ctas=max_ctas, extra_flags=flag)
        assert same_bits(sr_all[0], before[0]) and same_bits(sr_all[-1], before[-1]), f"{kind}: guard image written"
        outs[kind] = sr_all[1:B + 1]
    assert same_bits(lq_all, lq_before)
    close(outs["f32"], ref, ("sr", name), f"EPI_SR {name} {B}x{h}x{w} aux {aux}")
    sr32 = outs["f32"]
    assert same_bits(outs["f16"], sr32.half()), "fp16 output != fp32 output .half()"
    u8 = sr32.mul(255).add(0.5).clamp(0, 255).to(torch.uint8)
    assert torch.equal(outs["u8"], u8), f"uint8 output differs at {(outs['u8'] != u8).sum().item()} values"
    return ref


@pytest.mark.parametrize("name", SR_VARIANTS)
@pytest.mark.parametrize("case", SMALL_CASES, ids=small_id)
def test_sr_small(dev, monkeypatch, name, case):
    (n, h, w), mc = case
    run_sr(monkeypatch, dev, name, n, h, w, ((h + 3) // 4, (w + 3) // 4), max_ctas=mc)


SR_MODEL = [
    # (images per group, h, w, aux, groups)
    (2, 256, 256, (64, 64), 1),            # x4 of the training crop
    (1, 720, 1280, (180, 320), 1),         # x4 of a 180 x 320 frame
    (2, 96, 128, (48, 64), 1),             # x2
    (1, 128, 160, (37, 53), 1),            # a non-integer ratio, which the C-ABI accepts
    (2, 64, 64, (16, 16), 2),              # two weight groups in one launch
]


@pytest.mark.parametrize("name", SR_VARIANTS)
@pytest.mark.parametrize("case", SR_MODEL, ids=lambda c: f"{c[0]}x{c[1]}x{c[2]}_aux{c[3][0]}x{c[3][1]}_g{c[4]}")
def test_sr_model_shapes(dev, monkeypatch, name, case):
    n, h, w, aux, groups = case
    ref = run_sr(monkeypatch, dev, name, n, h, w, aux, groups=groups)
    # uint8 coverage: the values span the clamp on both sides and the rounding in between
    assert (ref < 0).any().item() and (ref > 1).any().item() and ((ref > 0.1) & (ref < 0.9)).double().mean().item() > 0.2


def test_sr_x3_plan_is_stacked(dev):
    """The x3 conv_last.2 ([W_hi | W_lo]: two 64-channel weight segments) stays on the stacked layout, so its EPI_SR takes
    the 4-column prefetch path (EPI_SR never uses split stores).  Recorded so that a planner change shows up here."""
    import ctypes as C
    from vsrlab_b200 import _lib as L
    g = L.ConvGeom()
    g.kh = g.kw = 3
    g.n_seg = 2
    g.seg_off[0], g.seg_c[0], g.seg_off[1], g.seg_c[1] = 0, 64, 64, 64
    g.cout, g.groups, g.dtype = 3, 1, L.BF16
    info = (C.c_int32 * 8)()
    assert L.load().vsrb_conv_plan_info(C.byref(g), info) == 0
    assert (info[0], info[1], info[3]) == (1, 16, 48)


# ----------------------------------------------------------------------------------------------------------------------
# EPI_CLEAN: cleaner.conv (3x3 64 -> 3): x += conv in place, NHWC shadow of the new frame
# ----------------------------------------------------------------------------------------------------------------------
CLEAN_VARIANTS = [
    # (variant, out_c)
    ("bf16", 16),            # 16-byte shadow store, addend prefetched
    ("bf16", 8),             # store_n: the generic store
    ("bf16", 3),
    ("bf16_classic", 16),
    ("x3", 32),              # split shadow [hi 16 | lo 16]: the generic store
    ("ffma", 4),
    ("ffma", 16),
]


def run_clean(monkeypatch, dev, name, out_c, n, h, w, max_ctas=0):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_NONE, BF16, BF16X2, EPI_CLEAN
    dt, sw = variant(name)
    env(monkeypatch, **sw)
    gen = torch.Generator(device=dev).manual_seed(seed_of("clean", name, out_c, n, h, w, max_ctas))
    convs = make_convs(64, 3, 3, 1, gen, dev)
    x = torch.randn(n, 64, h, w, generator=gen, device=dev)
    x0_all = torch.randn(n + 2, 3, h, w, generator=gen, device=dev)
    x0 = x0_all[1:n + 1]
    ref = x0.double() + conv_ref(x, convs, dt, n)      # a tile added twice is off by a whole conv value
    pc = ops.PackedConv(convs, [(0, 64)], dt)
    xin, ca = operand(x, dt)
    tdt = ops.TORCH_DT[dt]
    out_all = torch.full((n + 2, h, w, out_c), 7.0, dtype=tdt, device=dev)
    io_before, out_before = x0_all.clone(), out_all.clone()
    launch(pc, [xin], [ca], n, h, w, act=ACT_NONE, epilogue=EPI_CLEAN, out=out_all[1:n + 1], out_c=out_c, f32_io=x0,
           max_ctas=max_ctas)
    for i in (0, -1):
        assert same_bits(x0_all[i], io_before[i]) and same_bits(out_all[i], out_before[i]), "guard image written"
    close(x0, ref, ("clean", f"{name}/{out_c}"), f"EPI_CLEAN {name} out_c={out_c} {n}x{h}x{w}")
    v = x0.permute(0, 2, 3, 1)
    sh = out_all[1:n + 1]
    zero = lambda t: same_bits(t, torch.zeros_like(t))
    if dt == BF16X2:
        hi = v.to(torch.bfloat16)
        assert same_bits(sh[..., :3], hi) and same_bits(sh[..., 16:19], (v - hi.float()).to(torch.bfloat16))
        assert zero(sh[..., 3:16]) and zero(sh[..., 19:])
    else:
        assert same_bits(sh[..., :3], v.to(tdt)) and zero(sh[..., 3:])
    conv = torch.full_like(sh, 7.0)
    ops.nchw_to_nhwc(x0, conv, n, 3, h, w, out_c, dt)
    torch.cuda.synchronize()
    assert same_bits(sh, conv), "shadow != nchw_to_nhwc(new frame)"


@pytest.mark.parametrize("name,out_c", CLEAN_VARIANTS, ids=lambda v: str(v))
@pytest.mark.parametrize("case", SMALL_CASES, ids=small_id)
def test_clean_small(dev, monkeypatch, name, out_c, case):
    (n, h, w), mc = case
    run_clean(monkeypatch, dev, name, out_c, n, h, w, max_ctas=mc)


@pytest.mark.parametrize("name,out_c", CLEAN_VARIANTS, ids=lambda v: str(v))
def test_clean_model_shape(dev, monkeypatch, name, out_c):
    run_clean(monkeypatch, dev, name, out_c, 30, 64, 64)        # one cleaner chunk: 30 frames of 64 x 64


# ----------------------------------------------------------------------------------------------------------------------
# EPI_FLOW: SPyNet's last conv (7x7 16 -> 2): flow = flow_up + relu(conv)
# ----------------------------------------------------------------------------------------------------------------------
FLOW_VARIANTS = ("bf16", "bf16_classic", "x3", "ffma")


def run_flow(monkeypatch, dev, name, n, h, w, groups=1, max_ctas=0):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_RELU, EPI_FLOW
    dt, sw = variant(name)
    env(monkeypatch, **sw)
    gen = torch.Generator(device=dev).manual_seed(seed_of("flow", name, n, h, w, groups, max_ctas))
    B = n * groups
    convs = make_convs(16, 2, 7, groups, gen, dev, bias_shift=-0.3)
    x = torch.randn(B, 16, h, w, generator=gen, device=dev)
    fu_all = torch.randn(B + 2, h, w, 2, generator=gen, device=dev) * 4
    fu = fu_all[1:B + 1]
    pre = conv_ref(x, convs, dt, n)
    if B * h * w >= 64:
        assert (pre < 0).double().mean().item() > 0.25              # the ReLU has work to do
    ref = fu.double() + pre.clamp_min(0).permute(0, 2, 3, 1)
    pc = ops.PackedConv(convs, [(0, 16)], dt)
    xin, ca = operand(x, dt)
    fu_before = fu_all.clone()

    def run():
        fl_all = torch.full((B + 2, h, w, 2), math.nan, device=dev)
        launch(pc, [xin], [ca], B, h, w, act=ACT_RELU, epilogue=EPI_FLOW, f32_in=fu, f32_io=fl_all[1:B + 1], max_ctas=max_ctas)
        assert torch.isnan(fl_all[0]).all().item() and torch.isnan(fl_all[-1]).all().item(), "guard image written"
        return fl_all[1:B + 1]
    fl = run()
    assert same_bits(fu_all, fu_before)
    close(fl, ref, ("flow", name), f"EPI_FLOW {name} {B}x{h}x{w}")
    if name == "bf16":                     # 7x7 16 -> 2 (N = 112) runs on CTA pairs; without them it must not change a bit
        monkeypatch.setenv("VSRB_TC_NO_PAIR", "1")
        single = run()
        close(single, ref, ("flow", "bf16_single"), f"EPI_FLOW bf16_single {B}x{h}x{w}")
        assert same_bits(single, fl), "single-CTA kernel != CTA-pair kernel"


@pytest.mark.parametrize("name", FLOW_VARIANTS)
@pytest.mark.parametrize("case", SMALL_CASES, ids=small_id)
def test_flow_small(dev, monkeypatch, name, case):
    (n, h, w), mc = case
    run_flow(monkeypatch, dev, name, n, h, w, max_ctas=mc)


FLOW_MODEL = [
    # (pairs per group, h, w, groups): every SPyNet level of a 180 x 320 input (padded to 192 x 320) with the 12 flow
    # pairs of a 7-frame clip, the 1 x 1 top level of an input no larger than 32 x 32, and two weight groups
    *[(12, 192 >> k, 320 >> k, 1) for k in range(5, -1, -1)],
    (12, 1, 1, 1),
    (3, 24, 40, 2),
]


@pytest.mark.parametrize("name", FLOW_VARIANTS)
@pytest.mark.parametrize("case", FLOW_MODEL, ids=lambda c: f"{c[0]}x{c[1]}x{c[2]}_g{c[3]}")
def test_flow_model_shapes(dev, monkeypatch, name, case):
    n, h, w, groups = case
    run_flow(monkeypatch, dev, name, n, h, w, groups=groups)


def test_flow_plan_takes_pairs(dev):
    """7x7 16 -> 2 is stacked with N = 112 (>= 96, N/2 a multiple of 8): the launcher runs it on CTA pairs."""
    import ctypes as C
    from vsrlab_b200 import _lib as L
    g = L.ConvGeom()
    g.kh = g.kw = 7
    g.n_seg = 1
    g.seg_c[0] = 16
    g.cout, g.groups, g.dtype = 2, 1, L.BF16
    info = (C.c_int32 * 8)()
    assert L.load().vsrb_conv_plan_info(C.byref(g), info) == 0
    assert (info[0], info[1], info[3]) == (1, 16, 112)
