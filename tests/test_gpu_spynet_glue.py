"""Kernel-level checks of SPyNet's glue kernels and of the NCHW <-> NHWC layout kernels.

Inference runs SPyNet's pyramid, level inputs and final resize on these kernels only (training runs the same steps in
torch), so each is compared here with the same operation computed by torch in float64 on the device:

* `spynet_pyramid_base`: bilinear resize (align_corners=False) then (x - mean) / std, error <= 2^-20 * max(|ref|, 1);
  bit-exact to torch's fp32 (x - mean) / std when no resize is needed; channel 3 exactly 0;
* `avgpool2_c4`: each of five chained levels against fp64 avg_pool2d of its input, error <= 2^-22 * max(|ref|, 1);
* `spynet_level_input` (bf16, split-bf16 and fp32 layouts): flow_up = 2 * upsample(align_corners=True) of the previous
  flow (exactly 0 without one), the warped support frame against fp64 grid_sample(border, align_corners=True) at the
  coordinate-scaled bound of the warp tests, every stored channel bit-exact to the rounding of the fp32 values;
* `flow_resize`: bilinear resize (align_corners=False) times (w / Wp, h / Hp), error <= 2^-20 * max(|ref|, 1);
* `nchw_to_nhwc` / `nhwc_to_nchw`: bit-exact, padded channels 0, the 16-channel bf16 fast path equal to the generic kernel,
  and one size above the launch grid cap so that the grid-stride loops run.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from test_gpu_image_epilogues import bits, resize_ref, same_bits

pytestmark = pytest.mark.gpu

MEAN, STD = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from vsrlab_b200 import load
    load()
    return torch.device("cuda:0")


def gen_for(dev, *key):
    import zlib
    return torch.Generator(device=dev).manual_seed(zlib.crc32(repr(key).encode()))


def within(got, ref, rel, what):
    got = got.double()
    assert torch.isfinite(got).all().item(), f"{what}: values not finite (unwritten?)"
    bound = rel * max(ref.abs().max().item(), 1.0)
    err = (got - ref).abs().max().item()
    assert err <= bound, f"{what}: max err {err:.3g} > {bound:.3g}"


def sync():
    from vsrlab_b200 import ops
    torch.cuda.synchronize()
    assert ops.debug_status() == 0


# ----------------------------------------------------------------------------------------------------------------------
# pyramid base, avgpool, flow resize
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("h,w", [(180, 320), (33, 17), (1, 1), (64, 96)])
def test_pyramid_base(dev, h, w):
    from vsrlab_b200 import ops
    Fn = 3
    Hp, Wp = (h + 31) // 32 * 32, (w + 31) // 32 * 32
    frames = torch.rand(Fn, 3, h, w, generator=gen_for(dev, "pyr", h, w), device=dev)
    lvl = torch.full((Fn, Hp, Wp, 4), math.nan, device=dev)
    ops.spynet_pyramid_base(frames, lvl, Fn, h, w, Hp, Wp, MEAN, STD)
    sync()
    mean = torch.tensor(MEAN, dtype=torch.float64, device=dev).view(1, 3, 1, 1)
    std = torch.tensor(STD, dtype=torch.float64, device=dev).view(1, 3, 1, 1)
    ref = ((resize_ref(frames, Hp, Wp, False) - mean) / std).permute(0, 2, 3, 1)
    within(lvl[..., :3], ref, 2.0 ** -20, f"pyramid base {h}x{w} -> {Hp}x{Wp}")
    assert same_bits(lvl[..., 3], torch.zeros_like(lvl[..., 3]))
    if (Hp, Wp) == (h, w):
        t = (frames - mean.float()) / std.float()
        assert same_bits(lvl[..., :3], t.permute(0, 2, 3, 1).contiguous()), "not bit-exact to torch's fp32 normalisation"


@pytest.mark.parametrize("H,W", [(64, 96), (32, 32)])
def test_avgpool2_c4_chain(dev, H, W):
    from vsrlab_b200 import ops
    Fn = 3
    cur = torch.randn(Fn, H, W, 4, generator=gen_for(dev, "pool", H, W), device=dev)   # channel 3 non-zero on input
    for _ in range(5):
        nxt = torch.full((Fn, H // 2, W // 2, 4), math.nan, device=dev)
        ops.avgpool2_c4(cur, nxt, Fn, H, W)
        sync()
        ref = F.avg_pool2d(cur[..., :3].double().permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1)
        within(nxt[..., :3], ref, 2.0 ** -22, f"avgpool {H}x{W}")
        assert same_bits(nxt[..., 3], torch.zeros_like(nxt[..., 3]))
        cur, H, W = nxt, H // 2, W // 2


@pytest.mark.parametrize("Hp,Wp,h,w", [(192, 320, 180, 320), (64, 32, 33, 17), (32, 32, 1, 1)])
def test_flow_resize(dev, Hp, Wp, h, w):
    from vsrlab_b200 import ops
    P = 5
    fin = torch.randn(P, Hp, Wp, 2, generator=gen_for(dev, "resize", Hp, Wp, h, w), device=dev) * 3
    fout = torch.full((P, h, w, 2), math.nan, device=dev)
    ops.flow_resize(fin, fout, P, Hp, Wp, h, w)
    sync()
    ref = resize_ref(fin.permute(0, 3, 1, 2), h, w, False).permute(0, 2, 3, 1)
    ref = ref * torch.tensor([w / Wp, h / Hp], dtype=torch.float64, device=dev)
    within(fout, ref, 2.0 ** -20, f"flow_resize {Hp}x{Wp} -> {h}x{w}")


# ----------------------------------------------------------------------------------------------------------------------
# level input: [ref 3 | warped supp 3 | flow_up 2] in the three layouts
# ----------------------------------------------------------------------------------------------------------------------
def pair_indices(n, t, dev):
    from vsrlab_b200 import functional as VF
    return VF._pair_indices(n, t, dev)


@pytest.mark.parametrize("Hl,Wl", [(2, 2), (12, 20), (48, 80)])
@pytest.mark.parametrize("with_prev", [False, True])
def test_level_input(dev, Hl, Wl, with_prev):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16, BF16X2, F32
    n, t = 2, 4
    ref_idx, supp_idx = pair_indices(n, t, dev)                  # 12 pairs over 8 frames: frames are ref and supp
    P, Fn = ref_idx.numel(), n * t
    assert P != Fn
    g = gen_for(dev, "level", Hl, Wl, with_prev)
    lvl = torch.randn(Fn, Hl, Wl, 4, generator=g, device=dev)
    prev = (torch.randn(P, Hl // 2, Wl // 2, 2, generator=g, device=dev) * 3) if with_prev else None
    got = {}
    for dt, c_in in ((F32, 8), (BF16, 16), (BF16X2, 32)):
        fup = torch.full((P, Hl, Wl, 2), math.nan, device=dev)
        conv_in = torch.full((P, Hl, Wl, c_in), 7.0, dtype=torch.float32 if dt == F32 else torch.bfloat16, device=dev)
        ops.spynet_level_input(lvl, ref_idx, supp_idx, prev, fup, conv_in, P, Hl, Wl, c_in, dt)
        sync()
        got[dt] = (fup, conv_in)
    fup, v = got[F32]
    for dt in (BF16, BF16X2):
        assert same_bits(got[dt][0], fup), "flow_up depends on the layout"
    # flow_up
    if prev is None:
        assert same_bits(fup, torch.zeros_like(fup))
    else:
        ref_up = 2 * resize_ref(prev.permute(0, 3, 1, 2), Hl, Wl, True).permute(0, 2, 3, 1)
        within(fup, ref_up, 2.0 ** -20, "flow_up")
    # fp32 layout: the reference frame and flow_up exactly, the warped support frame against fp64 grid_sample
    li = ref_idx.long()
    assert same_bits(v[..., :3], lvl[li, ..., :3].contiguous())
    assert same_bits(v[..., 6:8], fup)
    supp = lvl[supp_idx.long(), ..., :3].double().permute(0, 3, 1, 2)
    gy, gx = torch.meshgrid(torch.arange(Hl, dtype=torch.float64, device=dev), torch.arange(Wl, dtype=torch.float64, device=dev),
                            indexing="ij")
    coords = torch.stack([gx + fup[..., 0].double(), gy + fup[..., 1].double()], -1)
    grid = torch.stack([2 * coords[..., 0] / max(Wl - 1, 1) - 1, 2 * coords[..., 1] / max(Hl - 1, 1) - 1], -1)
    warped = F.grid_sample(supp, grid, mode="bilinear", padding_mode="border", align_corners=True).permute(0, 2, 3, 1)
    tol = 5e-5 * (coords.abs().amax(dim=-1, keepdim=True) / 16).clamp_min(1.0)
    err = (v[..., 3:6].double() - warped).abs()
    assert (err <= tol).all().item(), f"warp: max err {err.max().item():.3g}, worst err/tol {(err / tol).max().item():.3g}"
    # bf16 / split layouts: the same values rounded, channels >= 8 (of each half) exactly 0
    vals = v[..., :8]
    hi = vals.to(torch.bfloat16)
    b16 = got[BF16][1]
    assert same_bits(b16[..., :8], hi) and same_bits(b16[..., 8:], torch.zeros_like(b16[..., 8:]))
    sp = got[BF16X2][1]
    assert same_bits(sp[..., :8], hi) and same_bits(sp[..., 16:24], (vals - hi.float()).to(torch.bfloat16))
    for z in (sp[..., 8:16], sp[..., 24:]):
        assert same_bits(z, torch.zeros_like(z))


# ----------------------------------------------------------------------------------------------------------------------
# layout kernels (bit-exact)
# ----------------------------------------------------------------------------------------------------------------------
def nhwc_expect(x, c_dst, dt):
    """What nchw_to_nhwc must store for fp32 [n, c, h, w] `x`."""
    from vsrlab_b200._lib import BF16, BF16X2
    n, c, h, w = x.shape
    v = x.permute(0, 2, 3, 1)
    if dt == BF16X2:
        e = torch.zeros(n, h, w, c_dst, dtype=torch.bfloat16, device=x.device)
        hi = v.to(torch.bfloat16)
        e[..., :c] = hi
        e[..., c_dst // 2:c_dst // 2 + c] = (v - hi.float()).to(torch.bfloat16)
        return e
    e = torch.zeros(n, h, w, c_dst, dtype=torch.bfloat16 if dt == BF16 else torch.float32, device=x.device)
    e[..., :c] = v.to(e.dtype)
    return e


LAYOUT_CASES = [
    # (dtype name, n, c, h, w, c_dst)
    ("f32", 3, 3, 17, 29, 4), ("f32", 2, 5, 9, 31, 12),
    ("bf16", 3, 3, 17, 29, 16),              # the 16-channel fast path
    ("bf16", 2, 5, 9, 31, 24), ("bf16", 2, 3, 1, 1, 8),
    ("bf16x2", 3, 3, 17, 29, 32), ("bf16x2", 2, 5, 9, 31, 48),
    ("bf16", 8, 3, 720, 1280, 16),           # 7.4 M pixels: more than the 148 * 32 blocks of 256 threads cover
    ("bf16x2", 8, 3, 720, 1280, 32),
]


def dtype_of(name):
    from vsrlab_b200._lib import BF16, BF16X2, F32
    return {"f32": F32, "bf16": BF16, "bf16x2": BF16X2}[name]


@pytest.mark.parametrize("name,n,c,h,w,c_dst", LAYOUT_CASES)
def test_nchw_to_nhwc(dev, name, n, c, h, w, c_dst):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16
    dt = dtype_of(name)
    x = torch.randn(n, c, h, w, generator=gen_for(dev, "n2n", name, n, c, h, w), device=dev) * 3
    exp = nhwc_expect(x, c_dst, dt)
    out = torch.full_like(exp, 7.0)
    ops.nchw_to_nhwc(x, out, n, c, h, w, c_dst, dt)
    sync()
    assert same_bits(out, exp)
    if dt == BF16 and c_dst == 16:
        # a destination that is not 16-byte aligned takes the generic kernel: it must store the same bits
        flat = torch.full((exp.numel() + 1,), 7.0, dtype=torch.bfloat16, device=dev)
        gen_out = flat[1:].view(exp.shape)
        ops.nchw_to_nhwc(x, gen_out, n, c, h, w, c_dst, dt)
        sync()
        assert same_bits(gen_out, out) and flat[0].item() == 7.0


@pytest.mark.parametrize("name,n,c,h,w,c_src", LAYOUT_CASES)
def test_nhwc_to_nchw(dev, name, n, c, h, w, c_src):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16X2, F32
    dt = dtype_of(name)
    g = gen_for(dev, "n2c", name, n, c, h, w)
    src = torch.randn(n, h, w, c_src, generator=g, device=dev)
    if dt == BF16X2:                             # lo parts of the size they have in a split tensor
        src[..., c_src // 2:] *= 2.0 ** -9
    src = src.to(torch.float32 if dt == F32 else torch.bfloat16)
    out = torch.full((n, c, h, w), math.nan, device=dev)
    ops.nhwc_to_nchw(src, out, n, c, h, w, c_src, dt)
    sync()
    if dt == BF16X2:
        exp = src[..., :c].float() + src[..., c_src // 2:c_src // 2 + c].float()
    else:
        exp = src[..., :c].float()
    assert same_bits(out, exp.permute(0, 3, 1, 2).contiguous())
