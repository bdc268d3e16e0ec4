"""flow_warp with every F.grid_sample mode (vsrb_flow_warp_ex / _ex_bwd, the drop-in flow_warp) against the reference
formula run by torch in fp64 on the same device: normalise the pixel grid x + flow with max(size-1, 1) whatever
align_corners is, then F.grid_sample(mode, padding_mode, align_corners).

Tolerances are those of the existing warp tests (fp32 5e-5 max-abs; bf16 2^-6 against bf16-rounded inputs, scaled by
max(|ref|, 1) for bicubic, whose outputs overshoot the inputs).  Those tests compare with an fp32 reference that rounds
the sample coordinate as the kernel does; against fp64 the kernel's fp32 coordinate itself is off by up to a few ulp
of |coordinate|, so the fp32 bound grows with it: 5e-5 * max(1, |coordinate| / 16) per pixel (about 2e-3 at the
+-500 px flows).  nearest is exact away from rounding ties."""
import itertools

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

MODES = ["bilinear", "nearest", "bicubic"]
PADS = ["zeros", "border", "reflection"]
COMBOS = list(itertools.product(MODES, PADS, [True, False]))


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from vsrlab_b200 import load
    load()
    return torch.device("cuda:0")


def bf16r(x):
    return x.to(torch.bfloat16).to(torch.float32)


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-12)).item()


def is_default(mode, pad, align):
    return mode == "bilinear" and pad != "reflection" and align


def ref_grid(flow, h, w):
    gy, gx = torch.meshgrid(torch.arange(h, dtype=flow.dtype, device=flow.device),
                            torch.arange(w, dtype=flow.dtype, device=flow.device), indexing="ij")
    px, py = gx + flow[..., 0], gy + flow[..., 1]
    return torch.stack((2.0 * px / max(w - 1, 1) - 1.0, 2.0 * py / max(h - 1, 1) - 1.0), dim=-1)


def ref_warp(x, flow, mode, pad, align):
    """the reference flow_warp (spynet.py:95-106) with the modes passed through"""
    return F.grid_sample(x, ref_grid(flow, x.shape[2], x.shape[3]), mode=mode, padding_mode=pad, align_corners=align)


def ref_coords(flow, h, w, align):
    """grid_sample's un-normalised sample coordinate (before padding), fp64 [n,h,w,2]"""
    g = ref_grid(flow, h, w)
    size = torch.tensor([w, h], dtype=g.dtype, device=g.device)
    return (g + 1) / 2 * (size - 1) if align else ((g + 1) * size - 1) / 2


def make_flow(kind, n, h, w, gen):
    shape = (n, h, w, 2)
    if kind == "rand20":
        return (torch.rand(shape, generator=gen) - 0.5) * 40
    if kind == "steps":                                  # integer and half-integer displacements
        return torch.randint(-16, 17, shape, generator=gen).float() / 2
    if kind == "far":                                    # +-500 px
        f = (torch.randint(0, 2, shape, generator=gen).float() * 2 - 1) * 500 + (torch.rand(shape, generator=gen) - 0.5) * 40
        f[0, 0, 0] = torch.tensor([500.0, -500.0])
        return f
    if kind == "bounce":                                 # up to three map sizes out: several reflections
        return (torch.rand(shape, generator=gen) - 0.5) * 6 * max(h, w)
    raise KeyError(kind)


SHAPES = [(2, 3, 19, 27), (1, 8, 1, 23), (2, 8, 17, 1), (1, 24, 7, 5), (1, 64, 13, 21)]
FLOWS = ["rand20", "steps", "far", "bounce"]


def check_forward(got, ref, coords, mode, prec, what):
    """got fp32 [n,c,h,w], ref fp64, coords fp64 [n,h,w,2] on the device"""
    got = got.double()
    if mode == "nearest":
        frac = coords - coords.floor()
        keep = ((frac - 0.5).abs() > 1e-3).all(dim=-1)[:, None].expand_as(ref)
        assert keep.float().mean().item() > 0.1, what
        bad = (got != ref) & keep
        assert not bad.any().item(), f"{what}: {bad.sum().item()} nearest samples differ"
        return
    if prec == "fp32":
        tol = 5e-5 * (coords.abs().amax(dim=-1) / 16).clamp_min(1.0)[:, None]
    else:
        tol = 2.0 ** -6 * (ref.abs().clamp_min(1.0) if mode == "bicubic" else torch.ones_like(ref))
    err = (got - ref).abs()
    assert (err <= tol).all().item(), f"{what}: max err {err.max().item():.3g}, worst err/tol {(err / tol).max().item():.3g}"


@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("mode,pad,align", COMBOS)
def test_forward_matches_grid_sample(dev, mode, pad, align, prec):
    from vsrlab.vsr.models.RealBasicVSR.modules.spynet import flow_warp
    from vsrlab_b200 import functional as VF
    gen = torch.Generator().manual_seed(7)
    for (n, c, h, w), kind in itertools.product(SHAPES, FLOWS):
        x = torch.randn(n, c, h, w, generator=gen)
        fl = make_flow(kind, n, h, w, gen)
        xd, fd = x.to(dev), fl.to(dev)
        with torch.no_grad():
            ref = ref_warp((bf16r(xd) if prec == "bf16" else xd).double(), fd.double(), mode, pad, align)
            with VF.precision(prec):
                got = flow_warp(xd, fd, mode, pad, align)
        assert got.shape == (n, c, h, w) and got.dtype == torch.float32
        check_forward(got, ref, ref_coords(fd.double(), h, w, align), mode, prec, f"{n}x{c}x{h}x{w} {kind}")


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("mode,pad,align", COMBOS)
def test_any_channel_count(dev, mode, pad, align, dtype):
    """24 channels straight through the autograd function (no padding to a power of two): the kernels' TPP = 0 path,
    forward and backward (dflow accumulated with atomics there)."""
    from vsrlab_b200 import autograd as AG
    from vsrlab_b200._lib import INTERP_BICUBIC, INTERP_BILINEAR, INTERP_NEAREST, PAD_BORDER, PAD_REFLECTION, PAD_ZEROS
    interp = {"bilinear": INTERP_BILINEAR, "nearest": INTERP_NEAREST, "bicubic": INTERP_BICUBIC}[mode]
    padding = {"zeros": PAD_ZEROS, "border": PAD_BORDER, "reflection": PAD_REFLECTION}[pad]
    gen = torch.Generator().manual_seed(13)
    x = bf16r(torch.randn(2, 24, 11, 13, generator=gen))
    fl = (torch.rand(2, 11, 13, 2, generator=gen) - 0.5) * 12
    gy = bf16r(torch.randn(2, 24, 11, 13, generator=gen))
    xr = x.double().to(dev).requires_grad_(True)
    fr = fl.double().to(dev).requires_grad_(True)
    ref = ref_warp(xr, fr, mode, pad, align)
    (ref * gy.double().to(dev)).sum().backward()
    xd = x.to(dev).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    fd = fl.to(dev).requires_grad_(True)
    out = AG.WarpExFn.apply(xd, fd, interp, padding, align)
    (out.float() * gy.to(dev)).sum().backward()
    prec = "bf16" if dtype == torch.bfloat16 else "fp32"
    check_forward(out.detach().float(), ref.detach(), ref_coords(fr.detach(), 11, 13, align), mode, prec, "c=24")
    bf = dtype == torch.bfloat16
    assert rel(xd.grad.float(), xr.grad) < (1e-2 if bf else 1e-5)
    if mode == "nearest":
        assert (fd.grad == 0).all().item()
    else:
        assert rel(fd.grad, fr.grad) < (2e-2 if bf else 1e-4)


@pytest.mark.parametrize("mode,pad,align", COMBOS)
def test_backward_through_dropin(dev, mode, pad, align):
    """dx and dflow of the drop-in flow_warp (fp32 data) against fp64 autograd of the reference formula."""
    from vsrlab.vsr.models.RealBasicVSR.modules.spynet import flow_warp
    gen = torch.Generator().manual_seed(11)
    shapes = [(2, 5, 17, 23), (1, 8, 7, 5)]
    if not is_default(mode, pad, align):
        # 1 x w and h x 1 maps: under align_corners the coordinate along the size-1 axis does not depend on the flow,
        # so torch's dflow there is 0.  The default mode runs the propagation kernel (flow_warp_bwd_kernel), which
        # returns a nonzero dflow on that axis and is left unchanged here.
        shapes += [(1, 8, 1, 19), (2, 3, 13, 1)]
    for n, c, h, w in shapes:
        x = bf16r(torch.randn(n, c, h, w, generator=gen))
        fl = (torch.rand(n, h, w, 2, generator=gen) - 0.5) * 12
        gy = bf16r(torch.randn(n, c, h, w, generator=gen))
        xr = x.double().to(dev).requires_grad_(True)
        fr = fl.double().to(dev).requires_grad_(True)
        (ref_warp(xr, fr, mode, pad, align) * gy.double().to(dev)).sum().backward()
        xd = x.to(dev).requires_grad_(True)
        fd = fl.to(dev).requires_grad_(True)
        (flow_warp(xd, fd, mode, pad, align) * gy.to(dev)).sum().backward()
        what = f"{n}x{c}x{h}x{w}"
        assert rel(xd.grad, xr.grad) < 1e-5, what
        if mode == "nearest":
            assert (fd.grad == 0).all().item(), what
        else:
            assert rel(fd.grad, fr.grad) < 1e-4, (what, rel(fd.grad, fr.grad))


@pytest.mark.parametrize("mode,pad,align", COMBOS)
def test_backward_bf16(dev, mode, pad, align):
    from vsrlab_b200 import autograd as AG
    from vsrlab_b200 import functional as VF
    gen = torch.Generator().manual_seed(17)
    x = bf16r(torch.randn(2, 64, 17, 23, generator=gen))
    fl = (torch.rand(2, 17, 23, 2, generator=gen) - 0.5) * 12
    gy = bf16r(torch.randn(2, 64, 17, 23, generator=gen))
    xr = x.double().to(dev).requires_grad_(True)
    fr = fl.double().to(dev).requires_grad_(True)
    (ref_warp(xr, fr, mode, pad, align) * gy.double().to(dev)).sum().backward()
    xd = x.to(dev).to(torch.bfloat16).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    fd = fl.to(dev).requires_grad_(True)
    out = AG.WarpExFn.apply(xd, fd, VF._WARP_INTERPS[mode], VF._WARP_PADS[pad], align)
    (out.float() * gy.to(dev)).sum().backward()
    assert rel(xd.grad.float(), xr.grad) < 1e-2
    if mode == "nearest":
        assert (fd.grad == 0).all().item()
    else:
        assert rel(fd.grad, fr.grad) < 2e-2


@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_default_mode_is_the_propagation_kernel(dev, pad):
    """(bilinear, zeros | border, align_corners): vsrb_flow_warp_ex and _ex_bwd give what vsrb_flow_warp / _bwd give,
    bit for bit (dx up to the order of its atomic additions)."""
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16, BF16X2, F32, INTERP_BILINEAR, PAD_BORDER, PAD_ZEROS
    padding = PAD_BORDER if pad == "border" else PAD_ZEROS
    gen = torch.Generator().manual_seed(5)
    n, h, w, c = 2, 45, 61, 64
    fl = ((torch.rand(n, h, w, 2, generator=gen) - 0.5) * 40).to(dev)
    fl[0, 0, 0] = torch.tensor([500.0, -500.0])
    for dt in (BF16, F32, BF16X2):
        x = torch.randn(n, h, w, c, generator=gen).to(dev).to(ops.TORCH_DT[dt])
        a, b = torch.empty_like(x), torch.empty_like(x)
        ops.flow_warp(x, fl, a, n, h, w, c, dt, padding)
        ops.flow_warp_ex(x, fl, b, n, h, w, c, dt, INTERP_BILINEAR, padding, True)
        assert torch.equal(a, b), dt
        if dt == BF16X2:
            continue
        dout = torch.randn(n, h, w, c, generator=gen).to(dev).to(ops.TORCH_DT[dt])
        dx_a, dx_b = torch.zeros(n, h, w, c, device=dev), torch.zeros(n, h, w, c, device=dev)
        df_a, df_b = torch.empty_like(fl), torch.empty_like(fl)
        ops.flow_warp_bwd(x, fl, dout, dx_a, df_a, n, h, w, c, dt, padding)
        ops.flow_warp_ex_bwd(x, fl, dout, dx_b, df_b, n, h, w, c, dt, INTERP_BILINEAR, padding, True)
        assert torch.equal(df_a, df_b), dt
        assert rel(dx_b, dx_a) < 1e-6, dt


@pytest.mark.parametrize("mode", MODES)
def test_non_finite_flows_do_not_fault(dev, mode):
    """inf / nan displacements next to ordinary ones: every launch completes and the ordinary pixels are unaffected
    (what a non-finite pixel itself yields is not specified)."""
    from vsrlab.vsr.models.RealBasicVSR.modules.spynet import flow_warp
    from vsrlab_b200 import functional as VF
    gen = torch.Generator().manual_seed(23)
    x = torch.randn(1, 8, 9, 11, generator=gen).to(dev)
    fl = (torch.rand(1, 9, 11, 2, generator=gen) - 0.5) * 10
    fl[0, 0, :4] = torch.tensor([[float("inf"), 0.0], [0.0, float("-inf")], [float("nan"), 1.0], [1e30, -1e30]])
    fl = fl.to(dev)
    finite = torch.isfinite(fl).all(dim=-1) & (fl.abs() < 1e6).all(dim=-1)
    for pad, align in itertools.product(PADS, [True, False]):
        with torch.no_grad(), VF.precision("fp32"):
            got = flow_warp(x, fl, mode, pad, align)
        torch.cuda.synchronize()
        ref = ref_warp(x.double(), torch.where(finite[..., None], fl, 0.0).double(), mode, pad, align)
        m = finite[:, None].expand_as(ref)
        check_forward(torch.where(m, got, 0.0), torch.where(m, ref, 0.0), ref_coords(torch.where(finite[..., None], fl, 0.0).double(),
                      9, 11, align), mode, "fp32", f"{pad} {align}")
