"""torch.use_deterministic_algorithms(True) on the training path: fixed-order weight / bias gradients, warp backward, loss
and metric sums (the *_det entry points), matrix resizes in the torch glue, and torch-style refusals of the ops without a
deterministic implementation.

Kernel bounds are those of the default kernels' tests against fp64 torch on the same bf16 operands: dW max-abs <= 1e-3 *
max|ref|, dB rel-L2 <= 1e-4 (test_gpu_backward_kernels.py); warp dx / dflow the bounds of
test_gpu_training.py::test_warp_gradients.  Every deterministic result must also be bitwise equal across two launches."""
import ctypes as C
import os
import subprocess
import sys
import textwrap
import warnings
import zlib
from pathlib import Path

import pytest
import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
CL = torch.channels_last
E_ARG = -1
FAKE = 1 << 20                                          # non-null, 16-byte aligned placeholder address, never read


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from vsrlab_b200 import load
    load()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def lib():
    from vsrlab_b200 import build, _lib
    build.build()
    return _lib.load()


@pytest.fixture
def det():
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(False)


@pytest.fixture
def poisoned_ws(monkeypatch):
    """Every workspace of the *_det entry points starts as all-ones bytes (NaN as fp32 and as fp64): a slot the kernels
    failed to write would show up as NaN in the result rather than be summed from memory that happened to be zero."""
    from vsrlab_b200 import ops
    real = ops._workspace

    def poisoned(nbytes, what, device):
        return real(nbytes, what, device).fill_(255)
    monkeypatch.setattr(ops, "_workspace", poisoned)


def bf16r(x):
    return x.to(torch.bfloat16).to(x.dtype)


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def maxabs(a, b):
    return (a.double() - b.double()).abs().max().item()


def randn(shape, gen, dev, scale=1.0):
    return bf16r(torch.randn(shape, generator=gen, device=dev) * scale)


def nhwc(x, c_alloc, fill=0.0):
    B, c, h, w = x.shape
    t = torch.full((B, c_alloc, h, w), fill, dtype=torch.bfloat16, device=x.device).contiguous(memory_format=CL)
    t[:, :c] = x
    return t


def geom_of(segs, cout, k=3):
    from vsrlab_b200 import autograd as AG
    return AG._wgrad_geom(torch.nn.Conv2d(sum(c for _, c in segs), cout, k, 1, k // 2), tuple(segs))


# ----------------------------------------------------------------------------------------------------------------------
# argument checks (no GPU): refused with VSRB_E_ARG and a message before the device is touched
# ----------------------------------------------------------------------------------------------------------------------
def test_det_entry_points_refuse_bad_arguments(lib):
    from vsrlab_b200 import _lib as L
    ptrs = (C.c_void_p * 2)(FAKE, None)
    cs = (C.c_int32 * 2)(16, 0)
    g = geom_of([(0, 16)], 16)
    g.kw = 1                                            # 3x1: the FFMA fallback, which has no deterministic variant
    assert lib.vsrb_conv2d_wgrad_det(C.byref(g), ptrs, cs, FAKE, 16, 1, 8, 8, 1, 16, FAKE, None, FAKE, 1 << 20, None) == E_ARG
    assert b"deterministic" in lib.vsrb_last_error()
    g.dtype, g.kw = L.F32, 3
    assert lib.vsrb_conv2d_wgrad_det(C.byref(g), ptrs, cs, FAKE, 16, 1, 8, 8, 1, 16, FAKE, None, FAKE, 1 << 20, None) == E_ARG
    g = geom_of([(0, 32)], 64)                          # multi: tensor-core shapes only
    assert lib.vsrb_conv2d_wgrad_multi_det(C.byref(g), 2, (C.c_void_p * 2)(FAKE, FAKE), (C.c_int32 * 1)(32),
                                           (C.c_void_p * 2)(FAKE, FAKE), 64, 1, 8, 8, 32, FAKE, None, FAKE, 1 << 20, None) == E_ARG
    assert lib.vsrb_conv2d_wgrad_det_workspace_bytes(None, 1, 1, 8, 8, 0) == 0
    # warp: workspace too small / unaligned / missing, reflection, a flow gradient over a non-power-of-two lane group
    need = lib.vsrb_flow_warp_bwd_det_workspace_bytes(2, 8, 8, 64)
    assert need == 16 + 2 * 8 * 8 * 64 * 8
    args = (FAKE, FAKE, FAKE, FAKE, None, 2, 8, 8, 64, L.BF16)
    assert lib.vsrb_flow_warp_bwd_det(*args, L.PAD_ZEROS, FAKE, need - 1, None) == E_ARG
    assert b"workspace" in lib.vsrb_last_error()
    assert lib.vsrb_flow_warp_bwd_det(*args, L.PAD_ZEROS, FAKE + 8, need, None) == E_ARG
    assert lib.vsrb_flow_warp_bwd_det(*args, L.PAD_ZEROS, None, need, None) == E_ARG
    assert lib.vsrb_flow_warp_bwd_det(*args, L.PAD_REFLECTION, FAKE, need, None) == E_ARG
    assert lib.vsrb_flow_warp_bwd_det(FAKE, FAKE, FAKE, None, FAKE, 2, 8, 8, 24, L.BF16, L.PAD_ZEROS, None, 0, None) == E_ARG
    assert b"power of two" in lib.vsrb_last_error()
    assert lib.vsrb_flow_warp_bwd_det(FAKE, FAKE, FAKE, FAKE, None, 2, 8, 8, 6, L.F32, L.PAD_ZEROS, FAKE, need, None) == E_ARG
    assert lib.vsrb_flow_warp_bwd_det_workspace_bytes(0, 8, 8, 64) == 0
    # loss / metric sums: a workspace below the query's size
    nb = lib.vsrb_charbonnier_det_workspace_bytes(1 << 20)
    assert nb > 0 and nb % 8 == 0
    assert lib.vsrb_charbonnier_det(FAKE, FAKE, 1 << 20, 1e-9, FAKE, None, None, 1.0, FAKE, nb - 8, None) == E_ARG
    assert lib.vsrb_charbonnier_resized_det(FAKE, FAKE, 3, 8, 8, 32, 32, 1e-9, FAKE, None, None, 1.0, None, 1 << 20, None) == E_ARG
    assert lib.vsrb_psnr_sums_det(FAKE, FAKE, 2, 100, FAKE, FAKE, lib.vsrb_psnr_sums_det_workspace_bytes(2, 100) - 8, None) == E_ARG
    assert lib.vsrb_ssim_sums_det_workspace_bytes(1, 3, 10, 32) == 0          # below the 11x11 window
    assert lib.vsrb_ssim_sums_det(FAKE, FAKE, 1, 3, 32, 32, 1, FAKE, FAKE, 8, None) == E_ARG


def test_alert_raises_or_warns_once(det):
    from vsrlab_b200 import ops
    with pytest.raises(RuntimeError, match="does not have a deterministic implementation"):
        ops.nondeterministic_alert("some op")
    torch.use_deterministic_algorithms(True, warn_only=True)
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        ops.nondeterministic_alert("another op")
        ops.nondeterministic_alert("another op")
    assert sum("another op" in str(r.message) for r in rec) == 1


# ----------------------------------------------------------------------------------------------------------------------
# the matrix resizes of the torch glue (CPU: the same products run on the GPU)
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", [((16, 24), (64, 96), False), ((180, 180), (192, 192), False), ((192, 192), (180, 180), False),
                                  ((37, 53), (64, 64), False), ((37, 53), (20, 71), True), ((8, 8), (16, 16), True)],
                         ids=["x4", "180to192", "192to180", "37x53up", "37x53_aligned", "x2_aligned"])
def test_matrix_resize_matches_interpolate(case):
    from vsrlab_b200 import autograd as AG
    (h, w), (oh, ow), ac = case
    g = torch.Generator().manual_seed(oh * 1000 + ow)
    x = torch.randn(2, 3, h, w, generator=g, dtype=torch.float64)
    gy = torch.randn(2, 3, oh, ow, generator=g, dtype=torch.float64)
    xr = x.clone().requires_grad_(True)
    F.interpolate(xr, size=(oh, ow), mode="bilinear", align_corners=ac).backward(gy)
    xm = x.float().requires_grad_(True)
    y = AG._resize_bilinear(xm, (oh, ow), ac)
    y.backward(gy.float())
    ref = F.interpolate(x, size=(oh, ow), mode="bilinear", align_corners=ac)
    assert rel(y.detach(), ref) < 1e-6
    assert rel(xm.grad, xr.grad) < 1e-6
    assert rel(AG._resize_bilinear_backward(gy.float(), (h, w), ac), xr.grad) < 1e-6
    if not ac and (oh, ow) == (4 * h, 4 * w):           # SrTailFn's d lq: torch's own backward kernel
        want = torch.ops.aten.upsample_bilinear2d_backward(gy, [oh, ow], [2, 3, h, w], False, None, None)
        assert rel(AG._resize_bilinear_backward(gy.float(), (h, w), False), want) < 1e-6


def test_same_size_resize_is_exact_identity():
    from vsrlab_b200 import autograd as AG
    x = torch.randn(2, 2, 13, 17)
    x[0, 0, 0, 0] = float("inf")                        # no 0 * inf from an identity product
    xr = x.clone().requires_grad_(True)
    y = AG._resize_bilinear(xr, (13, 17), False)
    assert torch.equal(y, x)
    g = torch.randn(2, 2, 13, 17)
    y.backward(g)
    assert torch.equal(xr.grad, g)
    assert torch.equal(AG._resize_bilinear_backward(g, (13, 17), False), g)


# ----------------------------------------------------------------------------------------------------------------------
# weight and bias gradients
# ----------------------------------------------------------------------------------------------------------------------
WGRAD_LAYERS = {
    "rb64": ([(0, 64)], 64),
    "up256": ([(0, 64)], 256),
    "stem67": ([(3, 64), (0, 3)], 64),                  # a tensor-core segment and a tap-stacking segment, bias kernel
}
WGRAD_SHAPES = [(1, 20, 28), (4, 45, 77), (120, 64, 64)]   # one CTA; ragged; the training batch (7 680 tiles)


def _det_twice(fn, *outs):
    """fn(*outs) on zeroed outputs twice: the two results."""
    res = []
    for _ in range(2):
        bufs = [None if o is None else torch.zeros_like(o) for o in outs]
        fn(*bufs)
        torch.cuda.synchronize()
        res.append(bufs)
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("shape", WGRAD_SHAPES, ids=lambda s: "n%d_%dx%d" % s)
@pytest.mark.parametrize("name", list(WGRAD_LAYERS))
def test_wgrad_det(dev, poisoned_ws, name, shape):
    from torch.nn.grad import conv2d_weight
    from vsrlab_b200 import ops
    segs, cout = WGRAD_LAYERS[name]
    B, h, w = shape
    cin = sum(c for _, c in segs)
    gen = torch.Generator(device=dev).manual_seed(zlib.crc32(repr((name, shape)).encode()))
    x = randn((B, cin, h, w), gen, dev)
    dz = randn((B, cout, h, w), gen, dev)
    ins = [nhwc(x[:, off:off + c], (c + 15) // 16 * 16 + 16, float("nan")) for off, c in segs]
    dzt = nhwc(dz, cout + 16, float("nan"))
    ref = conv2d_weight(x.double(), (cout, cin, 3, 3), dz.double(), padding=1)
    ref_b = dz.double().sum((0, 2, 3))
    geom = geom_of(segs, cout)
    (dw1, db1), (dw2, db2) = _det_twice(
        lambda dw, db: ops.conv2d_wgrad_det(geom, ins, [t.shape[1] for t in ins], dzt, dzt.shape[1], B, h, w, cin, dw, db),
        torch.empty(cout, cin, 3, 3, device=dev), torch.empty(cout, device=dev))
    assert maxabs(dw1, ref) <= 1e-3 * ref.abs().max().item()
    assert rel(db1, ref_b) <= 1e-4
    assert torch.equal(dw1, dw2) and torch.equal(db1, db2)


@pytest.mark.gpu
@pytest.mark.parametrize("n_chunks", [1, 2, 16, 17, 33])
def test_wgrad_multi_det(dev, poisoned_ws, n_chunks):
    from torch.nn.grad import conv2d_weight
    from vsrlab_b200 import ops
    n, h, w = 8, 64, 64
    gen = torch.Generator(device=dev).manual_seed(2000 + n_chunks)
    xs = [randn((n, 64, h, w), gen, dev) for _ in range(n_chunks)]
    dzs = [randn((n, 64, h, w), gen, dev) for _ in range(n_chunks)]
    chunks = [([nhwc(x, 64)], nhwc(dz, 64)) for x, dz in zip(xs, dzs)]
    x64, dz64 = torch.cat(xs).double(), torch.cat(dzs).double()
    ref = conv2d_weight(x64, (64, 64, 3, 3), dz64, padding=1)
    geom = geom_of([(0, 64)], 64)
    (dw1, db1), (dw2, db2) = _det_twice(lambda dw, db: ops.conv2d_wgrad_multi_det(geom, chunks, [64], 64, n, h, w, 64, dw, db),
                                        torch.empty(64, 64, 3, 3, device=dev), torch.empty(64, device=dev))
    assert maxabs(dw1, ref) <= 1e-3 * ref.abs().max().item()
    assert rel(db1, dz64.sum((0, 2, 3))) <= 1e-4
    assert torch.equal(dw1, dw2) and torch.equal(db1, db2)


@pytest.mark.gpu
@pytest.mark.parametrize("layer", [(8, 32), (32, 64), (64, 32), (32, 16), (16, 2)], ids=lambda l: "sp%dto%d" % l)
def test_wgrad_taps_det_spynet_7x7(dev, poisoned_ws, layer):
    from torch.nn.grad import conv2d_weight
    from vsrlab_b200 import ops
    cin, cout = layer
    B, h, w = 6, 40, 56
    gen = torch.Generator(device=dev).manual_seed(cin * 100 + cout)
    x = randn((B, cin, h, w), gen, dev)
    dz = randn((B, cout, h, w), gen, dev)
    xin, dzt = nhwc(x, (cin + 15) // 16 * 16, float("nan")), nhwc(dz, (cout + 15) // 16 * 16, float("nan"))
    if cin % 16:
        xin[:, cin:] = 0                                # the SPyNet input's padding channels are zero
    ref = conv2d_weight(x.double(), (cout, cin, 7, 7), dz.double(), padding=3)
    geom = geom_of([(0, cin)], cout, 7)
    (dw1, db1), (dw2, db2) = _det_twice(
        lambda dw, db: ops.conv2d_wgrad_det(geom, [xin], [xin.shape[1]], dzt, dzt.shape[1], B, h, w, cin, dw, db),
        torch.empty(cout, cin, 7, 7, device=dev), torch.empty(cout, device=dev))
    assert maxabs(dw1, ref) <= 1e-3 * ref.abs().max().item()
    assert rel(db1, dz.double().sum((0, 2, 3))) <= 1e-4
    assert torch.equal(dw1, dw2) and torch.equal(db1, db2)


@pytest.mark.gpu
def test_wgrad_multi_det_refuses_before_any_launch(dev):
    """A bad chunk in the second group of 16 is refused by the planning pass: nothing of the first group reaches dw."""
    from vsrlab_b200 import _lib as L, ops
    n, h, w, k = 2, 16, 32, 20
    gen = torch.Generator(device=dev).manual_seed(7)
    chunks = [([nhwc(randn((n, 64, h, w), gen, dev), 64)], nhwc(randn((n, 64, h, w), gen, dev), 64)) for _ in range(k)]
    geom = geom_of([(0, 64)], 64)
    lib = L.load()
    ws = torch.empty(lib.vsrb_conv2d_wgrad_det_workspace_bytes(C.byref(geom), k, n, h, w, 1), dtype=torch.uint8, device=dev)
    dw = torch.full((64, 64, 3, 3), 5.0, device=dev)
    db = torch.full((64,), 5.0, device=dev)
    ptrs = (C.c_void_p * k)(*[c[0][0].data_ptr() for c in chunks])
    dzs = (C.c_void_p * k)(*[c[1].data_ptr() for c in chunks])
    dzs[18] = chunks[18][1].data_ptr() + 2                              # misaligned: never dereferenced, refused
    rc = lib.vsrb_conv2d_wgrad_multi_det(C.byref(geom), k, ptrs, (C.c_int32 * 1)(64), dzs, 64, n, h, w, 64, ops._p(dw), ops._p(db),
                                         ops._p(ws), ws.numel(), ops._stream())
    torch.cuda.synchronize()
    assert rc == E_ARG and b"chunk" in lib.vsrb_last_error()
    assert (dw == 5.0).all() and (db == 5.0).all()


# ----------------------------------------------------------------------------------------------------------------------
# warp backward
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("flows", ["pm20", "collapse"])
@pytest.mark.parametrize("border", [False, True], ids=["zeros", "border"])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16_c64", "fp32_c4"])
def test_warp_bwd_det(dev, poisoned_ws, dtype, border, flows):
    from oracle import vsr_oracle as O
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16, F32, PAD_BORDER, PAD_ZEROS
    g = torch.Generator().manual_seed(21 + border + (flows == "collapse") * 2)
    c = 64 if dtype == torch.bfloat16 else 4
    n, h, w = 2, 29, 37
    x = bf16r(torch.randn(n, c, h, w, generator=g))
    if flows == "pm20":
        fl = (torch.rand(n, h, w, 2, generator=g) - 0.5) * 40
    else:                                               # every pixel lands within ~1.5 px of one of two points: long runs
        yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing="ij")
        tgt = torch.tensor([[5.3, 7.6], [20.2, 11.4]])[torch.randint(0, 2, (n, h, w), generator=g)]
        fl = torch.stack([tgt[..., 0] - xx, tgt[..., 1] - yy], -1) + (torch.rand(n, h, w, 2, generator=g) - 0.5) * 3
    gy = bf16r(torch.randn(n, c, h, w, generator=g))
    xr, fr = x.double().requires_grad_(True), fl.double().requires_grad_(True)
    (O.flow_warp(xr, fr, "border" if border else "zeros") * gy.double()).sum().backward()
    xd = x.to(dev).to(dtype).permute(0, 2, 3, 1).contiguous()
    dout = gy.to(dev).to(dtype).permute(0, 2, 3, 1).contiguous()
    fd = fl.to(dev).contiguous()
    dt, pad = (BF16 if dtype == torch.bfloat16 else F32), (PAD_BORDER if border else PAD_ZEROS)
    outs = []
    for _ in range(2):
        dx = torch.full((n, h, w, c), float("nan"), device=dev)
        dflow = torch.full((n, h, w, 2), float("nan"), device=dev)
        ops.flow_warp_bwd_det(xd, fd, dout, dx, dflow, n, h, w, c, dt, pad)
        torch.cuda.synchronize()
        outs.append((dx, dflow))
    (dx1, df1), (dx2, df2) = outs
    assert torch.equal(dx1, dx2) and torch.equal(df1, df2)
    assert rel(dx1.permute(0, 3, 1, 2).cpu(), xr.grad) < (1e-2 if dtype == torch.bfloat16 else 1e-5)
    assert rel(df1.cpu(), fr.grad) < (2e-2 if dtype == torch.bfloat16 else 1e-4)
    df0 = torch.full_like(df1, float("nan"))            # the default kernel's flow gradient, bit for bit
    ops.flow_warp_bwd(xd, fd, dout, None, df0, n, h, w, c, dt, pad)
    torch.cuda.synchronize()
    assert torch.equal(df0, df1)


@pytest.mark.gpu
def test_warp_bwd_det_nonfinite_dout_gives_nan(dev):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16, PAD_ZEROS
    n, h, w, c = 1, 8, 8, 8
    dout = torch.ones(n, h, w, c, dtype=torch.bfloat16, device=dev)
    dout[0, 3, 3, 0] = float("inf")
    dx = torch.zeros(n, h, w, c, device=dev)
    ops.flow_warp_bwd_det(None, torch.zeros(n, h, w, 2, device=dev), dout, dx, None, n, h, w, c, BF16, PAD_ZEROS)
    torch.cuda.synchronize()
    assert torch.isnan(dx).all()                        # GradScaler sees the overflow and skips the step


# ----------------------------------------------------------------------------------------------------------------------
# loss and metric sums
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_loss_and_metric_sums_det(dev, det, poisoned_ws):
    from vsrlab_b200 import losses
    g = torch.Generator(device=dev).manual_seed(5)
    sr = torch.rand(2, 5, 3, 96, 80, generator=g, device=dev).requires_grad_(True)
    hr = torch.rand(2, 5, 3, 96, 80, generator=g, device=dev)
    lq = torch.rand(2, 5, 3, 24, 20, generator=g, device=dev).requires_grad_(True)
    res = []
    for mode in (True, True, False):
        torch.use_deterministic_algorithms(mode)
        sr.grad = lq.grad = None
        loss = losses.realbasicvsr_loss(sr, hr, lq)
        loss.backward()
        p = losses.PSNR()(sr.detach().flatten(0, 1), hr.flatten(0, 1))
        s = losses.SSIM()(sr.detach().flatten(0, 1), hr.flatten(0, 1))
        res.append([loss.detach(), sr.grad.clone(), lq.grad.clone(), p, s])
    for a, b in zip(res[0], res[1]):
        assert torch.equal(a, b)                        # deterministic twice: bit for bit
    for a, b in zip(res[0], res[2]):
        assert rel(a, b) < 1e-6                         # against the atomics' sums


# ----------------------------------------------------------------------------------------------------------------------
# refusals, and the flag off
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("what", ["bicubic", "reflection", "conv1x3"])
def test_ops_without_deterministic_kernel_raise_or_warn(dev, det, what):
    from vsrlab.core.modules.conv import ConvReLU
    from vsrlab_b200 import functional as VF, ops

    def run():
        g = torch.Generator(device=dev).manual_seed(3)
        x = torch.rand(2, 8, 16, 24, generator=g, device=dev).requires_grad_(True)
        if what == "conv1x3":
            m = ConvReLU(8, 16, (1, 3), 1, (0, 1)).to(dev)
            with torch.autocast("cuda", dtype=torch.bfloat16):
                y = m(x)
        else:
            flow = ((torch.rand(2, 16, 24, 2, generator=g, device=dev) - 0.5) * 4).requires_grad_(True)
            y = VF.flow_warp(x, flow, "reflection" if what == "reflection" else "zeros",
                             "bicubic" if what == "bicubic" else "bilinear", align_corners=what != "reflection")
        y.float().sum().backward()
        torch.cuda.synchronize()
        return x.grad

    with pytest.raises(RuntimeError, match="deterministic"):
        run()
    torch.use_deterministic_algorithms(True, warn_only=True)
    ops._alerted.clear()                                # warned once per op and process
    with warnings.catch_warnings(record=True) as rec:
        warnings.simplefilter("always")
        gx = run()
    assert torch.isfinite(gx).all()
    assert any("does not have a deterministic implementation" in str(r.message) for r in rec)


@pytest.mark.gpu
def test_flag_off_calls_no_det_entry_point(dev, monkeypatch):
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import losses, ops

    def boom(*a, **k):
        raise AssertionError("a deterministic entry point ran with the flag off")
    for name in ("conv2d_wgrad_det", "conv2d_wgrad_multi_det", "flow_warp_bwd_det", "loss_sums_det"):
        monkeypatch.setattr(ops, name, boom)
    torch.manual_seed(0)
    net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=True).to(dev).train()
    g = torch.Generator().manual_seed(1)
    lr, hr = torch.rand(1, 3, 3, 32, 32, generator=g).to(dev), torch.rand(1, 3, 3, 128, 128, generator=g).to(dev)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        sr, lq = net(lr.clone())
    losses.realbasicvsr_loss(sr, hr, lq).backward()
    losses.PSNR()(sr.detach().flatten(0, 1), hr.flatten(0, 1))
    torch.cuda.synchronize()
    assert all(p.grad is not None for p in net.parameters() if p.requires_grad)


@pytest.mark.gpu
def test_graphed_train_step_flag_toggle_steps_once_per_call(dev, monkeypatch):
    """GraphedTrainStep captures a second graph when the deterministic flag changes; that capture's warm-up must not train.
    Each call is exactly one optimizer update: Adam's step count advances by one, and the parameters match one eager step
    (under the same flag) from the state before the call."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200.graphs import GraphedTrainStep
    monkeypatch.setenv("CUBLAS_WORKSPACE_CONFIG", ":4096:8")
    g = torch.Generator().manual_seed(12)
    batches = [(torch.rand(1, 3, 3, 32, 32, generator=g).to(dev), torch.rand(1, 3, 3, 128, 128, generator=g).to(dev))
               for _ in range(3)]

    def loss_fn(out, hr_):
        sr, lq = out
        return torch.sqrt((sr - hr_) ** 2 + 1e-9).mean() + torch.sqrt((lq - hr_[..., ::4, ::4]) ** 2 + 1e-9).mean()

    def make():
        torch.manual_seed(21)
        net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=True)
        net = net.to(dev).train()
        return net, torch.optim.Adam(net.parameters(), lr=2e-4, capturable=True)

    def twin_of(net, opt):
        """a copy of (net, opt) sharing no tensor with them"""
        t_net, t_opt = make()
        t_net.load_state_dict(net.state_dict())
        sd = opt.state_dict()
        sd["state"] = {k: {n: v.clone() if torch.is_tensor(v) else v for n, v in st.items()} for k, st in sd["state"].items()}
        t_opt.load_state_dict(sd)
        return t_net, t_opt

    net, opt = make()
    step = GraphedTrainStep(net, opt, loss_fn, batches[0], clip_grad_norm=1.0, warmup=3)

    def adam_steps():
        return {int(st["step"].item()) for st in opt.state.values()}
    assert adam_steps() == {3}
    try:
        for i, flag in enumerate((False, True, False)):
            torch.use_deterministic_algorithms(flag)
            lr, hr = batches[i]
            t_net, t_opt = twin_of(net, opt)                             # one eager step from the same state
            before = [p.detach().clone() for p in net.parameters()]
            step(lr, hr)
            torch.cuda.synchronize()
            assert adam_steps() == {4 + i}, (flag, adam_steps())
            with torch.autocast("cuda", dtype=torch.bfloat16):
                out = t_net(lr.clone())
            t_opt.zero_grad(set_to_none=True)
            loss_fn(out, hr).backward()
            torch.nn.utils.clip_grad_norm_(t_net.parameters(), 1.0)
            t_opt.step()
            moved = max(maxabs(a, b) for a, b in zip(t_net.parameters(), before))
            off = max(maxabs(a, b) for a, b in zip(net.parameters(), t_net.parameters()))
            assert moved > 0 and off < 0.25 * moved, (flag, off, moved)
    finally:
        torch.use_deterministic_algorithms(False)


# ----------------------------------------------------------------------------------------------------------------------
# the model: the reference AMP recipe, bit for bit
# ----------------------------------------------------------------------------------------------------------------------
RECIPE = textwrap.dedent(r'''
    import hashlib, sys, warnings
    import torch
    sys.path.insert(0, sys.argv[1])
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import graphs, losses
    torch.use_deterministic_algorithms(True)
    dev = torch.device("cuda:0")

    def run(shape):
        n, t, h, w = shape
        torch.manual_seed(0)
        net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=2, pretrained_flow=False, train_flow=True)
        net = net.to(dev).train()
        opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.99))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            scaler = torch.cuda.amp.GradScaler()
        g = torch.Generator().manual_seed(1)
        data = [(torch.rand(n, t, 3, h, w, generator=g).to(dev), torch.rand(n, t, 3, 4 * h, 4 * w, generator=g).to(dev))
                for _ in range(2)]
        out = []
        for i in range(8):
            lr, hr = data[i % 2]
            with torch.autocast("cuda", dtype=torch.bfloat16):
                sr, lq = net(lr.clone())
                loss = losses.realbasicvsr_loss(sr, hr, lq)
            scaler.scale(loss / 2).backward()
            if i % 2 == 1:
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
                scaler.step(opt)
                scaler.update()
                opt.zero_grad()
            out.append(loss.item())
            out.append(losses.PSNR()(sr.detach().flatten(0, 1).clamp(0, 1), hr.flatten(0, 1)).item())
        assert graphs.graphed_patterns(net) > 0, "the training graph was not captured"
        h_ = hashlib.sha256()
        for k, v in net.state_dict().items():
            h_.update(k.encode())
            h_.update(v.detach().cpu().contiguous().view(torch.uint8).numpy().tobytes() if v.numel() else b"")
        return out, h_.hexdigest()

    for shape in ((1, 3, 36, 44), (1, 3, 64, 64)):
        a, b = run(shape), run(shape)
        assert a[0] == b[0], (shape, a[0], b[0])
        assert a[1] == b[1], shape
        print("HASH", shape, a[1], flush=True)
''')


@pytest.mark.gpu
def test_reference_recipe_is_bit_reproducible(dev, tmp_path):
    script = tmp_path / "recipe.py"
    script.write_text(RECIPE)
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8", PYTHONPATH=str(ROOT))
    hashes = []
    for _ in range(2):
        r = subprocess.run([sys.executable, str(script), str(ROOT)], env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-6000:]
        hashes.append([ln for ln in r.stdout.splitlines() if ln.startswith("HASH")])
    assert len(hashes[0]) == 2 and hashes[0] == hashes[1], hashes
