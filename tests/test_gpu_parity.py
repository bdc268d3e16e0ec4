"""Parity of the CUDA path (through the C-ABI) against the CPU oracle and the golden fixtures.

Tolerances (north_star): fp32 mode max-abs <= 1e-4 on sr; flows <= 1e-2 px; bf16 mode PSNR
within 0.05 dB on [0,1] frames.  Kernel-level bf16 checks compare against the oracle run on
bf16-rounded operands: the only differences left are fp32 summation order and the final bf16
rounding of the stored activation (half an ulp: 2^-9 relative)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import build_state_dict
from oracle import vsr_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from vsrlab_b200 import load
    load()
    return torch.device("cuda:0")


def bf16r(x):
    return x.to(torch.bfloat16).to(torch.float32)


def T(a):
    return torch.from_numpy(np.asarray(a))


CONV_CASES = [
    # segs (OIHW offset, channels), cout, k, h, w, n, act, groups, pixshuf, residual
    ([(0, 64)], 64, 3, 16, 16, 1, "none", 1, 0, False),
    ([(0, 64)], 64, 1, 16, 16, 1, "none", 1, 0, False),
    ([(0, 64)], 64, 3, 37, 52, 3, "none", 1, 0, True),
    ([(0, 3)], 64, 3, 24, 33, 2, "lrelu", 1, 0, False),
    ([(3, 64), (0, 3)], 64, 3, 24, 40, 2, "lrelu", 2, 0, False),
    ([(0, 64), (64, 64)], 64, 1, 24, 40, 2, "lrelu", 1, 0, False),
    ([(0, 64)], 256, 3, 24, 40, 1, "none", 1, 2, False),
    ([(0, 64)], 3, 3, 24, 40, 2, "none", 1, 0, False),
    ([(0, 8)], 32, 7, 24, 40, 2, "relu", 1, 0, False),
    ([(0, 32)], 64, 7, 24, 40, 2, "relu", 1, 0, False),
    ([(0, 64)], 32, 7, 12, 20, 2, "relu", 1, 0, False),
    ([(0, 32)], 16, 7, 6, 10, 2, "relu", 1, 0, False),
    ([(0, 16)], 2, 7, 2, 2, 3, "relu", 1, 0, False),
    ([(0, 64)], 64, 3, 180, 320, 2, "relu", 1, 0, True),
]


def to_dev_nhwc(x_nchw, dt, dev):
    """[B,c,h,w] fp32 -> the NHWC device tensor of activation dtype `dt` (bf16 / fp32 / split-bf16 [hi|lo])."""
    from vsrlab_b200 import functional as VF, ops
    from vsrlab_b200._lib import BF16X2
    B, c, h, w = x_nchw.shape
    ca = VF._act_c(c, dt)
    t = torch.zeros(B, h, w, ca, dtype=ops.TORCH_DT[dt], device=dev)
    v = x_nchw.permute(0, 2, 3, 1).to(dev)
    if dt == BF16X2:
        hi = v.to(torch.bfloat16)
        t[..., :c] = hi
        t[..., ca // 2:ca // 2 + c] = (v - hi.float()).to(torch.bfloat16)
    else:
        t[..., :c] = v.to(ops.TORCH_DT[dt])
    return t, ca


def from_dev_nhwc(t, c, dt):
    from vsrlab_b200._lib import BF16X2
    if dt == BF16X2:
        half = t.shape[-1] // 2
        return (t[..., :c].float() + t[..., half:half + c].float()).permute(0, 3, 1, 2).cpu()
    return t[..., :c].float().permute(0, 3, 1, 2).cpu()


@pytest.mark.parametrize("mode", ["fp32", "bf16", "x3"])
@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: f"k{c[2]}_{c[0]}_{c[1]}_{c[3]}x{c[4]}")
def test_conv_kernels(dev, mode, case):
    """fp32 = FFMA kernel, bf16 = tcgen05 kernel, x3 = tcgen05 kernel in the fp32-accurate split-bf16 mode."""
    from vsrlab_b200 import functional as VF, ops
    from vsrlab_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, BF16, BF16X2, F32
    segs, cout, k, h, w, n, act, groups, pixshuf, residual = case
    dt = {"bf16": BF16, "fp32": F32, "x3": BF16X2}[mode]
    g = torch.Generator().manual_seed(hash((k, cout, h, w)) % 1000)
    cin = sum(c for _, c in segs)
    convs = []
    for _ in range(groups):
        cv = torch.nn.Conv2d(cin, cout, k, 1, k // 2)
        with torch.no_grad():
            cv.weight.copy_(torch.randn(cv.weight.shape, generator=g) / (cin * k * k) ** 0.5)
            cv.bias.copy_(torch.randn(cv.bias.shape, generator=g) * 0.1)
        convs.append(cv)
    B = n * groups
    x = torch.randn(B, cin, h, w, generator=g)
    res = torch.randn(B, cout, h, w, generator=g) if residual else None
    ys = []
    for gi in range(groups):
        xs, wg = x[gi * n:(gi + 1) * n], convs[gi].weight.detach()
        if dt == BF16:
            xs, wg = bf16r(xs), bf16r(wg)
        ys.append(F.conv2d(xs, wg, convs[gi].bias.detach(), padding=k // 2))
    y = torch.cat(ys)
    y = {"none": lambda v: v, "relu": O.relu, "lrelu": O.lrelu}[act](y)
    if residual:
        y = y + (bf16r(res) if dt == BF16 else res)
    if pixshuf:
        y = O.pixel_shuffle(y, 2)

    tdt = ops.TORCH_DT[dt]
    pc = ops.PackedConv([c.to(dev) for c in convs], segs, dt, pixshuf)
    ins, in_c = [], []
    for off, c in segs:
        t, ca = to_dev_nhwc(x[:, off:off + c], dt, dev)
        ins.append(t)
        in_c.append(ca)
    r = pixshuf or 1
    co = cout // (r * r)
    oc = VF._act_c(co, dt) if (r > 1 or dt == BF16X2) else pc.cout_pad
    out = torch.full((B, h * r, w * r, oc), 7.0, dtype=tdt, device=dev)
    rt, rc = None, 0
    if residual:
        rt, rc = to_dev_nhwc(res, dt, dev)
    ops.conv2d_fwd(pc, ins, in_c, B, h, w, act={"none": ACT_NONE, "relu": ACT_RELU, "lrelu": ACT_LRELU}[act], slope=0.1,
                   out=out, out_c=oc, residual=rt, res_c=rc)
    torch.cuda.synchronize()
    assert ops.debug_status() == 0
    got = from_dev_nhwc(out, co, dt)
    scale = max(y.abs().max().item(), 1.0)
    tol = (2.0 ** -8 if dt == BF16 else 2e-5) * scale        # bf16: half-ulp of the stored value (2^-9) + slack
    assert (got - y).abs().max().item() <= tol               # split-bf16 must be as good as the fp32 FFMA kernel
    if dt != BF16X2 and oc > co and not pixshuf:             # padded channels must come out as act(0) = 0
        assert out[..., co:].abs().max().item() == 0


PAIR_CASES = [
    # cin, cout, k, n, h, w, residual, pixshuf : shapes that take the CTA-pair (cta_group::2) kernels, with odd tile
    # counts (a dummy tile in the last pair), a single tile, ragged borders, and every kernel variant
    (64, 64, 3, 1, 4, 30, False, 0),        # exactly one tile: the peer CTA only has the dummy
    (64, 64, 3, 1, 12, 31, True, 0),        # 3 x 2 tiles, residual through the identity MMA
    (64, 64, 3, 3, 37, 52, False, 0),       # odd tile count, 3 images
    (32, 32, 3, 2, 20, 33, False, 0),       # 32-wide stacked tile (N = 96, two sub-tiles per stage)
    (64, 256, 3, 1, 17, 23, False, 2),      # classic layout, N = 128, pixel-shuffle store
    (64, 32, 7, 2, 13, 29, False, 0),       # 7x7, 64-byte K rows, half of 200 KB of weights resident per CTA
    (32, 64, 7, 1, 9, 27, False, 0),        # 7x7, two N blocks
    (32, 16, 7, 2, 6, 10, False, 0),
]


@pytest.mark.parametrize("case", PAIR_CASES, ids=lambda c: f"k{c[2]}_{c[0]}to{c[1]}_{c[4]}x{c[5]}")
def test_cta_pair_kernels_match_single_cta(dev, case, monkeypatch):
    """The pair kernels issue the same MMAs in the same order on the same operands as the single-CTA kernels, only as
    M = 256 instructions across two SMs: outputs must be bit-identical (and both must match the oracle conv)."""
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_NONE, ACT_RELU, BF16, VsrbError
    cin, cout, k, n, h, w, residual, pixshuf = case
    g = torch.Generator().manual_seed(cin * 131 + cout + h)
    cv = torch.nn.Conv2d(cin, cout, k, 1, k // 2)
    with torch.no_grad():
        cv.weight.copy_(torch.randn(cv.weight.shape, generator=g) / (cin * k * k) ** 0.5)
        cv.bias.copy_(torch.randn(cv.bias.shape, generator=g) * 0.1)
    x = torch.randn(n, cin, h, w, generator=g)
    res = torch.randn(n, cout, h, w, generator=g) if residual else None
    pc = ops.PackedConv([cv.to(dev)], [(0, cin)], BF16, pixshuf)
    xt, ca = to_dev_nhwc(x, BF16, dev)
    r = pixshuf or 1
    co = cout // (r * r)
    oc = (co + 15) // 16 * 16
    rt, rc = (None, 0) if res is None else to_dev_nhwc(res, BF16, dev)
    outs = []
    for no_pair in ("", "1"):
        if no_pair:
            monkeypatch.setenv("VSRB_TC_NO_PAIR", "1")
        else:
            monkeypatch.delenv("VSRB_TC_NO_PAIR", raising=False)
        out = torch.full((n, h * r, w * r, oc), 7.0, dtype=torch.bfloat16, device=dev)
        try:
            ops.conv2d_fwd(pc, [xt], [ca], n, h, w, act=ACT_NONE if residual else ACT_RELU, out=out, out_c=oc, residual=rt, res_c=rc)
        except VsrbError as e:
            # plans that keep half of a large weight block resident per CTA (7x7 with >= 32-channel K rows) only exist
            # as pairs: without them the library must refuse loudly, not fall back
            assert no_pair and k == 7 and "does not fit" in str(e)
            continue
        torch.cuda.synchronize()
        assert ops.debug_status() == 0
        outs.append(out)
    if len(outs) == 2:
        assert torch.equal(outs[0], outs[1])
    y = F.conv2d(bf16r(x), bf16r(cv.weight.detach().cpu()), cv.bias.detach().cpu(), padding=k // 2)
    y = y + bf16r(res) if residual else O.relu(y)
    if pixshuf:
        y = O.pixel_shuffle(y, 2)
    got = from_dev_nhwc(outs[0], co, BF16)
    assert (got - y).abs().max().item() <= 2.0 ** -8 * max(y.abs().max().item(), 1.0)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
@pytest.mark.parametrize("pad", ["zeros", "border"])
def test_flow_warp_golden_and_adversarial(dev, golden, mode, pad):
    from vsrlab.vsr.models.RealBasicVSR.modules.spynet import flow_warp
    from vsrlab_b200 import functional as VF
    g = golden("ops")
    x, fl = T(g["warp_x"]), T(g["warp_flow"])
    # fp32 mode stores activations as split-bf16 (hi + lo = 16 mantissa bits): 2^-17 relative, i.e. 3e-5 at |x| = 4
    tol = 5e-5 if mode == "fp32" else 2.0 ** -7
    with VF.precision(mode):
        got = flow_warp(x.to(dev), fl.to(dev), padding_mode=pad).cpu()
    assert (got - T(g[f"warp_{pad}"])).abs().max().item() <= tol
    # adversarial: integer, half-pixel, far out-of-bounds flows on a 64-channel map
    gen = torch.Generator().manual_seed(3)
    x = torch.randn(2, 64, 19, 27, generator=gen)
    fl = (torch.rand(2, 19, 27, 2, generator=gen) - 0.5) * 40
    fl[0, 0, :3] = torch.tensor([[0.0, 0.0], [1.0, 1.0], [0.5, 0.5]])
    fl[1, 3, 3] = torch.tensor([500.0, -500.0])
    fl[1, 18, 26] = torch.tensor([1e-4, 1e-4])
    ref = O.flow_warp(bf16r(x) if mode == "bf16" else x, fl, pad)
    with VF.precision(mode):
        got = flow_warp(x.to(dev), fl.to(dev), padding_mode=pad).cpu()
    assert (got - ref).abs().max().item() <= (5e-5 if mode == "fp32" else 2.0 ** -6)


def test_flow_warp_empty_and_bad_args(dev):
    from vsrlab_b200 import VsrbError, ops
    from vsrlab_b200._lib import BF16
    x = torch.zeros(1, 4, 4, 12, dtype=torch.bfloat16, device=dev)
    with pytest.raises(VsrbError):                            # 12 channels is not a multiple of 8
        ops.flow_warp(x, torch.zeros(1, 4, 4, 2, device=dev), torch.empty_like(x), 1, 4, 4, 12, BF16)


@pytest.mark.parametrize("tag,kind", [("a", "spynet"), ("b", "spynet"), ("c", "spynet_amp")])
def test_spynet_flows(dev, golden, tag, kind):
    """Flow fields within 1e-2 px of the reference in fp32 mode (and in bf16 mode at the
    reference's own flow magnitudes; the amplified case is reported, with a relative bound)."""
    from vsrlab_b200 import functional as VF
    g = golden("spynet")
    sp = build_state_dict(kind).to(dev).eval()
    ref, supp, want = T(g[f"{tag}_ref"]).to(dev), T(g[f"{tag}_supp"]).to(dev), T(g[f"{tag}_flow"])
    with torch.no_grad(), VF.precision("fp32"):
        fl = sp(ref, supp).cpu()
    assert fl.shape == want.shape
    assert (fl - want).abs().max().item() <= 1e-3
    with torch.no_grad(), VF.precision("bf16"):
        fl = sp(ref, supp).cpu()
    err = (fl - want).abs().max().item()
    assert err <= (1e-2 if kind == "spynet" else 0.03 * want.abs().max().item())


@pytest.mark.parametrize("name", ["cfg1", "ragged"])
def test_realbasicvsr_end_to_end(dev, golden, name):
    from vsrlab_b200 import functional as VF, ops
    g = golden(name)
    net = build_state_dict(name).to(dev).eval()
    sr_ref, lq_ref = T(g["sr"]), T(g["lq"])
    lr = T(g["lr"]).to(dev)
    with torch.no_grad(), VF.precision("fp32"):
        sr, lq = net(lr)
    torch.cuda.synchronize()
    assert lq.data_ptr() == lr.data_ptr()                     # in-place / aliasing contract (realbasicvsr.py:26-29)
    assert (sr.cpu() - sr_ref).abs().max().item() <= 1e-4     # north_star fp32 gate
    assert (lq.cpu() - lq_ref).abs().max().item() <= 1e-4
    lr = T(g["lr"]).to(dev)
    with torch.no_grad(), VF.precision("bf16"):
        sr16, _ = net(lr)
    hr = torch.rand(sr_ref.shape, generator=torch.Generator().manual_seed(9))
    assert abs(O.psnr(sr16.cpu(), hr) - O.psnr(sr_ref, hr)) <= 0.05    # north_star bf16 gate
    assert O.psnr(sr16.cpu(), sr_ref) > 40.0
    assert ops.debug_status() == 0


def test_flows_and_basicvsr_alone(dev, golden):
    from vsrlab_b200 import functional as VF
    g = golden("ragged")
    net = build_state_dict("ragged").to(dev).eval()
    lr = T(g["lr"]).to(dev)
    with torch.no_grad(), VF.precision("fp32"):
        ff, fb = net.basicvsr.compute_flow(lr)
        sr = net.basicvsr(lr)
    assert (ff.cpu() - T(g["basicvsr_flow_forward"])).abs().max().item() <= 1e-2
    assert (fb.cpu() - T(g["basicvsr_flow_backward"])).abs().max().item() <= 1e-2
    assert (sr.cpu() - T(g["basicvsr_sr"])).abs().max().item() <= 1e-4


def test_small_modules_match_golden(dev, golden):
    from vsrlab.core.modules.conv import ResidualBlock
    from vsrlab.core.modules.upsampling import PixelShufflePack
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import IterativeRefinement
    from vsrlab_b200 import functional as VF
    g = golden("ops")

    def sub(prefix):
        return {k[len(prefix):]: T(g[k]) for k in g.files if k.startswith(prefix)}
    tol = 5e-5      # fp32 mode = split-bf16 activations (16 mantissa bits) on the tensor cores; the gate is 1e-4
    with torch.no_grad(), VF.precision("fp32"):
        rb = ResidualBlock(3, 16, 2)
        rb.load_state_dict(sub("rb_sd."))
        assert (rb.to(dev)(T(g["rb_x"]).to(dev)).cpu() - T(g["rb_y"])).abs().max().item() <= tol
        ps = PixelShufflePack(16, 16, 2)
        ps.load_state_dict(sub("ps_sd."))
        assert (ps.to(dev)(T(g["ps_x"]).to(dev)).cpu() - T(g["ps_y"])).abs().max().item() <= tol
        ir = IterativeRefinement(16, 1)
        ir.load_state_dict(sub("ir_sd."))
        x = T(g["ir_x"]).to(dev)
        y = ir.to(dev)(x)
        assert y.data_ptr() == x.data_ptr()
        assert (y.cpu() - T(g["ir_y"])).abs().max().item() <= tol


def test_full_size_properties(dev):
    """BASELINE cfg3 size (one 180x320 frame pair): size-independent properties instead of an
    oracle run - a zero flow warps to the identity, and the conv is linear in its input."""
    from vsrlab_b200 import functional as VF, ops
    from vsrlab_b200._lib import ACT_NONE, BF16
    gen = torch.Generator().manual_seed(1)
    x = torch.randn(2, 180, 320, 64, generator=gen).to(dev).to(torch.bfloat16)
    out = torch.empty_like(x)
    ops.flow_warp(x, torch.zeros(2, 180, 320, 2, device=dev), out, 2, 180, 320, 64, BF16)
    # zero flow is the identity up to the reference's normalise/de-normalise round trip (spynet.py:101-105),
    # which moves the sample point by ~1e-6 * w pixels
    assert (out.float() - x.float()).abs().max().item() <= 2e-3
    from vsrlab_b200._lib import PAD_BORDER
    const = torch.arange(64, device=dev).to(torch.bfloat16).expand(2, 180, 320, 64).contiguous()
    fl = (torch.rand(2, 180, 320, 2, generator=gen).to(dev) - 0.5) * 100
    ops.flow_warp(const, fl, out, 2, 180, 320, 64, BF16, PAD_BORDER)
    assert (out.float() - const.float()).abs().max().item() <= 0.5       # bilinear weights sum to one (1 bf16 ulp at 63)
    cv = torch.nn.Conv2d(64, 64, 3, 1, 1, bias=False).to(dev)
    pc = ops.PackedConv([cv], [(0, 64)], BF16)
    ya, yb = torch.empty_like(x), torch.empty_like(x)
    ops.conv2d_fwd(pc, [x], [64], 2, 180, 320, act=ACT_NONE, out=ya, out_c=64)
    ops.conv2d_fwd(pc, [x * 2], [64], 2, 180, 320, act=ACT_NONE, out=yb, out_c=64)
    torch.cuda.synchronize()
    assert torch.equal(ya.float() * 2, yb.float())            # exact: scaling by 2 commutes with every rounding
    assert ops.debug_status() == 0


@pytest.mark.parametrize("mid,upscale,blocks", [(32, 4, 1), (64, 2, 1), (48, 4, 2)])
def test_other_widths_and_scales(dev, mid, upscale, blocks):
    """Constructor arguments other than the benchmarked ones (mid_channels, upscale) go through the generic
    kernel paths; checked against the CPU oracle on the module's own random-init weights."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import functional as VF, ops
    torch.manual_seed(mid + upscale)
    net = RealBasicVSR(cleaning_blocks=blocks, mid_channels=mid, upscale=upscale, res_blocks=blocks, pretrained_flow=False,
                       train_flow=False).eval()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    x = torch.rand(2, 3, 3, 24, 40, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        sr_ref, lq_ref = O.realbasicvsr(x.clone(), sd)
    net = net.to(dev)
    with torch.no_grad(), VF.precision("fp32"):
        sr, lq = net(x.clone().to(dev))
    assert sr.shape == sr_ref.shape
    assert (sr.cpu() - sr_ref).abs().max().item() <= 1e-4 and (lq.cpu() - lq_ref).abs().max().item() <= 1e-4
    with torch.no_grad(), VF.precision("bf16"):
        sr16, _ = net(x.clone().to(dev))
    assert O.psnr(sr16.cpu(), sr_ref) > 40.0
    assert ops.debug_status() == 0


@pytest.mark.parametrize("shape", [(1, 1, 3, 16, 16), (1, 2, 3, 8, 8), (3, 2, 3, 33, 17), (1, 4, 3, 70, 100)],
                         ids=lambda s: "x".join(map(str, s)))
def test_edge_shapes(dev, shape):
    """Degenerate clips: a single frame (no flow, no warp at all), two frames, images smaller than one tile,
    odd sizes that need the /32 resize inside SPyNet, several clips.  Checked against the CPU oracle."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import functional as VF, ops
    torch.manual_seed(17)
    net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=False).eval()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    x = torch.rand(*shape, generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        sr_ref, lq_ref = O.realbasicvsr(x.clone(), sd)
    net = net.to(dev)
    with torch.no_grad(), VF.precision("fp32"):
        sr, lq = net(x.clone().to(dev))
    assert (sr.cpu() - sr_ref).abs().max().item() <= 1e-4 and (lq.cpu() - lq_ref).abs().max().item() <= 1e-4
    with torch.no_grad(), VF.precision("bf16"):
        sr16, _ = net(x.clone().to(dev))
    assert O.psnr(sr16.cpu(), sr_ref) > 40.0
    assert ops.debug_status() == 0


def test_graph_replay_and_pdl_do_not_change_results(dev):
    """Scheduling features must be invisible in the numbers: eager launches, programmatic dependent launch between convs
    and CUDA-graph replay of the whole forward give bit-identical sr / lq (bf16 mode)."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import functional as VF, ops
    torch.manual_seed(5)
    model = RealBasicVSR(cleaning_blocks=2, mid_channels=64, upscale=4, res_blocks=2, pretrained_flow=False, train_flow=False)
    model = model.to(dev).eval()
    x = torch.rand(2, 4, 3, 40, 72, device=dev)
    keep = (VF.GRAPHS, ops.PDL)
    outs = []
    try:
        with VF.precision("bf16"), torch.no_grad():
            for graphs, pdl in ((False, False), (False, True), (True, True), (True, True)):
                VF.GRAPHS, ops.PDL = graphs, pdl
                VF.clear_caches()
                xi = x.clone()
                sr, lq = model(xi)
                torch.cuda.synchronize()
                assert ops.debug_status() == 0
                outs.append((sr.clone(), lq.clone()))
    finally:
        VF.GRAPHS, ops.PDL = keep
        VF.clear_caches()
    for sr, lq in outs[1:]:
        assert torch.equal(sr, outs[0][0]) and torch.equal(lq, outs[0][1])


def test_cfg2_spynet_256(dev, golden):
    """BASELINE.json configs[1]: SPyNet on a 7-frame 256x256 clip, both pair directions, against flows computed by
    the reference itself (tests/golden/cfg2.npz): <= 1e-2 px (north_star), in both precision modes."""
    from vsrlab_b200 import functional as VF, ops
    g = golden("cfg2")
    clip = torch.rand(7, 3, 256, 256, generator=torch.Generator().manual_seed(2024))
    assert abs(clip.double().sum().item() - float(g["clip_checksum"][0])) < 1e-6
    sp = build_state_dict("spynet").to(dev).eval()
    clip = clip.to(dev)
    for mode, tol in (("fp32", 1e-3), ("bf16", 1e-2)):
        with torch.no_grad(), VF.precision(mode):
            fb = sp(clip[:-1], clip[1:]).cpu()
            ff = sp(clip[1:], clip[:-1]).cpu()
        for nm, f in (("backward", fb), ("forward", ff)):
            assert f.shape == (6, 2, 256, 256)
            assert (f[:, :, 0::2, 1::2] - T(g[f"flow_{nm}_s2"])).abs().max().item() <= tol, (mode, nm)
    assert ops.debug_status() == 0


def _oracle_case(blocks, shape, seed):
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    torch.manual_seed(seed)
    net = RealBasicVSR(cleaning_blocks=blocks, mid_channels=64, upscale=4, res_blocks=blocks, pretrained_flow=False,
                       train_flow=False).eval()
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    x = torch.rand(*shape, generator=torch.Generator().manual_seed(seed + 1))
    with torch.no_grad():
        sr_ref, lq_ref = O.realbasicvsr(x.clone(), sd)
    return net, x, sr_ref, lq_ref


def _check_modes(net, x, sr_ref, lq_ref, dev):
    from vsrlab_b200 import functional as VF, ops
    with torch.no_grad(), VF.precision("fp32"):
        xin = x.clone().to(dev)
        sr, lq = net(xin)
    assert lq.data_ptr() == xin.data_ptr()
    e_sr, e_lq = (sr.cpu() - sr_ref).abs().max().item(), (lq.cpu() - lq_ref).abs().max().item()
    assert e_sr <= 1e-4 and e_lq <= 1e-4, (e_sr, e_lq)                     # north_star fp32 gate
    with torch.no_grad(), VF.precision("bf16"):
        sr16, lq16 = net(x.clone().to(dev))
    hr = torch.rand(sr_ref.shape, generator=torch.Generator().manual_seed(9))
    d = abs(O.psnr(sr16.cpu().clamp(0, 1), hr) - O.psnr(sr_ref.clamp(0, 1), hr))
    assert d <= 0.05, d                                                     # north_star bf16 gate
    assert O.psnr(sr16.cpu(), sr_ref) > 40.0 and O.psnr(lq16.cpu(), lq_ref) > 40.0
    assert ops.debug_status() == 0


@pytest.mark.parametrize("graphs", [False, True], ids=["eager", "graph"])
def test_multi_chunk_schedule_matches_oracle(dev, graphs):
    """The benchmark's schedule: several clips, more frames than one cleaner / tail chunk, chunk loops that iterate with
    a remainder (functional.py CLEAN_CHUNK / TAIL_CHUNK offset slicing), eager and as a replayed CUDA graph."""
    from vsrlab_b200 import functional as VF
    net, x, sr_ref, lq_ref = _oracle_case(2, (2, 9, 3, 36, 52), 31)
    net = net.to(dev)
    keep = (VF.CLEAN_CHUNK, VF.TAIL_CHUNK, VF.GRAPHS)
    try:
        VF.CLEAN_CHUNK, VF.TAIL_CHUNK, VF.GRAPHS = 4, 5, graphs            # 18 frames: 4+4+4+4+2 and 5+5+5+3
        VF.clear_caches()
        _check_modes(net, x, sr_ref, lq_ref, dev)
    finally:
        VF.CLEAN_CHUNK, VF.TAIL_CHUNK, VF.GRAPHS = keep
        VF.clear_caches()


def test_default_chunks_more_frames_than_a_chunk(dev):
    """Default chunk sizes (60 / 15) with 2 clips x 17 frames: B = 34 frames -> one cleaner chunk, tail chunks 15 + 15 + 4."""
    net, x, sr_ref, lq_ref = _oracle_case(1, (2, 17, 3, 24, 40), 41)
    _check_modes(net.to(dev), x, sr_ref, lq_ref, dev)


def test_headline_shape_180x320_matches_oracle(dev):
    """BASELINE cfg3 geometry (180x320 -> 720x1280, 5/5 blocks, experiment=basic) on 3 frames against the CPU oracle:
    the exact tile plans, the 180 -> 192 SPyNet resize and the CTA-pair kernels of the headline benchmark."""
    net, x, sr_ref, lq_ref = _oracle_case(5, (1, 3, 3, 180, 320), 51)
    assert sr_ref.shape == (1, 3, 3, 720, 1280)
    _check_modes(net.to(dev), x, sr_ref, lq_ref, dev)


def test_two_streams_same_shape_do_not_share_graph_buffers(dev):
    """Two CUDA streams running same-shaped clips through the same model (bench.py --streams 2, or two threads): each
    stream gets its own captured graph, static buffers and scratch set, so the results equal the sequential ones."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import functional as VF, ops
    torch.manual_seed(6)
    model = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=False)
    model = model.to(dev).eval()
    xs = [torch.rand(1, 4, 3, 40, 56, device=dev) for _ in range(2)]
    keep = VF.GRAPHS
    try:
        VF.GRAPHS = True
        VF.clear_caches()
        with VF.precision("bf16"), torch.no_grad():
            want = [tuple(t.clone() for t in model(x.clone())) for x in xs]          # sequential, default stream
            torch.cuda.synchronize()
            streams = [torch.cuda.Stream(device=dev) for _ in range(2)]
            for rep in range(3):                                                     # capture, then replays that overlap
                got = []
                for st, x in zip(streams, xs):
                    st.wait_stream(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(st):
                        got.append(model(x.clone()))
                for st in streams:
                    torch.cuda.current_stream(dev).wait_stream(st)
                torch.cuda.synchronize()
                for (sr, lq), (sr0, lq0) in zip(got, want):
                    assert torch.equal(sr, sr0) and torch.equal(lq, lq0), rep
        assert len({k[-1] for k in VF._graphs}) >= 2                                 # one capture per calling stream
        assert ops.debug_status() == 0
    finally:
        VF.GRAPHS = keep
        VF.clear_caches()


def test_graph_entries_own_their_workspaces(dev):
    """A re-capture (weights changed) must release the previous capture's buffers instead of piling up scratch sets."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import functional as VF
    torch.manual_seed(6)
    model = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=False)
    model = model.to(dev).eval()
    x = torch.rand(1, 3, 3, 64, 96, device=dev)
    keep = VF.GRAPHS
    try:
        VF.GRAPHS = True
        VF.clear_caches()
        mem = []
        with VF.precision("bf16"), torch.no_grad():
            for i in range(6):
                model(x.clone())
                torch.cuda.synchronize()
                mem.append(torch.cuda.memory_allocated(dev))
                with torch.no_grad():
                    for p in model.parameters():
                        p.add_(1e-6)                                                 # bumps _version: next call re-captures
        assert len(VF._graphs) == 1
        assert not VF._ws                                                            # nothing leaked into the shared scratch table
        assert max(mem[2:]) <= mem[1] * 1.10 + (8 << 20), mem                        # steady state, no growth per re-capture
    finally:
        VF.GRAPHS = keep
        VF.clear_caches()


def test_narrow_sr_output_matches_fp32(dev):
    """Opt-in `sr` dtypes: uint8 must be exactly what torchvision's save_image stores from the fp32 result
    (test.py:138-141: mul(255).add(0.5).clamp(0,255).to(uint8)); fp16 is the rounded fp32 value."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import functional as VF, ops
    torch.manual_seed(6)
    model = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=False)
    model = model.to(dev).eval()
    x = torch.rand(2, 3, 3, 36, 52, device=dev) * 1.2 - 0.1          # some values leave [0,1]: the clamp matters
    with VF.precision("bf16"), torch.no_grad():
        sr32, _ = model(x.clone())
        with VF.output_dtype("uint8"):
            sr8, lq8 = model(x.clone())
        with VF.output_dtype("fp16"):
            sr16, _ = model(x.clone())
    assert sr8.dtype == torch.uint8 and sr16.dtype == torch.float16 and lq8.dtype == torch.float32
    assert torch.equal(sr8, sr32.mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8))
    assert torch.equal(sr16, sr32.to(torch.float16))
    assert ops.debug_status() == 0


RING_CASES = [
    # n (images per group), h, w, groups, act, residual : the ring-walk kernel (conv_ring.cu) for 3x3 64->64
    (1, 4, 30, 1, "relu", False),          # fewer rows than lane quarters: empty walks
    (1, 1, 7, 1, "none", False),           # a single row, one partial strip
    (3, 37, 52, 1, "none", True),          # ragged strips, ranges that cross strip and image borders, residual
    (2, 180, 320, 1, "relu", False),       # headline geometry
    (2, 45, 64, 2, "lrelu", False),        # two weight groups
    (30, 64, 64, 1, "none", True),         # training patch geometry, many images
    (5, 23, 61, 1, "relu", False),         # strips = 3 with a 1-pixel last strip
]


@pytest.mark.parametrize("case", RING_CASES, ids=lambda c: f"n{c[0]}_{c[1]}x{c[2]}_g{c[3]}_{c[4]}{'_res' if c[5] else ''}")
def test_ring_walk_conv_matches_classic_and_oracle(dev, case, monkeypatch):
    """conv_ring_kernel against the stacked-layout kernel (same bf16 operands, fp32 accumulation in another order) and
    against the fp32 conv on bf16-rounded operands; padded output strides as the propagation loop uses them."""
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_LRELU, ACT_NONE, ACT_RELU, BF16
    n, h, w, groups, act, residual = case
    g = torch.Generator().manual_seed(n * 1000 + h * 10 + w)
    convs = []
    for _ in range(groups):
        cv = torch.nn.Conv2d(64, 64, 3, 1, 1)
        with torch.no_grad():
            cv.weight.copy_(torch.randn(cv.weight.shape, generator=g) / 24.0)
            cv.bias.copy_(torch.randn(cv.bias.shape, generator=g) * 0.1)
        convs.append(cv)
    B = n * groups
    x = torch.randn(B, 64, h, w, generator=g)
    res = torch.randn(B, 64, h, w, generator=g) if residual else None
    y = torch.cat([F.conv2d(bf16r(x[i * n:(i + 1) * n]), bf16r(convs[i].weight.detach()), convs[i].bias.detach(), padding=1)
                   for i in range(groups)])
    y = {"none": lambda v: v, "relu": O.relu, "lrelu": O.lrelu}[act](y)
    if residual:
        y = y + bf16r(res)
    pc = ops.PackedConv([c.to(dev) for c in convs], [(0, 64)], BF16)
    xt, _ = to_dev_nhwc(x, BF16, dev)
    rt = to_dev_nhwc(res, BF16, dev)[0] if residual else None
    # images of a group sit 2 frames apart and the groups far apart, like frame t of the [2, N, T, h, w, C] feature bank
    frame = h * w * 64
    outs = []
    for ring in (True, False):
        if ring:
            monkeypatch.setenv("VSRB_RING_MIN_ROWS", "0")
            monkeypatch.delenv("VSRB_TC_NO_RING", raising=False)
        else:
            monkeypatch.setenv("VSRB_TC_NO_RING", "1")
        bank = torch.full((groups, n, 2, h, w, 64), 7.0, dtype=torch.bfloat16, device=dev)
        k0 = ops.launch_count()
        ops.conv2d_fwd(pc, [xt], [64], B, h, w, act={"none": ACT_NONE, "relu": ACT_RELU, "lrelu": ACT_LRELU}[act], slope=0.1,
                       out=bank.data_ptr() + frame * 2, out_c=64, out_img_stride=2 * frame, out_group_stride=n * 2 * frame,
                       residual=rt, res_c=64 if residual else 0)
        torch.cuda.synchronize()
        assert ops.debug_status() == 0 and ops.launch_count() > k0
        assert (bank[:, :, 0].float() == 7.0).all()                  # the other frame of the bank is untouched
        outs.append(bank[:, :, 1].reshape(B, h, w, 64).float().permute(0, 3, 1, 2).cpu())
    scale = max(y.abs().max().item(), 1.0)
    assert (outs[0] - y).abs().max().item() <= 2.0 ** -8 * scale
    assert (outs[1] - y).abs().max().item() <= 2.0 ** -8 * scale
    assert (outs[0] - outs[1]).abs().max().item() <= 2.0 ** -7 * scale


def test_ring_walk_is_the_default_for_large_launches(dev, monkeypatch):
    """Without any override a cleaner-sized launch takes conv_ring_kernel."""
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_RELU, BF16
    monkeypatch.delenv("VSRB_TC_NO_RING", raising=False)
    monkeypatch.delenv("VSRB_RING_MIN_ROWS", raising=False)
    cv = torch.nn.Conv2d(64, 64, 3, 1, 1).to(dev)
    pc = ops.PackedConv([cv], [(0, 64)], BF16)
    x = torch.randn(8, 180, 320, 64, device=dev).to(torch.bfloat16)
    out = torch.empty_like(x)
    ops.conv2d_fwd(pc, [x], [64], 8, 180, 320, act=ACT_RELU, out=out, out_c=64)
    torch.cuda.synchronize()
    ref = F.relu(F.conv2d(x.float().permute(0, 3, 1, 2), cv.weight.to(torch.bfloat16).float(), cv.bias, padding=1))
    assert (out.float().permute(0, 3, 1, 2) - ref).abs().max().item() <= 2.0 ** -8 * max(ref.abs().max().item(), 1.0)
    assert ops.debug_status() == 0


STEM_CASES = [
    # n per group, h, w, groups, with 64-channel segment : image stems through the ring-walk kernel's K = 32 im2col operand
    (2, 37, 52, 1, False),       # cleaner stem 3 -> 64 (conv.py:97-98 behind realbasicvsr.py:21), ragged
    (30, 45, 80, 1, False),
    (2, 180, 320, 2, True),      # propagation stem cat([lr_i, feat]) -> 64 (basicvsr.py:56-58,71-73), both directions
    (3, 23, 61, 2, True),
    (1, 16, 16, 2, True),
]


@pytest.mark.parametrize("case", STEM_CASES, ids=lambda c: f"n{c[0]}_{c[1]}x{c[2]}_g{c[3]}_{'64+3' if c[4] else '3'}")
def test_ring_walk_stems_with_im2col_patches(dev, case, monkeypatch):
    """3 -> 64 and 64+3 -> 64 stems: the 3-channel segment as one K = 32 chunk of 3x3 patches (vsrb_im2col3x3_c3) on the
    ring-walk kernel, against the classic kernel and the fp32 conv on bf16-rounded operands; frames addressed through
    image / group strides like the two propagation directions do (group 1 walks the clip backwards)."""
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_LRELU, BF16
    n, h, w, groups, with_feat = case
    g = torch.Generator().manual_seed(n * 77 + h + w)
    cin = 67 if with_feat else 3
    convs = []
    for _ in range(groups):
        cv = torch.nn.Conv2d(cin, 64, 3, 1, 1)
        with torch.no_grad():
            cv.weight.copy_(torch.randn(cv.weight.shape, generator=g) / (cin * 9) ** 0.5)
            cv.bias.copy_(torch.randn(cv.bias.shape, generator=g) * 0.1)
        convs.append(cv)
    B = n * groups
    T = 3                                                     # frames per clip in the patch bank
    frames = torch.rand(n, T, 3, h, w, generator=g)           # the clip bank the patches are built from
    sel = [1, 2][:groups] if groups == 2 else [1]             # group 0 reads frame 1, group 1 frame 2 of every clip
    lr = torch.cat([frames[:, f] for f in sel])               # [B,3,h,w] in launch order
    feat = torch.randn(B, 64, h, w, generator=g) if with_feat else None
    x_full = torch.cat([lr, feat], 1) if with_feat else lr    # reference channel order: cat([lr_i, feat])
    y = torch.cat([F.conv2d(bf16r(x_full[i * n:(i + 1) * n]), bf16r(convs[i].weight.detach()), convs[i].bias.detach(), padding=1)
                   for i in range(groups)])
    y = O.lrelu(y)
    segs = [(3, 64), (0, 3)] if with_feat else [(0, 3)]
    pc = ops.PackedConv([c.to(dev) for c in convs], segs, BF16)
    lr_t, _ = to_dev_nhwc(lr, BF16, dev)
    ins, in_c = ([to_dev_nhwc(feat, BF16, dev)[0], lr_t], [64, 16]) if with_feat else ([lr_t], [16])
    patches = torch.empty(n * T, h, w, 32, dtype=torch.bfloat16, device=dev)
    ops.im2col3x3(frames.reshape(n * T, 3, h, w).to(dev).contiguous(), patches, n * T, h, w)
    pf = h * w * 32
    outs = []
    for ring in (True, False):
        if ring:
            monkeypatch.setenv("VSRB_RING_MIN_ROWS", "0")
            monkeypatch.delenv("VSRB_TC_NO_RING", raising=False)
        else:
            monkeypatch.setenv("VSRB_TC_NO_RING", "1")
        out = torch.full((B, h, w, 64), 7.0, dtype=torch.bfloat16, device=dev)
        ops.conv2d_fwd(pc, ins, in_c, B, h, w, act=ACT_LRELU, slope=0.1, out=out, out_c=64,
                       patch=patches.data_ptr() + sel[0] * pf * 2, patch_img_stride=T * pf, patch_group_stride=pf)
        torch.cuda.synchronize()
        assert ops.debug_status() == 0
        outs.append(out.float().permute(0, 3, 1, 2).cpu())
    scale = max(y.abs().max().item(), 1.0)
    assert (outs[0] - y).abs().max().item() <= 2.0 ** -8 * scale
    assert (outs[1] - y).abs().max().item() <= 2.0 ** -8 * scale


@pytest.mark.parametrize("shape", [(3, 37, 53), (2, 180, 320), (1, 5, 1500), (2, 1, 1), (1, 3, 2)], ids=str)
def test_im2col3x3_patches(dev, shape):
    """vsrb_im2col3x3_c3 (the K = 32 operand of the image stems): bit-exact bf16 of the 3x3 neighbourhoods, zero padded, in
    (ky, kx, c) order with five zero columns; rows wider than 1 363 pixels take the kernel without shared-memory staging."""
    from vsrlab_b200 import ops
    n, h, w = shape
    x = torch.rand(n, 3, h, w, generator=torch.Generator().manual_seed(n * h + w)).to(dev)
    p = torch.full((n, h, w, 32), float("nan"), dtype=torch.bfloat16, device=dev)
    ops.im2col3x3(x, p, n, h, w)
    want = F.unfold(x, 3, padding=1).view(n, 3, 9, h, w).permute(0, 3, 4, 2, 1).reshape(n, h, w, 27).to(torch.bfloat16)
    assert torch.equal(p[..., :27], want) and (p[..., 27:] == 0).all()
