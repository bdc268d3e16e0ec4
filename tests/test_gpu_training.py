"""Backward of the hot path (SURVEY §8 row a13): gradients from the CUDA kernels (input-gradient conv = forward
kernel with transposed packing, weight-gradient kernel, warp backward) against torch autograd through the CPU
oracle.  bf16 activations: gradients agree to bf16 noise, asserted as cosine similarity and relative L2 error."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

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


def rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def cos(a, b):
    return F.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0).item()


@pytest.mark.parametrize("case", [
    # (segs, cout, k, act, pixshuf, residual)
    ([(0, 64)], 64, 3, "relu", 0, False),
    ([(0, 64)], 64, 3, "none", 0, True),
    ([(3, 64), (0, 3)], 64, 3, "lrelu", 0, False),
    ([(0, 64), (64, 64)], 64, 1, "lrelu", 0, False),
    ([(0, 64)], 256, 3, "none", 2, False),
    ([(0, 64)], 3, 3, "none", 0, False),
    ([(0, 8)], 32, 7, "relu", 0, False),
    ([(0, 32)], 16, 7, "relu", 0, False),
], ids=lambda c: f"k{c[2]}_{c[0]}_{c[1]}_{c[3]}")
def test_conv_gradients(dev, case):
    from vsrlab_b200 import autograd as AG
    segs, cout, k, act, pixshuf, residual = case
    g = torch.Generator().manual_seed(7)
    cin = sum(c for _, c in segs)
    cv = torch.nn.Conv2d(cin, cout, k, 1, k // 2)
    with torch.no_grad():
        cv.weight.copy_(bf16r(torch.randn(cv.weight.shape, generator=g) / (cin * k * k) ** 0.5))
        cv.bias.copy_(torch.randn(cv.bias.shape, generator=g) * 0.1)
    B, h, w = 2, 20, 28
    x = bf16r(torch.randn(B, cin, h, w, generator=g))
    res = bf16r(torch.randn(B, cout, h, w, generator=g)) if residual else None
    r = pixshuf or 1
    gy = bf16r(torch.randn(B, cout // (r * r), h * r, w * r, generator=g))
    # oracle: fp32 autograd on the same bf16-representable operands
    xr = x.clone().requires_grad_(True)
    wr, br = cv.weight.detach().clone().requires_grad_(True), cv.bias.detach().clone().requires_grad_(True)
    rr = res.clone().requires_grad_(True) if residual else None
    y = F.conv2d(xr, wr, br, padding=k // 2)
    y = {"none": lambda v: v, "relu": O.relu, "lrelu": O.lrelu}[act](y)
    if residual:
        y = y + rr
    if pixshuf:
        y = O.pixel_shuffle(y, 2)
    (y * gy).sum().backward()
    # device
    cvd = torch.nn.Conv2d(cin, cout, k, 1, k // 2).to(dev)
    cvd.load_state_dict(cv.state_dict())
    ins = []
    for off, c in segs:
        ins.append(AG.to_cl16(x[:, off:off + c].to(dev)).requires_grad_(True))
    rd = AG.to_cl16(res.to(dev)).requires_grad_(True) if residual else None
    yd = AG.conv(cvd, ins, segs, act, 0.1, pixshuf, rd)
    co = cout // (r * r)
    (yd[:, :co].float() * gy.to(dev)).sum().backward()
    assert rel(yd[:, :co].float().cpu(), y.detach()) < 1e-2
    assert cos(cvd.weight.grad.cpu(), wr.grad) > 0.9995 and rel(cvd.weight.grad.cpu(), wr.grad) < 2e-2
    assert rel(cvd.bias.grad.cpu(), br.grad) < 2e-2
    for (off, c), t in zip(segs, ins):
        gx = t.grad[:, :c].float().cpu()
        assert cos(gx, xr.grad[:, off:off + c]) > 0.999 and rel(gx, xr.grad[:, off:off + c]) < 2e-2
        if t.shape[1] > c:
            assert t.grad[:, c:].abs().max().item() == 0          # padded channels get no gradient
    if residual:
        assert rel(rd.grad[:, :cout].float().cpu(), rr.grad) < 1e-2



TAPS_CASES = [
    # (K, cin, cin tensor channels, cout, B, h, w): SPyNet's five 7x7 layers at several pyramid sizes, image / 1x1 / odd widths
    (7, 8, 16, 32, 3, 32, 48), (7, 32, 32, 64, 2, 64, 64), (7, 64, 64, 32, 2, 32, 32), (7, 32, 32, 16, 3, 16, 16), (7, 16, 16, 2, 4, 20, 28),
    (7, 32, 32, 64, 5, 2, 2), (7, 64, 64, 32, 3, 4, 4), (7, 8, 16, 32, 2, 8, 8),
    (3, 3, 16, 64, 2, 20, 36), (1, 128, 128, 64, 2, 12, 20), (5, 24, 32, 40, 2, 18, 22), (3, 80, 80, 72, 1, 9, 17),
]


@pytest.mark.parametrize("case", TAPS_CASES, ids=lambda c: "k%d_%d(%d)->%d_b%d_%dx%d" % c)
def test_wgrad_taps_kernel(dev, case):
    """csrc/wgrad_taps.cu (tap-stacking tcgen05 weight gradient) against fp64 torch on the same bf16 operands, and against the
    mma.sync kernel it replaces (VSRB_WGRAD_MMA=1).  Padding channels of the activation tensors hold NaN: they must not leak."""
    import os
    from vsrlab_b200 import _lib as L
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import BF16
    K, cin, xc, cout, B, h, w = case
    g = torch.Generator().manual_seed(K * 1000 + cin + cout)
    x = bf16r(torch.randn(B, cin, h, w, generator=g))
    dz = bf16r(torch.randn(B, cout, h, w, generator=g))
    zc = (cout + 15) // 16 * 16
    CL = torch.channels_last
    xp = torch.full((B, xc, h, w), float("nan"), dtype=torch.bfloat16, device=dev).contiguous(memory_format=CL)
    zp = torch.full((B, zc, h, w), float("nan"), dtype=torch.bfloat16, device=dev).contiguous(memory_format=CL)
    xp[:, :cin] = x.to(dev)
    zp[:, :cout] = dz.to(dev)
    wr = torch.zeros(cout, cin, K, K, dtype=torch.float64, requires_grad=True)
    (F.conv2d(x.double(), wr, None, 1, K // 2) * dz.double()).sum().backward()
    geom = L.ConvGeom()
    geom.kh = geom.kw = K
    geom.n_seg, geom.cout, geom.pixshuf, geom.groups, geom.dtype, geom.transpose = 1, cout, 0, 1, BF16, 0
    geom.seg_off[0], geom.seg_c[0] = 0, cin
    outs = {}
    for mode in ("taps", "mma") if K != 5 else ("taps",):       # (the mma.sync kernel has no 5x5 instance)
        if mode == "mma":
            os.environ["VSRB_WGRAD_MMA"] = "1"
        try:
            dw = torch.zeros(cout, cin, K, K, dtype=torch.float32, device=dev)
            db = torch.zeros(cout, dtype=torch.float32, device=dev)
            ops.conv2d_wgrad(geom, [xp], [xc], zp, zc, B, h, w, cin, dw, db)
            ops.conv2d_wgrad(geom, [xp], [xc], zp, zc, B, h, w, cin, dw, None)          # accumulates
            torch.cuda.synchronize()
        finally:
            os.environ.pop("VSRB_WGRAD_MMA", None)
        outs[mode] = dw.cpu() / 2
        assert torch.isfinite(dw).all()
        assert rel(db.cpu(), dz.sum((0, 2, 3))) < 1e-3
    scale = wr.grad.abs().max().item()
    assert (outs["taps"].double() - wr.grad).abs().max().item() < 2e-3 * scale + 1e-4, (outs["taps"].double() - wr.grad).abs().max().item()
    assert rel(outs["taps"], wr.grad.float()) < 1e-3
    if "mma" in outs:
        assert rel(outs["taps"], outs["mma"]) < 1e-3


@pytest.mark.parametrize("border,dtype", [(False, torch.bfloat16), (True, torch.float32)])
def test_warp_gradients(dev, border, dtype):
    from vsrlab_b200 import autograd as AG
    g = torch.Generator().manual_seed(11)
    c = 64 if dtype == torch.bfloat16 else 4
    x = bf16r(torch.randn(2, c, 17, 23, generator=g))
    fl = (torch.rand(2, 17, 23, 2, generator=g) - 0.5) * 12
    gy = bf16r(torch.randn(2, c, 17, 23, generator=g))
    xr, fr = x.clone().requires_grad_(True), fl.clone().requires_grad_(True)
    (O.flow_warp(xr, fr, "border" if border else "zeros") * gy).sum().backward()
    xd = x.to(dev).to(dtype).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    fd = fl.to(dev).requires_grad_(True)
    (AG.WarpFn.apply(xd, fd, border).float() * gy.to(dev)).sum().backward()
    assert rel(xd.grad.float().cpu(), xr.grad) < (1e-2 if dtype == torch.bfloat16 else 1e-5)
    assert rel(fd.grad.cpu(), fr.grad) < (2e-2 if dtype == torch.bfloat16 else 1e-4)


@pytest.mark.parametrize("train_flow", [False, True])
def test_realbasicvsr_training_step_gradients(dev, train_flow):
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    torch.manual_seed(3)
    net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=train_flow)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    g = torch.Generator().manual_seed(4)
    lr = torch.rand(1, 3, 3, 32, 32, generator=g)
    hr = torch.rand(1, 3, 3, 128, 128, generator=g)
    # oracle: fp32 autograd on CPU, Charbonnier-style loss as train.py uses (core/losses.py:10-18)
    P = {k: v.clone().requires_grad_(v.is_floating_point() and not k.endswith(("mean", "std"))) for k, v in sd.items()}
    sr_o, lq_o = O.realbasicvsr(lr.clone(), P)
    loss_o = torch.sqrt((sr_o - hr) ** 2 + 1e-9).mean() + torch.sqrt((lq_o - F.interpolate(hr[0], size=(32, 32), mode="bilinear")) ** 2 + 1e-9).mean()
    loss_o.backward()
    net = net.to(dev).train()
    x = lr.clone().to(dev)
    with torch.autocast("cuda", dtype=torch.bfloat16):
        sr, lq = net(x)
    assert sr.dtype == torch.float32 and sr.requires_grad
    loss = torch.sqrt((sr - hr.to(dev)) ** 2 + 1e-9).mean() + \
        torch.sqrt((lq - F.interpolate(hr[0].to(dev), size=(32, 32), mode="bilinear")) ** 2 + 1e-9).mean()
    loss.backward()
    assert abs(loss.item() - loss_o.item()) < 2e-3
    assert torch.allclose(x.cpu(), lq.detach().cpu())             # the caller's clip now holds the cleaned frames
    # per-tensor direction, and the direction of the whole gradient.  bf16 activations flip a few ReLU masks on
    # the 1x1 .. 4x4 pyramid levels of SPyNet, so tiny tensors there are noisier than the rest.
    got, want = [], []
    for name, p in net.named_parameters():
        ref = P[name].grad
        if not p.requires_grad:
            assert p.grad is None
            continue
        assert p.grad is not None, name
        assert torch.isfinite(p.grad).all(), name
        if ref is None or ref.norm() < 1e-7:
            continue
        got.append(p.grad.flatten().cpu())
        want.append(ref.flatten())
        assert cos(p.grad.cpu(), ref) > (0.90 if "spynet" in name else 0.97), (name, cos(p.grad.cpu(), ref))
    assert cos(torch.cat(got), torch.cat(want)) > 0.99
    assert rel(torch.cat(got), torch.cat(want)) < 0.1


@pytest.mark.parametrize("case", [
    # (segs, cout, k, h, w): shapes of the mma.sync weight-gradient kernel (7x7, 1x1, narrow segments, ragged widths)
    ([(0, 8)], 32, 7, 13, 37),
    ([(0, 32)], 64, 7, 9, 40),
    ([(0, 64)], 32, 7, 12, 33),
    ([(0, 16)], 2, 7, 6, 10),
    ([(0, 64), (64, 64)], 64, 1, 10, 35),
    ([(0, 3)], 64, 3, 11, 31),
    ([(0, 64)], 3, 3, 11, 31),
], ids=lambda c: f"k{c[2]}_{c[0]}_{c[1]}")
def test_wgrad_mma_matches_ffma_and_fp32(dev, case, monkeypatch):
    """dW / db of the warp-MMA kernel against the FFMA kernel on the same bf16 data (only the summation order differs)
    and against fp32 autograd."""
    from vsrlab_b200 import autograd as AG, ops
    segs, cout, k, h, w = case
    g = torch.Generator().manual_seed(5)
    cin = sum(c for _, c in segs)
    B = 3
    x = bf16r(torch.randn(B, cin, h, w, generator=g))
    dz = bf16r(torch.randn(B, cout, h, w, generator=g))
    cv = torch.nn.Conv2d(cin, cout, k, 1, k // 2)
    geom = AG._wgrad_geom(cv, tuple(segs))
    ins = [AG.to_cl16(x[:, off:off + c].to(dev)) for off, c in segs]
    dzd = AG.to_cl16(dz.to(dev))
    res = []
    for ffma in ("", "1"):
        if ffma:
            monkeypatch.setenv("VSRB_WGRAD_FFMA", "1")
        else:
            monkeypatch.delenv("VSRB_WGRAD_FFMA", raising=False)
        dw = torch.zeros(cout, cin, k, k, device=dev)
        db = torch.zeros(cout, device=dev)
        ops.conv2d_wgrad(geom, ins, [t.shape[1] for t in ins], dzd, dzd.shape[1], B, h, w, cin, dw, db)
        torch.cuda.synchronize()
        res.append((dw.cpu(), db.cpu()))
    wr = torch.zeros(cout, cin, k, k, requires_grad=True)
    (F.conv2d(x, wr, None, padding=k // 2) * dz).sum().backward()
    scale = wr.grad.abs().max().item()
    assert (res[0][0] - res[1][0]).abs().max().item() <= 1e-4 * scale
    assert (res[0][0] - wr.grad).abs().max().item() <= 1e-4 * scale
    assert (res[0][1] - dz.sum((0, 2, 3))).abs().max().item() <= 1e-3 * dz.sum((0, 2, 3)).abs().max().item()


def test_batched_wgrad_equals_per_use(dev):
    """Inside batched_wgrad() a conv used several times gets ONE weight-gradient launch from its _WeightNode; the
    parameter gradients must equal those of the per-use path, and hooks on the parameter must fire exactly once."""
    from vsrlab_b200 import autograd as AG
    torch.manual_seed(2)
    cv = torch.nn.Conv2d(64, 64, 3, 1, 1).to(dev)
    xs = [AG.to_cl16(bf16r(torch.randn(2, 64, 12, 20)).to(dev)).requires_grad_(True) for _ in range(3)]
    fired = []
    cv.weight.register_hook(lambda g_: fired.append(1))

    def run(batched):
        for t in xs:
            t.grad = None
        cv.zero_grad(set_to_none=True)
        fired.clear()
        y = 0
        if batched:
            with AG.batched_wgrad():
                for i, t in enumerate(xs):
                    y = y + AG.conv(cv, [t], [(0, 64)], "relu").float().mul(i + 1.0).sum()
        else:
            for i, t in enumerate(xs):
                y = y + AG.conv(cv, [t], [(0, 64)], "relu").float().mul(i + 1.0).sum()
        y.backward()
        return cv.weight.grad.clone(), cv.bias.grad.clone(), [t.grad.clone() for t in xs], len(fired)

    w0, b0, g0, n0 = run(False)
    w1, b1, g1, n1 = run(True)
    assert n1 == 1
    assert rel(w1, w0) < 1e-5 and rel(b1, b0) < 1e-5
    for a, b in zip(g1, g0):
        assert torch.equal(a, b)


def test_pixel_unshuffle2_matches_torch(dev):
    """vsrb_pixel_unshuffle2 (bf16 NHWC) against F.pixel_unshuffle: pure data movement, bit-exact."""
    from vsrlab_b200 import ops
    g = torch.Generator().manual_seed(9)
    for (n, h, w, c) in [(2, 5, 7, 64), (1, 3, 4, 8), (3, 16, 9, 32)]:
        src = torch.randn(n, c, 2 * h, 2 * w, generator=g).to(torch.bfloat16).to(dev).contiguous(memory_format=torch.channels_last)
        dst = torch.empty((n, 4 * c, h, w), dtype=torch.bfloat16, device=dev).contiguous(memory_format=torch.channels_last)
        ops.pixel_unshuffle2(src, dst, n, h, w, c)
        torch.cuda.synchronize()
        assert torch.equal(dst, F.pixel_unshuffle(src, 2))


def test_graphed_train_step_matches_eager(dev):
    """vsrlab_b200.graphs.GraphedTrainStep (forward + backward + clip + Adam replayed from one CUDA graph) follows the same
    loss trajectory as the eager loop from the same initial weights."""
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200.graphs import GraphedTrainStep
    g = torch.Generator().manual_seed(12)
    lr = torch.rand(2, 3, 3, 32, 32, generator=g).to(dev)
    hr = torch.rand(2, 3, 3, 128, 128, generator=g).to(dev)

    def loss_fn(out, hr_):
        sr, lq = out
        return torch.sqrt((sr - hr_) ** 2 + 1e-9).mean() + \
            torch.sqrt((lq - F.interpolate(hr_.flatten(0, 1), size=(32, 32), mode="bilinear").view_as(lq)) ** 2 + 1e-9).mean()

    def make():
        torch.manual_seed(21)
        net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=True)
        net = net.to(dev).train()
        return net, torch.optim.Adam(net.parameters(), lr=2e-4, capturable=True)

    net_e, opt_e = make()
    eager = []
    for _ in range(6):
        x = lr.clone()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            out = net_e(x)
        loss = loss_fn(out, hr)
        opt_e.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(net_e.parameters(), 1.0)
        opt_e.step()
        eager.append(loss.item())
    net_g, opt_g = make()
    step = GraphedTrainStep(net_g, opt_g, loss_fn, (lr, hr), clip_grad_norm=1.0, warmup=3)     # 3 real steps; capture runs nothing
    graphed = [step(lr, hr).item() for _ in range(3)]                                           # steps 4, 5 and 6
    assert eager[-1] < eager[0]
    for a_, b_ in zip(graphed, eager[3:]):
        assert abs(a_ - b_) < 2e-3, (graphed, eager)


def _charbonnier(a, b):
    return torch.sqrt((a - b) ** 2 + 1e-9).mean()


def _compute_loss(sr, hr, lq):
    """reference core/utils.py:235-240 (kornia `resize` = bilinear, align_corners=False, no antialias)."""
    _, _, c, h, w = lq.shape
    return _charbonnier(sr, hr) + _charbonnier(lq, F.interpolate(hr.flatten(0, 1), size=(h, w), mode="bilinear").view_as(lq))


def test_reference_amp_recipe_fp16_gradscaler_grad_accumulation(dev):
    """The reference's training sequence, verbatim (train.py:74,90-98; core/utils.py:270-280): fp16-requesting
    `torch.cuda.amp.autocast()`, `GradScaler` (loss scaled by 65 536), `num_grad_acc = 4` micro-steps,
    `unscale_` -> `clip_grad_norm_(1.0)` -> `scaler.step` -> `scaler.update` -> `scheduler.step` -> `zero_grad`.
    The kernels compute the scaled gradients in bf16 with fp32 accumulation: after `unscale_` they must be finite,
    match the unscaled bf16-autocast gradients, the scaler must not skip the step, and the loss must go down."""
    import warnings
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    num_grad_acc, clip = 4, 1.0
    g = torch.Generator().manual_seed(77)
    data = [(torch.rand(2, 3, 3, 32, 32, generator=g).to(dev), torch.rand(2, 3, 3, 128, 128, generator=g).to(dev))
            for _ in range(num_grad_acc)]

    def make():
        torch.manual_seed(8)
        net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=True)
        return net.to(dev).train()

    # (a) gradients of the recipe's accumulated, scaled backward == plain bf16-autocast gradients of the mean loss
    net_a = make()
    for lr, hr in data:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            sr, lq = net_a(lr.clone())
        (_compute_loss(sr, hr, lq) / num_grad_acc).backward()
    want = {n: p.grad.clone() for n, p in net_a.named_parameters()}

    net = make()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.99))
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=600000, eta_min=1e-7)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        scaler = torch.cuda.amp.GradScaler()
    assert scaler.get_scale() == 65536.0
    losses, stepped = [], 0
    for epoch in range(4):
        for i, (lr, hr) in enumerate(data):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                ctx = torch.cuda.amp.autocast()
            with ctx:
                x = lr.clone()
                sr, lq = net(x)
                loss = _compute_loss(sr, hr, lq)
            assert sr.dtype == torch.float32 and lq.dtype == torch.float32
            # update_weights (core/utils.py:270-280)
            scaler.scale(loss / num_grad_acc).backward()
            if (i + 1) % num_grad_acc == 0:
                scaler.unscale_(opt)
                if epoch == 0:
                    got = torch.cat([p.grad.flatten() for _, p in net.named_parameters()])
                    ref = torch.cat([want[n].flatten() for n, _ in net.named_parameters()])
                    assert torch.isfinite(got).all()
                    assert cos(got.cpu(), ref.cpu()) > 0.999 and rel(got.cpu(), ref.cpu()) < 0.05
                torch.nn.utils.clip_grad_norm_(net.parameters(), clip)
                before = [p.detach().clone() for p in net.parameters()]
                scaler.step(opt)
                scaler.update()
                sched.step()
                opt.zero_grad()
                stepped += int(any(not torch.equal(a, b.detach()) for a, b in zip(before, net.parameters())))
            losses.append(loss.item())
    assert stepped == 4                                     # no step skipped by the inf check
    assert scaler.get_scale() >= 65536.0
    first, last = sum(losses[:num_grad_acc]), sum(losses[-num_grad_acc:])
    assert last < first, (first, last)


def test_submodules_are_differentiable(dev):
    """Every drop-in module is differentiable on its own, like the reference's nn.Modules (not only the two top-level
    models): ConvReLU, ResidualBlock, ResidualConv, PixelShufflePack, SpynetModule, Spynet, flow_warp, cleaner."""
    from vsrlab.core.modules.conv import ConvReLU, ResidualBlock, ResidualConv
    from vsrlab.core.modules.upsampling import PixelShufflePack
    from vsrlab.vsr.models.RealBasicVSR.modules.spynet import Spynet, flow_warp
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import IterativeRefinement
    g = torch.Generator().manual_seed(31)

    def check(mod, x, ref_fn, tol=3e-2):
        """module output / gradients vs fp32 autograd through the oracle on CPU"""
        sd = {k: v.detach().cpu().clone().requires_grad_(v.is_floating_point() and v.requires_grad) for k, v in mod.state_dict(keep_vars=True).items()}
        xr = x.clone().requires_grad_(True)
        yr = ref_fn(xr, sd)
        w = torch.randn(yr.shape, generator=g)
        (yr * w).sum().backward()
        xd = x.clone().to(dev).requires_grad_(True)
        y = mod.to(dev)(xd)
        assert y.grad_fn is not None and y.dtype == torch.float32 and y.shape == yr.shape
        (y * w.to(dev)).sum().backward()
        assert rel(y.detach().cpu(), yr.detach()) < tol
        assert cos(xd.grad.cpu(), xr.grad) > 0.99
        for n, p in mod.named_parameters():
            if p.requires_grad and sd[n].grad is not None and sd[n].grad.norm() > 1e-6:
                assert p.grad is not None and cos(p.grad.cpu(), sd[n].grad) > 0.97, n

    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", RuntimeWarning)          # "training path runs bf16" notice outside autocast
        torch.manual_seed(1)
        check(ConvReLU(16, 32, 3, 1, 1), torch.randn(2, 16, 12, 20, generator=g),
              lambda x, P: O.relu(O.conv(x, P, "conv.0")))
        check(ResidualBlock(3, 64, 2), torch.rand(2, 3, 12, 20, generator=g), lambda x, P: O.residual_block(x, P, ""))
        check(ResidualConv(64), torch.randn(1, 64, 9, 11, generator=g),
              lambda x, P: x + O.conv(O.relu(O.conv(x, P, "conv1")), P, "conv2"))
        check(PixelShufflePack(64, 64, 2), torch.randn(1, 64, 6, 10, generator=g), lambda x, P: O.pixel_shuffle_pack(x, P, ""))
        ir = IterativeRefinement(64, 1)
        x5 = torch.rand(1, 2, 3, 12, 16, generator=g)
        check(ir, x5, lambda x, P: O.cleaner(x.clone(), {"cleaner." + k: v for k, v in P.items()}))
        # flow_warp: gradient wrt features and flow
        x = torch.randn(2, 8, 11, 13, generator=g)
        fl = (torch.rand(2, 11, 13, 2, generator=g) - 0.5) * 6
        xr, fr = x.clone().requires_grad_(True), fl.clone().requires_grad_(True)
        O.flow_warp(xr, fr, "zeros").pow(2).sum().backward()
        xd, fd = x.to(dev).requires_grad_(True), fl.to(dev).requires_grad_(True)
        y = flow_warp(xd, fd)
        assert y.grad_fn is not None
        y.pow(2).sum().backward()
        assert rel(xd.grad.cpu(), xr.grad) < 1e-4 and rel(fd.grad.cpu(), fr.grad) < 1e-3
        # Spynet trained stand-alone: parameters get gradients
        torch.manual_seed(3)
        sp = Spynet().to(dev)
        a, b = torch.rand(1, 3, 64, 64, generator=g).to(dev), torch.rand(1, 3, 64, 64, generator=g).to(dev)
        fl = sp(a, b)
        assert fl.grad_fn is not None and fl.shape == (1, 2, 64, 64)
        fl.abs().sum().backward()
        assert all(p.grad is not None and torch.isfinite(p.grad).all() for p in sp.parameters())
    # with nothing to differentiate the fast raw-kernel path is used and returns a plain tensor
    with torch.no_grad():
        assert sp(a, b).grad_fn is None


def test_unsupported_conv_geometry_is_refused(dev):
    """ConvReLU forwards *args to nn.Conv2d (reference conv.py:19); a stride-2 or dilated conv must fail loudly."""
    from vsrlab.core.modules.conv import ConvReLU
    from vsrlab_b200 import VsrbError
    m = ConvReLU(16, 16, 3, 2, 1).to(dev)
    with pytest.raises(VsrbError), torch.no_grad():
        m(torch.randn(1, 16, 8, 8, device=dev))


def _ddp_worker(rank, world, port, q):
    import os
    import torch.distributed as dist
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    torch.manual_seed(0)
    model = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=True).to(dev).train()
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[rank])          # reference core/utils.py:147-151
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.99))
    g = torch.Generator().manual_seed(100 + rank)                                      # every rank its own shard of the data
    lr = torch.rand(2, 3, 3, 32, 32, generator=g).to(dev)
    hr = torch.rand(2, 3, 3, 128, 128, generator=g).to(dev)
    losses = []
    for _ in range(3):
        with torch.autocast("cuda", dtype=torch.bfloat16):
            sr, lq = net(lr.clone())
        loss = _compute_loss(sr, hr, lq)
        opt.zero_grad(set_to_none=True)
        loss.backward()                                                                # DDP all-reduce (NCCL) fires here
        torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
        opt.step()
        losses.append(loss.item())
    flat = torch.cat([p.detach().flatten() for p in model.parameters()])
    ref = flat.clone()
    dist.broadcast(ref, 0)
    grads = torch.cat([p.grad.flatten() for p in model.parameters()])
    gref = grads.clone()
    dist.broadcast(gref, 0)
    q.put((rank, bool(torch.equal(flat, ref)), bool(torch.equal(grads, gref)), losses, bool(torch.isfinite(flat).all())))
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_ddp_nccl_two_ranks_replicas_stay_identical():
    """Training-side multi-GPU split (SURVEY §8e): DDP over NCCL, different data per rank, all-reduced gradients and
    weights bit-identical across replicas after three optimizer steps."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_ddp_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=600) for _ in range(2))
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for rank, same_w, same_g, losses, finite in res:
        assert same_w and same_g and finite, (rank, same_w, same_g)
    assert res[0][3] != res[1][3]                       # the ranks really saw different data


def test_training_forward_is_graphed_after_warmup_and_matches_eager(dev):
    """vsrlab_b200.graphs.training_forward: after three eager calls with one shape the model's forward and backward replay
    from CUDA graphs inside the caller's unchanged AMP loop (autocast + GradScaler + accumulation + clip + Adam).  Same
    losses and weights as the eager path (the weight-gradient atomics make the two runs differ in the last bits only),
    in-place refinement of the input kept, other shapes / no_grad calls unaffected."""
    import warnings
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import graphs

    def run(use_graphs):
        graphs.TRAIN_GRAPHS = use_graphs
        torch.manual_seed(0)
        net = RealBasicVSR(cleaning_blocks=1, mid_channels=64, upscale=4, res_blocks=1, pretrained_flow=False, train_flow=True).to(dev).train()
        opt = torch.optim.Adam(net.parameters(), lr=1e-4)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            scaler = torch.cuda.amp.GradScaler()
        g = torch.Generator().manual_seed(1)
        losses = []
        for i in range(8):
            lr = torch.rand(2, 5, 3, 32, 32, generator=g).to(dev)
            hr = torch.rand(2, 5, 3, 128, 128, generator=g).to(dev)
            lr0 = lr.clone()
            with torch.autocast("cuda", dtype=torch.float16):
                sr, lq = net(lr)
                loss = torch.sqrt((sr - hr) ** 2 + 1e-9).mean() + torch.sqrt((lq - F.interpolate(hr.flatten(0, 1), size=(32, 32), mode="bilinear").view_as(lq)) ** 2 + 1e-9).mean()
            assert torch.equal(lr, lq.detach()) and not torch.equal(lr, lr0)          # refined in place, as the reference
            scaler.scale(loss / 2).backward()
            if i % 2 == 1:
                scaler.unscale_(opt)
                torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
                scaler.step(opt)
                scaler.update()
                opt.zero_grad()
            losses.append(loss.item())
        graphed = graphs.graphed_patterns(net) > 0
        if graphed:
            entry = next(e for e in graphs._train_entries[id(net)]["by_key"].values() if e.graphed is not None)
            # two forwards before one backward: the second must not clobber what the graph saved for the first
            xa, xb = torch.rand(2, 5, 3, 32, 32, device=dev), torch.rand(2, 5, 3, 32, 32, device=dev)
            with torch.autocast("cuda", dtype=torch.float16):
                sa, _ = net(xa.clone())
                assert entry.graphed.pending
                sb, _ = net(xb.clone())                     # runs eagerly
            opt.zero_grad()
            (sa.mean() + 2 * sb.mean()).backward()
            ga = torch.cat([p.grad.flatten() for p in net.parameters()])
            assert not entry.graphed.pending
            graphs.TRAIN_GRAPHS = False
            opt.zero_grad()
            with torch.autocast("cuda", dtype=torch.float16):
                sa2, _ = net(xa.clone())
                sb2, _ = net(xb.clone())
            (sa2.mean() + 2 * sb2.mean()).backward()
            graphs.TRAIN_GRAPHS = True
            ge = torch.cat([p.grad.flatten() for p in net.parameters()])
            assert cos(ga, ge) > 0.9999 and rel(ga, ge) < 2e-2
            opt.zero_grad()
            # gradient accumulation over two REPLAYED micro-steps: p.grad must be g1 + g2 (not a view of the graph's static
            # gradient buffer that the second replay overwrites)
            def accumulate():
                opt.zero_grad(set_to_none=True)
                for xin, wgt in ((xa, 1.0), (xb, 3.0)):
                    with torch.autocast("cuda", dtype=torch.float16):
                        s_, _ = net(xin.clone())
                    (wgt * s_.mean()).backward()
                return torch.cat([p.grad.flatten() for p in net.parameters()])
            g_acc = accumulate()
            assert not entry.graphed.pending
            graphs.TRAIN_GRAPHS = False
            g_ref = accumulate()
            graphs.TRAIN_GRAPHS = True
            assert cos(g_acc, g_ref) > 0.9999 and rel(g_acc, g_ref) < 2e-2, (cos(g_acc, g_ref), rel(g_acc, g_ref))
            opt.zero_grad()
        # another shape and a no_grad call keep working
        with torch.autocast("cuda", dtype=torch.float16):
            sr2, _ = net(torch.rand(1, 3, 3, 16, 24, device=dev))
        sr2.mean().backward()
        net.eval()
        with torch.no_grad():
            sr3, _ = net(torch.rand(1, 3, 3, 16, 24, device=dev))
        assert sr3.shape == (1, 3, 3, 64, 96)
        return losses, torch.cat([p.detach().flatten() for p in net.parameters()]), graphed

    try:
        l_g, w_g, graphed = run(True)
        l_e, w_e, not_graphed = run(False)
    finally:
        graphs.TRAIN_GRAPHS = True
    assert graphed and not not_graphed
    assert max(abs(a - b) / abs(b) for a, b in zip(l_g, l_e)) < 2e-3, (l_g, l_e)
    assert cos(w_g, w_e) > 0.99999 and rel(w_g, w_e) < 1e-3
