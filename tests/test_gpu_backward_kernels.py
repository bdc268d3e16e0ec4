"""Kernel-level checks of the backward pass against float64 references on bf16-representable operands.

The training step spends its convolution time in three places: the input-gradient convs (the forward kernels on dz with
weights packed `transpose = 1`), the tensor-core weight gradient (`wgrad_tc_kernel`, single launch or one launch over the
uses of a recurrent conv) and the fused residual-block node (`ResBlockFn`).  Each is compared here with the same
operation computed by torch in float64 (on the GPU) from the same bf16 values, at the bounds of the forward tests:

* input gradient: max-abs error <= 2^-8 * max(|ref|, 1) (the output is stored as bf16: half an ulp is 2^-9), padded
  output channels exactly 0, CTA-pair and single-CTA kernels bit-identical;
* weight gradient: max-abs error <= 1e-3 * max|ref| - and each test shows that this bound is below half of what one
  64-pixel tile (4 rows x 16 pixels, the kernel's unit of work) contributes, so a lost or doubled tile fails;
  bias gradient rel-L2 <= 1e-4;
* residual-block node: cos >= 0.9999 and rel-L2 <= 1e-2 per gradient tensor against fp64 autograd through the oracle,
  whose activations are not rounded to bf16 (the kernels' are); swapping the two weight groups swaps the results.
"""
import zlib

import pytest
import torch
import torch.nn.functional as F
from torch.nn.grad import conv2d_input, conv2d_weight

from oracle import vsr_oracle as O

pytestmark = pytest.mark.gpu

CL = torch.channels_last
# the kernel selection switches of the conv launcher (read at pack and at launch time)
SWITCHES = ("VSRB_RING_MIN_ROWS", "VSRB_TC_NO_RING", "VSRB_TC_NO_PAIR", "VSRB_TC_NO_STACK", "VSRB_RING_DEBUG",
            "VSRB_WG_DEBUG", "VSRB_TC_DEBUG")


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    from vsrlab_b200 import load
    load()
    return torch.device("cuda:0")


def bf16r(x):
    return x.to(torch.bfloat16).to(x.dtype)


def rel(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


def cos(a, b):
    return F.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0).item()


def maxabs(a, b):
    return (a.double() - b.double()).abs().max().item()


def env(monkeypatch, **kv):
    """Clear every kernel switch, then set `kv`."""
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in kv.items():
        monkeypatch.setenv(k, v)


def randn(shape, gen, dev, scale=1.0):
    """bf16-representable normal values, fp32, on `dev`."""
    return bf16r(torch.randn(shape, generator=gen, device=dev) * scale)


def make_conv(cin, cout, k, gen, dev, wscale=1.0):
    cv = torch.nn.Conv2d(cin, cout, k, 1, k // 2).to(dev)
    with torch.no_grad():
        cv.weight.copy_(randn(cv.weight.shape, gen, dev, wscale / (cin * k * k) ** 0.5))
        cv.bias.copy_(randn(cv.bias.shape, gen, dev, 0.1))
    return cv


def nhwc(x, c_alloc, fill=0.0):
    """[B, c, h, w] fp32 -> bf16 channels_last [B, c_alloc, h, w]; channels >= c hold `fill`."""
    B, c, h, w = x.shape
    t = torch.full((B, c_alloc, h, w), fill, dtype=torch.bfloat16, device=x.device).contiguous(memory_format=CL)
    t[:, :c] = x
    return t


def seed_of(*key):
    return zlib.crc32(repr(key).encode())          # stable across processes (str hashes are salted)


def pad16(c):
    return (c + 15) // 16 * 16


def ring_steps_reset():
    import ctypes
    from vsrlab_b200 import _lib as L
    stats = (ctypes.c_uint64 * 8)()
    L.check(L.load().vsrb_ring_debug_stats(stats, 1), "vsrb_ring_debug_stats")
    return stats[2]


# ----------------------------------------------------------------------------------------------------------------------
# A. input-gradient convolution: PackedConvT + conv2d_fwd
# ----------------------------------------------------------------------------------------------------------------------
# forward layer -> (segments as autograd.py passes them, cout, k); the gradient conv maps cout -> sum(segment channels)
LAYERS = {
    "rb64": ([(0, 64)], 64, 3),                   # resblock convs, conv_last.0: 64 -> 64, ring-walk geometry
    "stem67": ([(3, 64), (0, 3)], 64, 3),         # propagation stem cat([lr, feat]): 64 -> 67 (padded to 80)
    "cstem3": ([(0, 3)], 64, 3),                  # cleaner stem: 64 -> 3
    "img3": ([(0, 64)], 3, 3),                    # cleaner.conv / conv_last.2: 3 (16-channel dz) -> 64
    "up256": ([(0, 64)], 256, 3),                 # upsamplers (dz un-shuffled): 256 -> 64
    "point": ([(0, 64), (64, 64)], 64, 1),        # point_conv 1x1: 64 -> 128
    "sp8to32": ([(0, 8)], 32, 7),                 # SPyNet's 7x7 stack (train_flow), each reversed
    "sp32to64": ([(0, 32)], 64, 7),
    "sp64to32": ([(0, 64)], 32, 7),
    "sp32to16": ([(0, 32)], 16, 7),
    "sp16to2": ([(0, 16)], 2, 7),
}
RING_LAYERS = ("rb64",)

DGRAD_CASES = [
    # (layer, images per group, h, w, groups, fused residual)
    *[(name, 2, 13, 37, 1, False) for name in LAYERS],        # ragged: h % 4, w % 16 and w % 30 all non-zero
    *[(name, 1, 1, 23, 1, False) for name in LAYERS],         # a single row
    ("rb64", 2, 13, 37, 1, True),
    ("rb64", 1, 1, 23, 1, True),
    ("rb64", 8, 64, 64, 2, False),                            # propagation batch: both directions as weight groups
    ("rb64", 8, 64, 64, 2, True),                             # ... as ResBlockFn.dgrad passes conv1 (skip fused)
    ("stem67", 8, 64, 64, 2, False),
    ("rb64", 120, 64, 64, 1, False),                          # cleaner batch: the ring-walk kernel by default
    ("rb64", 120, 64, 64, 1, True),
    ("cstem3", 120, 64, 64, 1, False),
    ("img3", 120, 64, 64, 1, False),
    ("rb64", 2, 256, 256, 1, False),                          # HR: conv_last.0, the upsampler, conv_last.2
    ("up256", 2, 256, 256, 1, False),
    ("img3", 2, 256, 256, 1, False),
    *[(name, 4, 64, 64, 1, False) for name in LAYERS if name.startswith("sp")],   # SPyNet's top pyramid level
]

# kernel choices for one launch: ring = ring-walk kernel forced; pair = the tile kernel (CTA pairs where the plan allows);
# single = the tile kernel without pairs; classic = the un-stacked layout
VARIANTS = {
    "default": {},
    "ring": {"VSRB_RING_MIN_ROWS": "0"},
    "pair": {"VSRB_TC_NO_RING": "1"},
    "single": {"VSRB_TC_NO_RING": "1", "VSRB_TC_NO_PAIR": "1"},
    "classic": {"VSRB_TC_NO_RING": "1", "VSRB_TC_NO_STACK": "1"},
}


@pytest.mark.parametrize("case", DGRAD_CASES, ids=lambda c: f"{c[0]}_n{c[1]}_{c[2]}x{c[3]}_g{c[4]}{'_res' if c[5] else ''}")
def test_input_gradient_conv(dev, case, monkeypatch):
    from vsrlab_b200 import ops
    from vsrlab_b200._lib import ACT_NONE, BF16, VsrbError
    name, n, h, w, G, residual = case
    segs, cout, k = LAYERS[name]
    cin = sum(c for _, c in segs)
    gen = torch.Generator(device=dev).manual_seed(seed_of(*case))
    convs = [make_conv(cin, cout, k, gen, dev) for _ in range(G)]
    B = n * G
    dz = randn((B, cout, h, w), gen, dev)
    dzt = nhwc(dz, pad16(cout))                       # the training path's dz: padded channels hold zeros
    res = randn((B, cin, h, w), gen, dev) if residual else None
    rest = nhwc(res, cin) if residual else None

    def ref_for(order):
        parts = []
        for gi in range(G):
            wgt = convs[order[gi]].weight.detach().double()
            parts.append(conv2d_input((n, cin, h, w), wgt, dz[gi * n:(gi + 1) * n].double(), padding=k // 2))
        r = torch.cat(parts)
        return r + res.double() if residual else r

    ref = ref_for(list(range(G)))
    tol = 2.0 ** -8 * max(ref.abs().max().item(), 1.0)
    cpad = pad16(cin)
    outs = {}
    for var, kv in VARIANTS.items():
        if var == "ring" and name not in RING_LAYERS:
            continue
        env(monkeypatch, VSRB_RING_DEBUG="64", **kv)  # bit 64: the ring-walk kernel counts its steps
        pt = ops.PackedConvT(convs, BF16)
        assert pt.cout_pad == cpad
        out = torch.full((B, cpad, h, w), float("nan"), dtype=torch.bfloat16, device=dev).contiguous(memory_format=CL)
        ring_steps_reset()
        try:
            ops.conv2d_fwd(pt, [dzt], [dzt.shape[1]], B, h, w, act=ACT_NONE, out=out, out_c=cpad, residual=rest,
                           res_c=cin if residual else 0)
        except VsrbError as e:
            # 7x7 plans that keep half of a large weight block resident per CTA only exist as pairs: without pairs (or
            # in the un-stacked layout) the launcher must refuse loudly, not fall back
            assert k == 7 and var in ("single", "classic") and "does not fit" in str(e), (var, str(e))
            continue
        torch.cuda.synchronize()
        assert ops.debug_status() == 0
        steps = ring_steps_reset()
        if var in ("pair", "single", "classic"):
            assert steps == 0, var
        elif var == "ring" or (var == "default" and name in RING_LAYERS and B * h >= 120 * 64):
            assert steps > 0, f"{var}: the launch did not run on the ring-walk kernel"
        got = out[:, :cin].double()
        err = maxabs(got, ref)
        assert err <= tol, (var, err, tol)
        assert (out[:, cin:] == 0).all(), var                 # padded channels: exactly 0, not NaN or stale
        outs[var] = out
    assert "default" in outs and "pair" in outs
    if "single" in outs:
        assert torch.equal(outs["pair"], outs["single"])     # same MMAs in the same order, as M = 256 across two SMs
    if G == 2:
        # each group has its own weights: the other group's weights give a result the bound would reject
        assert maxabs(outs["default"][:, :cin], ref_for([1, 0])) > 8 * tol


# ----------------------------------------------------------------------------------------------------------------------
# B. one weight-gradient launch: ops.conv2d_wgrad on the tensor-core shapes
# ----------------------------------------------------------------------------------------------------------------------
WGRAD_LAYERS = {
    "rb64": ([(0, 64)], 64),          # 3x3 64 -> 64
    "up256": ([(0, 64)], 256),        # 3x3 64 -> 256: four 64-wide output blocks in one launch (blockIdx.y)
    "stem67": ([(3, 64), (0, 3)], 64),   # 64-channel segment on wgrad_tc (seg_off 3, cin_total 67), 3 channels on wgrad_taps
}
WGRAD_SHAPES = [(1, 20, 28), (120, 64, 64), (4, 45, 77)]   # one CTA; the training batch (7 680 tiles); ragged, 7 CTAs


def tile_movement(x64, dz64, k):
    """Smallest max-abs change of the fp64 weight gradient when one full 64-pixel tile (4 rows x 16 pixels of one image,
    the weight-gradient kernel's unit of work) is left out; sampled at the first, a middle and the last full tile."""
    B, _, h, w = dz64.shape
    ty_n, tx_n = h // 4, w // 16
    moves = []
    for i, ty, tx in ((0, 0, 0), (B // 2, ty_n // 2, tx_n // 2), (B - 1, ty_n - 1, tx_n - 1)):
        m = torch.zeros_like(dz64[i:i + 1])
        m[..., 4 * ty:4 * ty + 4, 16 * tx:16 * tx + 16] = dz64[i:i + 1, :, 4 * ty:4 * ty + 4, 16 * tx:16 * tx + 16]
        moves.append(conv2d_weight(x64[i:i + 1], (dz64.shape[1], x64.shape[1], k, k), m, padding=k // 2).abs().max().item())
    return min(moves)


@pytest.mark.parametrize("shape", WGRAD_SHAPES, ids=lambda s: "n%d_%dx%d" % s)
@pytest.mark.parametrize("name", list(WGRAD_LAYERS))
def test_weight_gradient_single_launch(dev, name, shape, monkeypatch):
    from vsrlab_b200 import autograd as AG, ops
    segs, cout = WGRAD_LAYERS[name]
    B, h, w = shape
    cin = sum(c for _, c in segs)
    gen = torch.Generator(device=dev).manual_seed(seed_of(name, *shape))
    x = randn((B, cin, h, w), gen, dev)                   # OIHW channel order (stem: [lr 3 | feat 64])
    dz = randn((B, cout, h, w), gen, dev)
    # the kernels read their segments and the first `cout` dz channels only: every other channel holds NaN
    ins = [nhwc(x[:, off:off + c], pad16(c) + (16 if c % 16 == 0 else 0), float("nan")) for off, c in segs]
    dzt = nhwc(dz, cout + 16, float("nan"))
    x64, dz64 = x.double(), dz.double()
    ref = conv2d_weight(x64, (cout, cin, 3, 3), dz64, padding=1)
    ref_b = dz64.sum((0, 2, 3))
    tol = 1e-3 * ref.abs().max().item()
    move = tile_movement(x64, dz64, 3)
    assert tol < 0.5 * move, (tol, move)                  # one lost or doubled tile would exceed the bound
    geom = AG._wgrad_geom(torch.nn.Conv2d(cin, cout, 3, 1, 1), tuple(segs))

    def run(dw, db):
        ops.conv2d_wgrad(geom, ins, [t.shape[1] for t in ins], dzt, dzt.shape[1], B, h, w, cin, dw, db)
        torch.cuda.synchronize()
        assert ops.debug_status() == 0

    env(monkeypatch)
    dw = torch.zeros(cout, cin, 3, 3, device=dev)
    db = torch.zeros(cout, device=dev)
    run(dw, db)
    dw1, db1 = dw.clone(), db.clone()
    assert torch.isfinite(dw1).all() and torch.isfinite(db1).all()
    assert maxabs(dw1, ref) <= tol, (maxabs(dw1, ref), tol)
    assert rel(db1, ref_b) <= 1e-4
    run(dw, db)                                           # a second call accumulates
    assert maxabs(dw, 2 * dw1) <= tol and maxabs(dw / 2, ref) <= tol
    assert rel(db, 2 * db1) <= 1e-4


# ----------------------------------------------------------------------------------------------------------------------
# C. one launch over the uses of a recurrent conv: ops.conv2d_wgrad_multi and _WeightNode
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("bias", [True, False], ids=["bias", "nobias"])
@pytest.mark.parametrize("n_chunks", [1, 2, 15, 16, 17, 33])
def test_weight_gradient_multi_chunk(dev, n_chunks, bias, monkeypatch):
    """The launcher walks the chunks in groups of 16 (one tensor map pair per chunk in the kernel parameters); the bias
    rides along once per group.  Chunks are separate allocations, so a chunk read through the wrong pointer shows."""
    from vsrlab_b200 import autograd as AG, ops
    env(monkeypatch)
    n, h, w = 8, 64, 64
    gen = torch.Generator(device=dev).manual_seed(1000 + n_chunks)
    xs = [randn((n, 64, h, w), gen, dev) for _ in range(n_chunks)]
    dzs = [randn((n, 64, h, w), gen, dev) for _ in range(n_chunks)]
    chunks = [([nhwc(x, 64)], nhwc(dz, 64)) for x, dz in zip(xs, dzs)]
    x64, dz64 = torch.cat(xs).double(), torch.cat(dzs).double()
    ref = conv2d_weight(x64, (64, 64, 3, 3), dz64, padding=1)
    ref_b = dz64.sum((0, 2, 3))
    tol = 1e-3 * ref.abs().max().item()
    assert tol < 0.5 * tile_movement(x64, dz64, 3)
    geom = AG._wgrad_geom(torch.nn.Conv2d(64, 64, 3, 1, 1), ((0, 64),))
    dw = torch.zeros(64, 64, 3, 3, device=dev)
    db = torch.zeros(64, device=dev) if bias else None
    ops.conv2d_wgrad_multi(geom, chunks, [64], 64, n, h, w, 64, dw, db)
    torch.cuda.synchronize()
    assert ops.debug_status() == 0
    assert maxabs(dw, ref) <= tol, (maxabs(dw, ref), tol)
    # the same gradient from one launch on the concatenated batch
    dw_c = torch.zeros_like(dw)
    db_c = torch.zeros_like(db) if bias else None
    x_cat = torch.cat([c[0][0] for c in chunks]).contiguous(memory_format=CL)
    dz_cat = torch.cat([c[1] for c in chunks]).contiguous(memory_format=CL)
    ops.conv2d_wgrad(geom, [x_cat], [64], dz_cat, 64, n * n_chunks, h, w, 64, dw_c, db_c)
    torch.cuda.synchronize()
    assert maxabs(dw, dw_c) <= tol
    if bias:
        assert rel(db, ref_b) <= 1e-4 and rel(db, db_c) <= 1e-4


def test_batched_wgrad_scope_17_uses(dev, monkeypatch):
    """17 uses of one conv inside batched_wgrad(): one _WeightNode launches the multi-chunk weight gradient (two groups of
    chunks); the parameter gets the fp64 gradient, and its hooks fire once."""
    from vsrlab_b200 import autograd as AG
    env(monkeypatch)
    gen = torch.Generator(device=dev).manual_seed(17)
    cv = make_conv(64, 64, 3, gen, dev)
    xs = [randn((8, 64, 64, 64), gen, dev) for _ in range(17)]
    gys = [randn((8, 64, 64, 64), gen, dev) for _ in range(17)]
    fired = {"w": 0, "b": 0}
    cv.weight.register_hook(lambda _g: fired.__setitem__("w", fired["w"] + 1))
    cv.bias.register_hook(lambda _g: fired.__setitem__("b", fired["b"] + 1))
    loss = 0
    with AG.batched_wgrad():
        for x, gy in zip(xs, gys):
            y = AG.conv(cv, [nhwc(x, 64)], [(0, 64)], "none")
            loss = loss + (y.float() * gy).sum()
    loss.backward()
    torch.cuda.synchronize()
    assert fired == {"w": 1, "b": 1}
    # no activation: dz of use k is exactly gy_k, so the fp64 reference is the exact gradient of these operands
    x64, g64 = torch.cat(xs).double(), torch.cat(gys).double()
    ref = conv2d_weight(x64, (64, 64, 3, 3), g64, padding=1)
    assert maxabs(cv.weight.grad, ref) <= 1e-3 * ref.abs().max().item()
    assert rel(cv.bias.grad, g64.sum((0, 2, 3))) <= 1e-4


# ----------------------------------------------------------------------------------------------------------------------
# D. ResBlockFn with two weight groups (the propagation's backward and forward ResidualBlocks)
# ----------------------------------------------------------------------------------------------------------------------
N_USES = 17                  # > 16: the weight gradients of every conv go through two groups of chunks


def _propagation_blocks(dev):
    from vsrlab.core.modules.conv import ResidualBlock
    gen = torch.Generator(device=dev).manual_seed(23)
    rbs = []
    for _ in range(2):
        rb = ResidualBlock(67, 64, 2).to(dev)
        with torch.no_grad():
            for name, p in rb.named_parameters():
                if name.endswith("weight"):
                    fan = p.shape[1] * 9
                    p.copy_(randn(p.shape, gen, dev, (1.0 if name.startswith("conv.") else 0.5) / fan ** 0.5))
                else:
                    p.copy_(randn(p.shape, gen, dev, 0.1))
        rbs.append(rb)
    return rbs


def _run_resblocks(rbs, feats, lrs, wts):
    """loss = sum_k w_k . resblock(rbs, [feat_k, lr_k]); returns (input gradients, parameter gradients per block)."""
    from vsrlab_b200 import autograd as AG
    for rb in rbs:
        rb.zero_grad(set_to_none=True)
    fi = [nhwc(f, 64).requires_grad_(True) for f in feats]
    li = [nhwc(l, 16).requires_grad_(True) for l in lrs]
    loss = 0
    with AG.batched_wgrad():
        for f, l, wk in zip(fi, li, wts):
            y = AG.resblock(tuple(rbs), [f, l], [(3, 64), (0, 3)])
            loss = loss + (y.float() * wk).sum()
    loss.backward()
    torch.cuda.synchronize()
    return [t.grad for t in fi], [t.grad for t in li], [{k: p.grad.clone() for k, p in rb.named_parameters()} for rb in rbs]


def _emulated_resblock(x, P, gy):
    """ResBlockFn's forward and backward in fp64 from the bf16 operands, rounding to bf16 wherever the kernels store a
    tensor (activations, input gradients with the fused skip term, the LeakyReLU gradient).  Returns (dx, {name: grad})."""
    r = bf16r
    nb = O.count_blocks(P, "")

    def conv(t, name):
        return F.conv2d(t, P[name + ".weight"], P[name + ".bias"], padding=1)

    def dgrad(name, dz, shape):
        return conv2d_input(shape, P[name + ".weight"], dz, padding=1)
    grads = {}

    def wgrad(name, xin, dz):
        grads[name + ".weight"] = conv2d_weight(xin, P[name + ".weight"].shape, dz, padding=1)
        grads[name + ".bias"] = dz.sum((0, 2, 3))
    x0 = r(O.lrelu(conv(x, "conv.0")))
    acts, a = [x0], x0
    for i in range(nb):
        t = r(O.relu(conv(a, f"res_block.{i}.conv1")))
        a = r(conv(t, f"res_block.{i}.conv2") + a)
        acts += [t, a]
    g = gy
    for i in range(nb - 1, -1, -1):
        xin, t = acts[2 * i], acts[2 * i + 1]
        c1, c2 = f"res_block.{i}.conv1", f"res_block.{i}.conv2"
        wgrad(c2, t, g)
        dz1 = r(dgrad(c2, g, t.shape)) * (t > 0)
        wgrad(c1, xin, dz1)
        g = r(dgrad(c1, dz1, xin.shape) + g)
    dz0 = r(torch.where(x0 > 0, g, g * 0.1))
    wgrad("conv.0", x, dz0)
    return r(dgrad("conv.0", dz0, x.shape)), grads


def test_resblock_node_two_groups(dev, monkeypatch):
    """The propagation's two ResidualBlocks (segments [(3, 64), (0, 3)], 2 sub-blocks) as the weight groups of one
    ResBlockFn per use, 8 images per group at 64 x 64, 17 uses inside one batched_wgrad() scope.

    Two references, both fp64 from the same bf16 operands:
    * the same arithmetic with every tensor the kernels store rounded to bf16 (`_emulated_resblock`): what is left is fp32
      accumulation order (and the rare bf16 rounding it tips), so cos >= 0.9999 and rel-L2 <= 1e-2 per tensor.  Measured
      on a B200 (1000 W): worst cos 0.999991, worst rel-L2 4.4e-3;
    * autograd through the oracle, whose activations stay fp64.  Against it the emulation itself is 3.4e-2 .. 4.0e-2
      rel-L2 off on the conv1 gradients (cos >= 0.9992; four seeds, 8 images at 48 x 48 on the CPU): bf16 activations
      flip a few ReLU masks of conv1's output, and each flip moves a whole term.  So the bound is cos >= 0.998, rel-L2 <= 8e-2;
      measured on a B200: worst cos 0.999202, worst rel-L2 4.1e-2, i.e. what the rounding alone gives."""
    from vsrlab_b200 import ops
    env(monkeypatch)
    n, h, w = 8, 64, 64
    rbs = _propagation_blocks(dev)
    gen = torch.Generator(device=dev).manual_seed(24)
    feats = [randn((2 * n, 64, h, w), gen, dev) for _ in range(N_USES)]
    lrs = [bf16r(torch.rand((2 * n, 3, h, w), generator=gen, device=dev)) for _ in range(N_USES)]
    wts = [randn((2 * n, 64, h, w), gen, dev) for _ in range(N_USES)]
    d_feat, d_lr, d_par = _run_resblocks(rbs, feats, lrs, wts)
    assert ops.debug_status() == 0

    # images [0, n) run block 0, [n, 2n) block 1
    P = [{k: v.detach().double().requires_grad_(True) for k, v in rb.state_dict().items()} for rb in rbs]
    xr = [torch.cat([l, f], 1).double().requires_grad_(True) for f, l in zip(feats, lrs)]
    loss = 0
    for x, wk in zip(xr, wts):
        y = torch.cat([O.residual_block(x[gi * n:(gi + 1) * n], P[gi], "") for gi in range(2)])
        loss = loss + (y * wk.double()).sum()
    loss.backward()
    Pd = [{k: v.detach() for k, v in p.items()} for p in P]
    em_par = [{k: torch.zeros_like(v) for k, v in p.items()} for p in Pd]
    em_dx = []
    for x, wk in zip(xr, wts):
        parts = []
        for gi in range(2):
            sl = slice(gi * n, (gi + 1) * n)
            dx, gr = _emulated_resblock(x.detach()[sl], Pd[gi], wk[sl].double())
            parts.append(dx)
            for k, v in gr.items():
                em_par[gi][k] += v
        em_dx.append(torch.cat(parts))
    worst = {}

    def check(got, want, ref, what):
        c, r = cos(got, want), rel(got, want)
        wc, wr = worst.get(ref, (1.0, 0.0))
        worst[ref] = (min(wc, c), max(wr, r))
        bound = (0.9999, 1e-2) if ref == "emulated" else (0.998, 8e-2)
        assert c >= bound[0] and r <= bound[1], (ref, what, c, r)

    for gi in range(2):
        for k, g in d_par[gi].items():
            check(g, em_par[gi][k], "emulated", f"block {gi} {k}")
            check(g, P[gi][k].grad, "oracle", f"block {gi} {k}")
    for i in range(N_USES):
        for ref, want in (("emulated", em_dx[i]), ("oracle", xr[i].grad)):
            check(d_feat[i][:, :64], want[:, 3:], ref, f"feat {i}")
            check(d_lr[i][:, :3], want[:, :3], ref, f"lr {i}")
        assert (d_lr[i][:, 3:] == 0).all()
    for ref, (c, r) in worst.items():
        print(f"resblock node vs {ref}: worst cos {c:.6f}, worst rel-L2 {r:.2e}")

    # group swap: the blocks in the other order and the two halves of every batch exchanged
    def swap(t):
        return torch.cat([t[n:], t[:n]])
    s_feat, s_lr, s_par = _run_resblocks(rbs[::-1], [swap(t) for t in feats], [swap(t) for t in lrs], [swap(t) for t in wts])
    for i in range(N_USES):
        assert torch.equal(s_feat[i], swap(d_feat[i])) and torch.equal(s_lr[i], swap(d_lr[i]))
    for gi in range(2):
        for k, g in d_par[gi].items():
            assert rel(s_par[1 - gi][k], g) <= 1e-5, (gi, k)          # only the order of the atomics differs
