"""Host side of the hot path: schedules the sm_100a kernels for the reference's
nn.Module forwards (Real-BasicVSR / BasicVSR / SPyNet / ResidualBlock / ...).

Everything here is orchestration: NHWC workspaces, packed-weight cache, which
kernel runs on what.  All arithmetic happens in libvsrb200.so.  Precision mode:

* ``fp32``  - fp32 activations, FFMA convolution; matches the reference's fp32
  path to <= 1e-4 max-abs.  Default outside autocast (reference test.py runs fp32).
* ``bf16``  - bf16 NHWC activations, tcgen05/TMEM implicit-GEMM convolution with fp32
  accumulate; flows, the cleaner's running frame and the output stay fp32.
  Default under ``torch.autocast`` (reference train.py:93), or force it with
  ``vsrlab_b200.set_precision("bf16")`` / ``VSRLAB_B200_PRECISION=bf16``.
"""
from __future__ import annotations

import contextlib
import os
import weakref
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import ops
from ._lib import (ACT_LRELU, ACT_NONE, ACT_RELU, BF16, BF16X2, EPI_CLEAN, EPI_FLOW, EPI_NHWC, EPI_SR, F32, INTERP_BICUBIC,
                   INTERP_BILINEAR, INTERP_NEAREST, PAD_BORDER, PAD_REFLECTION, PAD_ZEROS, VsrbError)

_forced: Optional[int] = None
# "fp32" = fp32-accurate mode.  Default implementation: split-bf16 (x = hi + lo) on the tensor cores, three MMA passes
# per product (hi*hi + lo*hi + hi*lo), fp32 accumulate; VSRB_FP32_IMPL=ffma selects the plain FFMA kernel instead.
_FP32 = F32 if os.environ.get("VSRB_FP32_IMPL", "x3") == "ffma" else BF16X2
_NAMES = {"bf16": BF16, "fp32": _FP32, "f32": _FP32, "fp32_ffma": F32, "fp32_x3": BF16X2}

# tunables: frames / images per launch batch.  Measured on B200 (gpurun_out bench4*): the ~8 us fixed cost per
# launch outweighs L2 residency, so batches are large; the tail is capped by the HR buffers (118 MB per frame).
CLEAN_CHUNK = int(os.environ.get("VSRB_CLEAN_CHUNK", "60"))
TAIL_CHUNK = int(os.environ.get("VSRB_TAIL_CHUNK", "15"))
# the image stems (3 -> 64, 64+3 -> 64) read the frame as 3x3 im2col patches (K = 32 on the ring-walk kernel); 0 = nine K = 16 chunks
STEM_PATCHES = os.environ.get("VSRB_STEM_PATCHES", "1") == "1"


# Opt-in narrow `sr` output (default None = fp32, the reference's dtype).  "fp16" halves and "uint8" quarters the bytes a
# caller moves to the host; "uint8" holds exactly what the reference's PNG dump stores (test.py:138-141 ->
# torchvision save_image: mul(255).add(0.5).clamp(0,255).to(uint8)), computed from the fp32 result inside the last conv.
_OUT_DTYPES = {None: (torch.float32, 0), "fp32": (torch.float32, 0), "fp16": (torch.float16, 4), "uint8": (torch.uint8, 2)}
_out_dtype: Optional[str] = None


def set_output_dtype(kind: Optional[str]) -> None:
    """None / 'fp32' (default), 'fp16' or 'uint8' for the `sr` tensor of the no_grad forward."""
    global _out_dtype
    if kind not in _OUT_DTYPES:
        raise ValueError(f"output dtype {kind!r}: choose from None, 'fp32', 'fp16', 'uint8'")
    _out_dtype = None if kind == "fp32" else kind


@contextlib.contextmanager
def output_dtype(kind: Optional[str]):
    old = _out_dtype
    set_output_dtype(kind)
    try:
        yield
    finally:
        set_output_dtype(old)


def set_precision(mode: Optional[str]) -> None:
    """Force 'bf16' / 'fp32', or None to follow autocast."""
    global _forced
    _forced = None if mode is None else _NAMES[mode]


@contextlib.contextmanager
def precision(mode: str):
    global _forced
    old = _forced
    _forced = _NAMES[mode]
    try:
        yield
    finally:
        _forced = old


def current_dtype() -> int:
    if _forced is not None:
        return _forced
    env = os.environ.get("VSRLAB_B200_PRECISION")
    if env:
        return _NAMES[env]
    return BF16 if torch.is_autocast_enabled() else _FP32


# --------------------------------------------------------------------------------------
# caches
# --------------------------------------------------------------------------------------
_packed: Dict[tuple, ops.PackedConv] = {}
_ws: Dict[tuple, torch.Tensor] = {}
_ws_private: List[Dict[tuple, torch.Tensor]] = []      # innermost private scratch set (owned by a CUDA-graph entry)
_consts: Dict[tuple, object] = {}


def _same_objects(refs, objs) -> bool:
    """id() values are recycled after garbage collection: a cache hit must be for the very same live modules."""
    return len(refs) == len(objs) and all(r() is o for r, o in zip(refs, objs))


# Set while graphs.py captures a TRAINING forward / backward: the weights change between replays, so the pack kernels
# must be recorded in the graph instead of being skipped by the cache below.  (The inference graphs are re-captured when a
# weight changes and keep using the cache.)
REPACK_IN_CAPTURE = False


def packed(convs: Sequence[torch.nn.Conv2d], segs: Sequence[Tuple[int, int]], dt: int, pixshuf: int = 0) -> ops.PackedConv:
    if REPACK_IN_CAPTURE and torch.cuda.is_current_stream_capturing():
        return ops.PackedConv(convs, segs, dt, pixshuf)
    key = (tuple(id(c) for c in convs), tuple(segs), dt, pixshuf)
    pc = _packed.get(key)
    if pc is None or pc.stamp != ops.PackedConv.stamp_of(convs) or not _same_objects(pc.owners, convs):
        pc = ops.PackedConv(convs, segs, dt, pixshuf)
        # the entry dies with its owners (per-call holders of derived weights - spectral norm - would pile up otherwise; a
        # recycled id whose new entry gets popped by a stale callback only costs one re-pack)
        pc.owners = [weakref.ref(c, lambda _r, k=key: _packed.pop(k, None)) for c in convs]
        _packed[key] = pc
    return pc


def ws(name: str, shape: Sequence[int], dtype: torch.dtype, device) -> torch.Tensor:
    """Named scratch tensor, grown on demand and reused across calls (never shrinks)."""
    n = 1
    for s in shape:
        n *= int(s)
    if _ws_private:
        # warm-up / capture of a CUDA graph: the scratch set belongs to that graph entry and dies with it
        table, key = _ws_private[-1], (name, dtype, str(device))
    else:
        # eager launches, per stream: two clips processed on two streams must not share scratch memory
        table, key = _ws, (name, dtype, str(device), torch.cuda.current_stream(device).cuda_stream)
    t = table.get(key)
    if t is None or t.numel() < n:
        t = torch.empty(max(n, 1), dtype=dtype, device=device)
        table[key] = t
    return t[:n].view(*shape)


@contextlib.contextmanager
def _private_workspaces(table: Dict[tuple, torch.Tensor]):
    _ws_private.append(table)
    try:
        yield table
    finally:
        _ws_private.pop()


def clear_caches() -> None:
    _packed.clear()
    _ws.clear()
    _consts.clear()
    _graphs.clear()


def _check_input(x: torch.Tensor, what: str) -> torch.Tensor:
    ops.require_cuda(x, what)
    if x.dtype != torch.float32:
        x = x.float()
    return x


def _wants_grad(mod, *tensors) -> bool:
    """True when the call must be recorded for autograd: grad mode on and something to differentiate - a trainable
    parameter of `mod` (a module, a sequence of modules, or None) or an input that requires grad.  Every module-level
    entry point checks this and routes to `autograd.py`; the raw kernels below never return a tensor that silently lost
    its graph (the reference modules are plain differentiable nn.Modules)."""
    if not torch.is_grad_enabled():
        return False
    if any(isinstance(t, torch.Tensor) and t.requires_grad for t in tensors):
        return True
    mods = [] if mod is None else (list(mod) if isinstance(mod, (list, tuple)) else [mod])
    return any(p.requires_grad for m in mods for p in m.parameters())


_warned_bf16_training = False


def _autograd():
    """The differentiable path (autograd.py).  It computes in bf16 with fp32 accumulation whatever the precision mode:
    warn once when the caller asked for fp32 (no autocast, `set_precision('fp32')`), instead of silently degrading."""
    global _warned_bf16_training
    if current_dtype() != BF16 and not _warned_bf16_training:
        import warnings
        _warned_bf16_training = True
        warnings.warn("vsrlab_b200: the differentiable (training) path runs bf16 activations with fp32 accumulation; "
                      "fp32 precision was requested (no autocast / set_precision('fp32')) and applies to no_grad calls only. "
                      "Wrap evaluation in torch.no_grad() for fp32-accurate outputs.", RuntimeWarning, stacklevel=3)
    from . import autograd as AG
    return AG


def _act_c(c: int, dt: int) -> int:
    """channels allocated per pixel for a c-channel activation"""
    if dt == BF16X2:
        return 2 * ((c + 15) // 16 * 16)       # [hi | lo]
    return (c + 15) // 16 * 16 if dt == BF16 else (c + 3) // 4 * 4


def _to_nhwc(x: torch.Tensor, dt: int, name: str, c_alloc: Optional[int] = None) -> Tuple[torch.Tensor, int]:
    n, c, h, w = x.shape
    ca = c_alloc or _act_c(c, dt)
    t = ws(name, (n, h, w, ca), ops.TORCH_DT[dt], x.device)
    ops.nchw_to_nhwc(x.contiguous(), t, n, c, h, w, ca, dt)
    return t, ca


def _to_nchw(t: torch.Tensor, n: int, c: int, h: int, w: int, c_src: int, dt: int) -> torch.Tensor:
    out = torch.empty(n, c, h, w, dtype=torch.float32, device=t.device)
    ops.nhwc_to_nchw(t, out, n, c, h, w, c_src, dt)
    return out


# --------------------------------------------------------------------------------------
# module-level entry points (NCHW fp32 in / out, like the reference modules)
# --------------------------------------------------------------------------------------
_ACTS = {"none": ACT_NONE, "relu": ACT_RELU, "lrelu": ACT_LRELU}


def conv2d(x: torch.Tensor, conv: torch.nn.Conv2d, act: str = "none", slope: float = 0.1, pixel_shuffle: int = 0) -> torch.Tensor:
    """act(conv(x)) [+ PixelShuffle]: ConvReLU (conv.py:21), PixelShufflePack (upsampling.py:10-12)."""
    x = _check_input(x, "input")
    if _wants_grad(conv, x):
        AG = _autograd()
        r = pixel_shuffle or 1
        y = AG.conv(conv, [AG.to_cl16(x)], [(0, x.shape[1])], act, slope, pixel_shuffle)
        return y[:, :conv.out_channels // (r * r)].float().contiguous()
    dt = current_dtype()
    n, c, h, w = x.shape
    xin, ca = _to_nhwc(x, dt, "m_in")
    pc = packed([conv], [(0, c)], dt, pixel_shuffle)
    r = pixel_shuffle or 1
    co = conv.out_channels // (r * r)
    oc = _act_c(co, dt) if (r > 1 or dt == BF16X2) else pc.cout_pad
    out = ws("m_out", (n, h * r, w * r, oc), ops.TORCH_DT[dt], x.device)
    ops.conv2d_fwd(pc, [xin], [ca], n, h, w, act=_ACTS[act], slope=slope, out=out, out_c=oc)
    return _to_nchw(out, n, co, h * r, w * r, oc, dt)


def conv_chain(x: torch.Tensor, convs: Sequence[torch.nn.Conv2d], act: str = "relu") -> torch.Tensor:
    """act(conv(...act(conv(x)))) - SpynetModule (spynet.py:13-21)."""
    x = _check_input(x, "input")
    if _wants_grad(list(convs), x):
        AG = _autograd()
        y = AG.to_cl16(x)
        for conv in convs:
            y = AG.conv(conv, [y], [(0, conv.in_channels)], act)
        return y[:, :convs[-1].out_channels].float().contiguous()
    dt = current_dtype()
    n, c, h, w = x.shape
    cur, ca = _to_nhwc(x, dt, "m_in")
    for j, conv in enumerate(convs):
        pc = packed([conv], [(0, conv.in_channels)], dt)
        oc = _act_c(conv.out_channels, dt) if dt == BF16X2 else pc.cout_pad
        out = ws(f"m_chain{j % 2}", (n, h, w, oc), ops.TORCH_DT[dt], x.device)
        ops.conv2d_fwd(pc, [cur], [ca], n, h, w, act=_ACTS[act], out=out, out_c=oc)
        cur, ca = out, oc
    return _to_nchw(cur, n, convs[-1].out_channels, h, w, ca, dt)


def _run_resblocks(cur, ca, stem_pc, block_pcs, n, h, w, mid_c, dt, device, tag, final_out=None, final_strides=(0, 0),
                   extra_in=None, extra_c=0, groups=1, stem_patch=None, stem_patch_strides=(0, 0)):
    """stem (+LeakyReLU) then residual blocks on NHWC buffers; returns (tensor, channels).
    If `final_out` is given the last conv of the chain writes there (raw address allowed)."""
    tdt = ops.TORCH_DT[dt]
    bufs = [ws(f"{tag}_r{i}", (n, h, w, mid_c), tdt, device) for i in range(3)]
    nconv = (1 if stem_pc is not None else 0) + 2 * len(block_pcs)
    done = 0

    def target(i):
        nonlocal done
        done += 1
        if done == nconv and final_out is not None:
            return final_out, final_strides
        return bufs[i], (0, 0)

    free = [0, 1, 2]
    if stem_pc is not None:
        o, st = target(free[0])
        ins, cs = ([cur, extra_in], [ca, extra_c]) if extra_in is not None else ([cur], [ca])
        ops.conv2d_fwd(stem_pc, ins, cs, n, h, w, act=ACT_LRELU, slope=0.1, out=o, out_c=mid_c,
                       out_img_stride=st[0], out_group_stride=st[1], patch=stem_patch, patch_img_stride=stem_patch_strides[0],
                       patch_group_stride=stem_patch_strides[1])
        cur, ca, cur_i = o, mid_c, free[0]
    else:
        cur_i = -1
    for (p1, p2) in block_pcs:
        avail = [i for i in (0, 1, 2) if i != cur_i]
        t1, _ = target(avail[0])
        ops.conv2d_fwd(p1, [cur], [ca], n, h, w, act=ACT_RELU, out=t1, out_c=mid_c)
        o, st = target(avail[1])
        ops.conv2d_fwd(p2, [t1], [mid_c], n, h, w, act=ACT_NONE, out=o, out_c=mid_c, residual=cur, res_c=ca,
                       out_img_stride=st[0], out_group_stride=st[1])
        cur, ca, cur_i = o, mid_c, avail[1]
    return cur, ca


def residual_stack(x: torch.Tensor, stem: Optional[torch.nn.Conv2d], blocks: Sequence[torch.nn.Module]) -> torch.Tensor:
    """ResidualBlock / ResidualConv forward (conv.py:89-92, 101-103)."""
    x = _check_input(x, "input")
    mid = stem.out_channels if stem is not None else blocks[0].conv1.out_channels
    if _wants_grad(([stem] if stem is not None else []) + [cv for b in blocks for cv in (b.conv1, b.conv2)], x):
        AG = _autograd()
        y = AG.to_cl16(x)
        if stem is not None:
            y = AG.conv(stem, [y], [(0, x.shape[1])], "lrelu")
        for b in blocks:
            t = AG.conv(b.conv1, [y], [(0, mid)], "relu")
            y = AG.conv(b.conv2, [t], [(0, mid)], "none", residual=y)
        return y[:, :mid].float().contiguous()
    dt = current_dtype()
    n, c, h, w = x.shape
    mid_c = _act_c(mid, dt)
    cur, ca = _to_nhwc(x, dt, "m_in", None if stem is not None else mid_c)
    stem_pc = packed([stem], [(0, c)], dt) if stem is not None else None
    bpcs = [(packed([b.conv1], [(0, mid)], dt), packed([b.conv2], [(0, mid)], dt)) for b in blocks]
    cur, ca = _run_resblocks(cur, ca, stem_pc, bpcs, n, h, w, mid_c, dt, x.device, "m")
    return _to_nchw(cur, n, mid, h, w, ca, dt)


def spectral_conv2d(x: torch.Tensor, sc) -> torch.Tensor:
    """SpectralConv.forward (conv.py:6-13): conv with the spectrally normalised weight, no bias, no activation."""
    x = _check_input(x, "input")
    AG = _autograd() if _wants_grad(sc, x) else None
    from . import autograd as A
    with (contextlib.nullcontext() if AG is not None else torch.no_grad()):
        y = A.spectral_conv(sc, A.to_cl16(x), "none", 0.0)
    return y[:, :sc.conv.out_channels].float().contiguous()


def unet_discriminator_forward(D, img: torch.Tensor) -> torch.Tensor:
    """UNetDiscriminator.forward (unet-discriminator.py:19-31) on the conv kernels; bf16 activations, fp32 logits."""
    img = _check_input(img, "img")
    if img.shape[-2] % 8 or img.shape[-1] % 8:
        raise VsrbError("UNetDiscriminator needs sides that are multiples of 8 (three stride-2 encoders)")
    from . import autograd as A
    if _wants_grad(D, img):
        _autograd()
        return A.unet_discriminator(D, img)
    with torch.no_grad():
        return A.unet_discriminator(D, img)


_WARP_PADS = {"zeros": PAD_ZEROS, "border": PAD_BORDER, "reflection": PAD_REFLECTION}
_WARP_INTERPS = {"bilinear": INTERP_BILINEAR, "nearest": INTERP_NEAREST, "bicubic": INTERP_BICUBIC}


def flow_warp(x: torch.Tensor, flow: torch.Tensor, padding_mode: str = "zeros", interpolation: str = "bilinear",
              align_corners: bool = True) -> torch.Tensor:
    """flow_warp(x [T,c,h,w], flow [T,h,w,2]) (spynet.py:95-106) with any mode F.grid_sample accepts.  The propagation
    warp's mode (bilinear, zeros / border, align_corners) runs the propagation kernel; the others run flow_warp_ex (fp32
    NHWC in fp32 mode, bf16 in bf16 mode)."""
    if padding_mode not in _WARP_PADS:
        raise ValueError(f"flow_warp: padding_mode must be 'zeros', 'border' or 'reflection', got {padding_mode!r}")
    if interpolation not in _WARP_INTERPS:
        raise ValueError(f"flow_warp: interpolation must be 'bilinear', 'nearest' or 'bicubic', got {interpolation!r}")
    align_corners = bool(align_corners)
    if interpolation != "bilinear" or padding_mode == "reflection" or not align_corners:
        return _flow_warp_ex(x, flow, _WARP_INTERPS[interpolation], _WARP_PADS[padding_mode], align_corners)
    x = _check_input(x, "input")
    flow = _check_input(flow, "flow").contiguous()
    n, c, h, w = x.shape
    if _wants_grad(None, x, flow):
        # differentiable in the features and in the flow (fp32 data: a loss may sit right on top of it)
        AG = _autograd()
        nv = 1
        while nv * 4 < c:
            nv *= 2
        xp = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, nv * 4 - c)).contiguous(memory_format=torch.channels_last)
        return AG.WarpFn.apply(xp, flow, padding_mode == "border")[:, :c].contiguous()
    dt = current_dtype()
    if dt == BF16X2:
        ca = _act_c(c, dt)
    else:
        vec = 8 if dt == BF16 else 4
        nv = 1
        while nv * vec < c:                # the kernel splits a pixel over a power-of-two number of 16-byte vectors
            nv *= 2
        ca = nv * vec
    xin, _ = _to_nhwc(x, dt, "m_in", ca)
    out = ws("m_out", (n, h, w, ca), ops.TORCH_DT[dt], x.device)
    ops.flow_warp(xin, flow, out, n, h, w, ca, dt, PAD_BORDER if padding_mode == "border" else PAD_ZEROS)
    return _to_nchw(out, n, c, h, w, ca, dt)


def _flow_warp_ex(x: torch.Tensor, flow: torch.Tensor, interp: int, pad: int, align_corners: bool) -> torch.Tensor:
    x = _check_input(x, "input")
    flow = _check_input(flow, "flow").contiguous()
    n, c, h, w = x.shape
    nv = 1
    if _wants_grad(None, x, flow):
        AG = _autograd()
        while nv * 4 < c:
            nv *= 2
        xp = torch.nn.functional.pad(x, (0, 0, 0, 0, 0, nv * 4 - c)).contiguous(memory_format=torch.channels_last)
        return AG.WarpExFn.apply(xp, flow, interp, pad, align_corners)[:, :c].contiguous()
    # fp32 mode (split-bf16 or FFMA) runs the fp32 NHWC kernel: a memory-bound gather that moves as many bytes as the
    # split-bf16 [hi | lo] layout would, and is exact
    dt = BF16 if current_dtype() == BF16 else F32
    vec = 8 if dt == BF16 else 4
    while nv * vec < c:                    # a power-of-two number of 16-byte vectors per pixel
        nv *= 2
    ca = nv * vec
    xin, _ = _to_nhwc(x, dt, "m_in", ca)
    out = ws("m_out", (n, h, w, ca), ops.TORCH_DT[dt], x.device)
    ops.flow_warp_ex(xin, flow, out, n, h, w, ca, dt, interp, pad, align_corners)
    return _to_nchw(out, n, c, h, w, ca, dt)


# --------------------------------------------------------------------------------------
# SPyNet
# --------------------------------------------------------------------------------------
def _spynet_consts(sp) -> Tuple[List[float], List[float]]:
    key = ("spynet_norm", id(sp), sp.mean.data_ptr(), sp.mean._version, sp.std._version)
    v = _consts.get(key)
    if v is None or v[2]() is not sp:
        v = (sp.mean.detach().flatten().cpu().tolist(), sp.std.detach().flatten().cpu().tolist(), weakref.ref(sp))
        _consts[key] = v
    return v[0], v[1]


def _spynet_run(sp, frames: torch.Tensor, ref_idx: torch.Tensor, supp_idx: torch.Tensor, dt: int, resize: bool = True) -> torch.Tensor:
    """frames [F,3,h,w] fp32 contiguous; pair p = (frames[ref_idx[p]], frames[supp_idx[p]]).
    Returns flows [P,h,w,2] fp32 (channels-last, the layout flow_warp consumes)."""
    F_, _, h, w = frames.shape
    dev = frames.device
    ops.TAG = "spynet"
    if resize:
        Hp, Wp = (h + 31) // 32 * 32, (w + 31) // 32 * 32
    else:
        if h % 32 or w % 32:
            raise VsrbError("Spynet.compute_flow needs sides that are multiples of 32 (reference spynet.py:49)")
        Hp, Wp = h, w
    mean, std = _spynet_consts(sp)
    tdt = ops.TORCH_DT[dt]
    lv = [ws(f"sp_pyr{k}", (F_, Hp >> k, Wp >> k, 4), torch.float32, dev) for k in range(6)]
    ops.spynet_pyramid_base(frames, lv[0], F_, h, w, Hp, Wp, mean, std)
    for k in range(1, 6):
        ops.avgpool2_c4(lv[k - 1], lv[k], F_, Hp >> (k - 1), Wp >> (k - 1))
    P = ref_idx.numel()
    cin0 = {BF16: 16, F32: 8, BF16X2: 32}[dt]
    chans = [cin0, _act_c(32, dt), _act_c(64, dt), _act_c(32, dt), _act_c(16, dt)]
    full = [ws(f"sp_act{j}", (P, Hp, Wp, chans[j]), tdt, dev) for j in range(5)]
    fup_full = ws("sp_fup", (P, Hp, Wp, 2), torch.float32, dev)
    fl_full = [ws(f"sp_flow{j}", (P, Hp, Wp, 2), torch.float32, dev) for j in range(2)]
    flow_prev = None
    for level in range(6):
        k = 5 - level
        Hl, Wl = Hp >> k, Wp >> k
        npx = P * Hl * Wl
        act = [full[j].view(-1)[: npx * chans[j]].view(P, Hl, Wl, chans[j]) for j in range(5)]
        fup = fup_full.view(-1)[: npx * 2].view(P, Hl, Wl, 2)
        fl = fl_full[level % 2].view(-1)[: npx * 2].view(P, Hl, Wl, 2)
        ops.spynet_level_input(lv[k], ref_idx, supp_idx, flow_prev, fup, act[0], P, Hl, Wl, cin0, dt)
        mods = sp.basic_module[level].basic_module
        for j in range(5):
            conv = mods[j].conv[0]
            pc = packed([conv], [(0, conv.in_channels)], dt)
            if j < 4:
                ops.conv2d_fwd(pc, [act[j]], [chans[j]], P, Hl, Wl, act=ACT_RELU, out=act[j + 1], out_c=chans[j + 1])
            else:   # flow = flow_up + relu(conv) fused in the epilogue (spynet.py:65)
                ops.conv2d_fwd(pc, [act[j]], [chans[j]], P, Hl, Wl, act=ACT_RELU, epilogue=EPI_FLOW, f32_in=fup, f32_io=fl)
        flow_prev = fl
    if (Hp, Wp) == (h, w):
        return flow_prev.clone()
    out = torch.empty(P, h, w, 2, dtype=torch.float32, device=dev)
    ops.flow_resize(flow_prev, out, P, Hp, Wp, h, w)
    return out


def spynet_flow(sp, ref: torch.Tensor, supp: torch.Tensor, resize: bool = True) -> torch.Tensor:
    """Spynet.forward / compute_flow: [T,3,h,w] x2 -> [T,2,h,w] (spynet.py:38-93)."""
    ref = _check_input(ref, "ref")
    supp = _check_input(supp, "supp")
    if _wants_grad(sp, ref, supp):
        if not resize and (ref.shape[-2] % 32 or ref.shape[-1] % 32):
            raise VsrbError("Spynet.compute_flow needs sides that are multiples of 32 (reference spynet.py:49)")
        return _autograd().spynet(sp, ref, supp)
    t = ref.shape[0]
    frames = torch.cat([ref, supp], 0).contiguous()
    idx = torch.arange(2 * t, dtype=torch.int32, device=ref.device)
    flows = _spynet_run(sp, frames, idx[:t].contiguous(), idx[t:].contiguous(), current_dtype(), resize)
    return flows.permute(0, 3, 1, 2).contiguous()


def _pair_indices(n: int, t: int, device) -> Tuple[torch.Tensor, torch.Tensor]:
    """First n*(t-1) pairs: backward flows (ref=frame i, supp=i+1); then forward (ref=i+1, supp=i).
    Reference basicvsr.py:30-37."""
    key = ("pairs", n, t, str(device))
    v = _consts.get(key)
    if v is None:
        base = (torch.arange(n, dtype=torch.int32).view(n, 1) * t + torch.arange(t - 1, dtype=torch.int32).view(1, t - 1)).reshape(-1)
        ref = torch.cat([base, base + 1]).to(device)
        supp = torch.cat([base + 1, base]).to(device)
        v = (ref.contiguous(), supp.contiguous())
        _consts[key] = v
    return v


def basicvsr_flows(bv, lrs: torch.Tensor):
    """BasicVSR.compute_flow: (flow_forward, flow_backward), each [n*(t-1),2,h,w] (basicvsr.py:30-37)."""
    lrs = _check_input(lrs, "lrs")
    n, t, c, h, w = lrs.shape
    if _wants_grad(bv.spynet, lrs):
        a, b = lrs[:, :-1].reshape(-1, c, h, w), lrs[:, 1:].reshape(-1, c, h, w)
        AG = _autograd()
        return AG.spynet(bv.spynet, b, a), AG.spynet(bv.spynet, a, b)        # (forward, backward): basicvsr.py:35-37
    ref, supp = _pair_indices(n, t, lrs.device)
    flows = _spynet_run(bv.spynet, lrs.contiguous().view(n * t, c, h, w), ref, supp, current_dtype())
    m = n * (t - 1)
    fb = flows[:m].permute(0, 3, 1, 2).contiguous()
    ff = flows[m:].permute(0, 3, 1, 2).contiguous()
    return ff, fb


# --------------------------------------------------------------------------------------
# cleaner / BasicVSR / Real-BasicVSR
# --------------------------------------------------------------------------------------
def _cleaner_run(cl, x: torch.Tensor, dt: int) -> torch.Tensor:
    """x [B,3,h,w] fp32 contiguous, refined in place (realbasicvsr.py:24-30).
    Returns the NHWC copy of the refined frames (input of the propagation stems)."""
    B, c, h, w = x.shape
    dev = x.device
    ops.TAG = "cleaner"
    tdt = ops.TORCH_DT[dt]
    mid = cl.resblock.conv[0].out_channels
    mid_c = _act_c(mid, dt)
    clr = _act_c(3, dt)
    x_nhwc = ws("x_nhwc", (B, h, w, clr), tdt, dev)
    ops.nchw_to_nhwc(x, x_nhwc, B, c, h, w, clr, dt)
    stem = packed([cl.resblock.conv[0]], [(0, 3)], dt)
    blocks = [(packed([b.conv1], [(0, mid)], dt), packed([b.conv2], [(0, mid)], dt)) for b in cl.resblock.res_block]
    last = packed([cl.conv], [(0, mid)], dt)
    chunk = max(1, min(B, CLEAN_CHUNK))
    # bf16 mode: the 3 -> 64 stem reads the frame as 3x3 im2col patches (one K = 32 chunk on the ring-walk kernel)
    patches = ws("cl_patch", (chunk, h, w, 32), torch.bfloat16, dev) if (dt == BF16 and mid == 64 and STEM_PATCHES) else None
    for _ in range(cl.steps):
        for b0 in range(0, B, chunk):
            nb = min(chunk, B - b0)
            if patches is not None:
                ops.im2col3x3(x[b0:b0 + nb], patches, nb, h, w)
            cur, ca = _run_resblocks(x_nhwc[b0:b0 + nb], clr, stem, blocks, nb, h, w, mid_c, dt, dev, "cl", stem_patch=patches)
            ops.conv2d_fwd(last, [cur], [ca], nb, h, w, act=ACT_NONE, epilogue=EPI_CLEAN, out=x_nhwc[b0:b0 + nb], out_c=clr,
                           f32_io=x[b0:b0 + nb])
    return x_nhwc


def cleaner_forward(cl, x: torch.Tensor) -> torch.Tensor:
    x = _check_input(x, "input")
    if not x.is_contiguous():
        raise RuntimeError("IterativeRefinement works in place on a view of its input; pass a contiguous tensor")
    n, t, c, h, w = x.shape
    if _wants_grad(cl, x):
        AG = _autograd()
        with AG.batched_wgrad():
            y = AG.cleaner(cl, x.reshape(n * t, c, h, w)).view(n, t, c, h, w)
        if not x.requires_grad:                  # what the reference's in-place refinement leaves in the caller's tensor
            with torch.no_grad():
                x.copy_(y)
        return y
    _cleaner_run(cl, x.view(n * t, c, h, w), current_dtype())
    return x


def _basicvsr_run(bv, lrs: torch.Tensor, dt: int, x_nhwc: Optional[torch.Tensor] = None) -> torch.Tensor:
    """lrs [n,t,3,h,w] fp32 contiguous -> sr [n,t,3,s*h,s*w] fp32 (basicvsr.py:39-83)."""
    n, t, c, h, w = lrs.shape
    dev = lrs.device
    tdt = ops.TORCH_DT[dt]
    es = ops.ESIZE[dt]
    mid = bv.mid_channels
    mid_c = _act_c(mid, dt)
    clr = _act_c(3, dt)
    x_flat = lrs.view(n * t, c, h, w)
    if x_nhwc is None:
        x_nhwc = ws("x_nhwc", (n * t, h, w, clr), tdt, dev)
        ops.nchw_to_nhwc(x_flat, x_nhwc, n * t, c, h, w, clr, dt)

    # ---- optical flow, both directions in one batch (basicvsr.py:30-37) -----------------
    flows = None
    if t > 1:
        ref, supp = _pair_indices(n, t, dev)
        flows = _spynet_run(bv.spynet, x_flat, ref, supp, dt)          # [2*n*(t-1), h, w, 2]
        m = n * (t - 1)
        flows_b, flows_f = flows[:m], flows[m:]

    # ---- bidirectional propagation: both directions run as two weight groups ------------
    ops.TAG = "propagation"
    pairs = ws("lr_pairs", (t, 2 * n, h, w, clr), tdt, dev)
    key = ("pair_gather", n, t, str(dev))
    if key not in _consts:                                             # step s: [frame t-1-s | frame s] of every clip
        _consts[key] = torch.tensor([i * t + (t - 1 - s if g == 0 else s) for s in range(t) for g in range(2) for i in range(n)],
                                    device=dev)
    torch.index_select(x_nhwc.view(n * t, h * w * clr), 0, _consts[key], out=pairs.view(t * 2 * n, h * w * clr))
    bank = ws("feat_bank", (2, n, t, h, w, mid_c), tdt, dev)           # [0]=backward, [1]=forward features
    fbk, ffw = bank[0], bank[1]
    frame_el = h * w * mid_c
    bwd, fwd = bv.backward_resblocks, bv.forward_resblocks
    stem = packed([bwd.conv[0], fwd.conv[0]], [(3, mid), (0, 3)], dt)   # cat([lr_i, feat]) order kept via seg_off
    blocks = [(packed([a.conv1, b.conv1], [(0, mid)], dt), packed([a.conv2, b.conv2], [(0, mid)], dt))
              for a, b in zip(bwd.res_block, fwd.res_block)]
    warped = ws("feat_warp", (2 * n, h, w, mid_c), tdt, dev)
    # bf16 mode: the 3-channel half of cat([lr_i, feat]) enters the stem as 3x3 im2col patches of the frame, built once per clip
    lr_patch = None
    if dt == BF16 and mid == 64 and STEM_PATCHES:
        lr_patch = ws("lr_patch", (n * t, h, w, 32), torch.bfloat16, dev)
        ops.im2col3x3(x_flat, lr_patch, n * t, h, w)
    pf = h * w * 32                                                      # elements of one frame of patches
    for s in range(t):
        if s == 0:
            warped.zero_()
        elif dt == BF16:
            # both directions in one launch: backward chain = bank frame t-s warped by flows_b[t-1-s], forward chain = bank
            # frame s-1 warped by flows_f[s-1] (basicvsr.py:52-54, 66-69)
            xb, xf = fbk.data_ptr() + (t - s) * frame_el * es, ffw.data_ptr() + (s - 1) * frame_el * es
            wb, wf = flows_b.data_ptr() + (t - 1 - s) * h * w * 8, flows_f.data_ptr() + (s - 1) * h * w * 8
            ops.flow_warp_groups(xb, (t * frame_el, (xf - xb) // es), wb, ((t - 1) * h * w, (wf - wb) // 8), warped, n, 2, h, w, mid_c, dt,
                                 PAD_ZEROS)
        else:
            ops.flow_warp(fbk.data_ptr() + (t - s) * frame_el * es, flows_b.data_ptr() + (t - 1 - s) * h * w * 8, warped[:n],
                          n, h, w, mid_c, dt, PAD_ZEROS, x_img_stride=t * frame_el, flow_img_stride=(t - 1) * h * w)
            ops.flow_warp(ffw.data_ptr() + (s - 1) * frame_el * es, flows_f.data_ptr() + (s - 1) * h * w * 8, warped[n:],
                          n, h, w, mid_c, dt, PAD_ZEROS, x_img_stride=t * frame_el, flow_img_stride=(t - 1) * h * w)
        o_b = fbk.data_ptr() + (t - 1 - s) * frame_el * es
        o_f = ffw.data_ptr() + s * frame_el * es
        # group 0 (backward chain) reads frame t-1-s of every clip, group 1 (forward chain) frame s
        _run_resblocks(warped, mid_c, stem, blocks, 2 * n, h, w, mid_c, dt, dev, "pp", final_out=o_b,
                       final_strides=(t * frame_el, (o_f - o_b) // es), extra_in=pairs[s], extra_c=clr, groups=2,
                       stem_patch=None if lr_patch is None else lr_patch.data_ptr() + (t - 1 - s) * pf * 2,
                       stem_patch_strides=(t * pf, (2 * s - (t - 1)) * pf))

    # ---- fusion + upsampling + reconstruction, batched over frames (basicvsr.py:75-83) --
    ops.TAG = "tail"
    n_up = len(bv.upsample)
    scale = 2 ** n_up
    H, W = h * scale, w * scale
    sr_dtype, sr_flag = _OUT_DTYPES[_out_dtype]
    sr = torch.empty(n, t, 3, H, W, dtype=sr_dtype, device=dev)
    sr_flat = sr.view(n * t, 3, H, W)
    point = packed([bv.point_conv[0]], [(0, mid), (mid, mid)], dt)
    ups = [packed([u.upconv], [(0, mid)], dt, 2) for u in bv.upsample]
    cl0 = packed([bv.conv_last[0]], [(0, mid)], dt)
    cl2 = packed([bv.conv_last[2]], [(0, bv.conv_last[2].in_channels)], dt)
    c_last = _act_c(bv.conv_last[0].out_channels, dt)
    fb_flat, ff_flat = fbk.view(n * t, h, w, mid_c), ffw.view(n * t, h, w, mid_c)
    B = n * t
    chunk = max(1, min(B, TAIL_CHUNK))
    for b0 in range(0, B, chunk):
        nb = min(chunk, B - b0)
        cur = ws("tl_p", (nb, h, w, mid_c), tdt, dev)
        ops.conv2d_fwd(point, [fb_flat[b0:b0 + nb], ff_flat[b0:b0 + nb]], [mid_c, mid_c], nb, h, w, act=ACT_LRELU, slope=0.1,
                       out=cur, out_c=mid_c)
        hh, ww = h, w
        for i, up in enumerate(ups):
            nxt = ws(f"tl_u{i}", (nb, 2 * hh, 2 * ww, mid_c), tdt, dev)
            ops.conv2d_fwd(up, [cur], [mid_c], nb, hh, ww, act=ACT_NONE, out=nxt, out_c=mid_c)
            cur, hh, ww = nxt, 2 * hh, 2 * ww
        hr = ws("tl_h", (nb, H, W, c_last), tdt, dev)
        ops.conv2d_fwd(cl0, [cur], [mid_c], nb, H, W, act=ACT_LRELU, slope=0.1, out=hr, out_c=c_last)
        ops.conv2d_fwd(cl2, [hr], [c_last], nb, H, W, act=ACT_NONE, epilogue=EPI_SR, f32_io=sr_flat[b0:b0 + nb],
                       f32_in=x_flat[b0:b0 + nb], aux_hw=(h, w), extra_flags=sr_flag)
    return sr


def basicvsr_forward(bv, lrs: torch.Tensor) -> torch.Tensor:
    if _wants_grad(bv, lrs):
        AG = _autograd()
        ops.require_cuda(lrs, "lrs")
        with AG.batched_wgrad():
            return AG.basicvsr(bv, lrs.float())
    lrs = _check_input(lrs, "lrs").contiguous()
    return _basicvsr_run(bv, lrs, current_dtype())


def realbasicvsr_forward(model, lr: torch.Tensor):
    """(sr, lq) = RealBasicVSR.forward; `lq` is `lr` itself, refined in place (realbasicvsr.py:11-15, 26-29)."""
    ops.require_cuda(lr, "lr")
    if _wants_grad(model, lr):
        _autograd()
        from . import graphs
        return graphs.training_forward(model, lr)
    if lr.dtype != torch.float32:
        raise VsrbError("RealBasicVSR refines its input in place and needs an fp32 tensor (reference realbasicvsr.py:29)")
    if not lr.is_contiguous():
        raise RuntimeError("RealBasicVSR works in place on a view of its input; pass a contiguous tensor")
    dt = current_dtype()
    if GRAPHS and ops.PROFILE is None:
        return _graphed_forward(model, lr, dt)
    n, t, c, h, w = lr.shape
    x_nhwc = _cleaner_run(model.cleaner, lr.view(n * t, c, h, w), dt)
    sr = _basicvsr_run(model.basicvsr, lr, dt, x_nhwc)
    return sr, lr


# --------------------------------------------------------------------------------------
# CUDA-graph replay of the whole forward (several hundred dependent launches per call)
# --------------------------------------------------------------------------------------
GRAPHS = os.environ.get("VSRB_GRAPHS", "1") == "1"      # VSRB_GRAPHS=0: launch every kernel eagerly
MAX_GRAPHS = 4                                          # captured (model, shape, precision, stream) combinations kept alive
# Opt-in: return the graph's static `sr` buffer itself instead of a copy (saves a 663 MB device copy per cfg3 step).
# The tensor is then only valid until the next call with the same model / shape / stream.
GRAPH_OUTPUT_VIEW = os.environ.get("VSRB_GRAPH_OUTPUT_VIEW", "0") == "1"
_graphs: Dict[tuple, "_GraphEntry"] = {}
_capture_streams: Dict[str, torch.cuda.Stream] = {}     # one long-lived capture stream per device
# kernels of libvsrb200.so launched through graph replays (vsrb_launch_count only sees direct launches; a replay
# launches every kernel node recorded at capture time)
_replayed_launches = 0


def replayed_launches() -> int:
    return _replayed_launches


def _weights_stamp(model) -> tuple:
    return tuple((p.data_ptr(), p._version) for p in model.parameters())


class _GraphEntry:
    """One captured forward.  It owns everything the graph's kernels touch: the static input / output and the private
    scratch set (`workspaces`), so dropping the entry (eviction, re-capture after a weight update) frees them, and no
    other capture or eager call can grow / free a buffer whose address is baked into this graph."""
    __slots__ = ("stamp", "graph", "static_in", "static_sr", "model", "n_kernels", "workspaces")


def _capture_stream(device) -> torch.cuda.Stream:
    st = _capture_streams.get(str(device))
    if st is None:
        st = _capture_streams[str(device)] = torch.cuda.Stream(device=device)
    return st


def _evict_graphs(keep_free_fraction: float = 0.25, device=None) -> None:
    """Oldest-first eviction: at most MAX_GRAPHS captures, and none of the old ones once the device runs short of memory
    (a capture of cfg3 pins several GB of workspaces; test.py's ragged last window is a second shape per video)."""
    while len(_graphs) >= MAX_GRAPHS:
        _graphs.pop(next(iter(_graphs)))
    if device is not None and _graphs:
        free, total = torch.cuda.mem_get_info(device)
        if free < keep_free_fraction * total:
            _graphs.clear()
            torch.cuda.empty_cache()


def _graphed_forward(model, lr: torch.Tensor, dt: int):
    """Capture `cleaner + BasicVSR` once per (model weights, shape, precision, calling stream) and replay it.  The captured
    graph works on a private input buffer; the caller's `lr` receives the cleaned frames afterwards, so the in-place
    contract (`lq is lr`, overwritten) is unchanged, and `sr` is copied out of the graph's static output.  The calling
    stream is part of the key: two streams (or threads) running same-shaped clips get a capture each, so they never share
    the static buffers; within one stream, replays and the copies around them are stream-ordered."""
    cur = torch.cuda.current_stream(lr.device)
    key = (id(model), dt, tuple(lr.shape), str(lr.device), _out_dtype, cur.cuda_stream)
    stamp = _weights_stamp(model)
    entry = _graphs.get(key)
    if entry is None or entry.stamp != stamp or entry.model() is not model:
        _graphs.pop(key, None)                     # a stale capture releases its buffers before the new one allocates
        entry = None
        _evict_graphs(device=lr.device)
        n, t, c, h, w = lr.shape
        entry = _GraphEntry()
        entry.stamp, entry.model, entry.workspaces = stamp, weakref.ref(model), {}
        entry.static_in = torch.empty_like(lr)
        side = _capture_stream(lr.device)
        side.wait_stream(cur)
        with _private_workspaces(entry.workspaces):
            with torch.cuda.stream(side):          # warm-up on the capture stream: packs weights, sizes the workspaces
                entry.static_in.copy_(lr)
                x_nhwc = _cleaner_run(model.cleaner, entry.static_in.view(n * t, c, h, w), dt)
                _basicvsr_run(model.basicvsr, entry.static_in, dt, x_nhwc)
            cur.wait_stream(side)
            torch.cuda.synchronize(lr.device)
            entry.graph = torch.cuda.CUDAGraph()
            k0 = ops.launch_count()
            with torch.cuda.graph(entry.graph, stream=side):
                x_nhwc = _cleaner_run(model.cleaner, entry.static_in.view(n * t, c, h, w), dt)
                entry.static_sr = _basicvsr_run(model.basicvsr, entry.static_in, dt, x_nhwc)
            entry.n_kernels = ops.launch_count() - k0
        _graphs[key] = entry
    global _replayed_launches
    entry.static_in.copy_(lr)
    entry.graph.replay()
    _replayed_launches += entry.n_kernels
    lr.copy_(entry.static_in)
    return (entry.static_sr if GRAPH_OUTPUT_VIEW else entry.static_sr.clone()), lr
