"""Tensor-level wrappers around the C-ABI: they only turn torch tensors into raw
device pointers + sizes and enqueue on torch's current CUDA stream.  torch is
used for device memory and streams, nothing else."""
from __future__ import annotations

import ctypes as C
import os
import warnings
from typing import Optional, Sequence, Tuple

import torch

from . import _lib as L
from ._lib import (ACT_LRELU, ACT_NONE, ACT_RELU, BF16, BF16X2, EPI_CLEAN, EPI_FLOW, EPI_NHWC, EPI_SR, F32, INTERP_BILINEAR,
                   PAD_BORDER, PAD_ZEROS)

# BF16X2 = split-bf16 (fp32-accurate tensor-core mode): per pixel [hi C | lo C] bf16, value = hi + lo
TORCH_DT = {BF16: torch.bfloat16, F32: torch.float32, BF16X2: torch.bfloat16}
ESIZE = {BF16: 2, F32: 4, BF16X2: 2}


# bench.py sets this to a list to time every launch with CUDA events on the launching stream:
# entries are (kind, start_event, end_event, algorithmic work: FLOPs for convs, bytes otherwise)
PROFILE = None
PROFILE_SHAPES = os.environ.get("VSRB_PROFILE_SHAPES") == "1"
# Programmatic dependent launch between consecutive convs: the next conv's grid is scheduled while the current one drains
# (its producer and epilogue roles wait on griddepcontrol.wait before touching activations).  +2 % at cfg3 inside the
# replayed graph (CUPTI shows ~6 us between kernels otherwise); VSRB_PDL=0 turns it off.
PDL = os.environ.get("VSRB_PDL", "1") == "1"
TAG = ""          # set by the scheduler so profile entries can be grouped by network part


class _Timed:
    def __init__(self, kind: str, work: float):
        self.kind, self.work = kind, work

    def __enter__(self):
        if PROFILE is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if PROFILE is not None:
            self.e1.record()
            PROFILE.append((self.kind, self.e0, self.e1, self.work, TAG))
        return False


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def _stream() -> C.c_void_p:
    # the raw handle of torch's current stream; the private accessor skips ~3 us of Stream-object construction per launch
    if _raw_stream is not None:
        return C.c_void_p(_raw_stream(torch.cuda.current_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t) -> Optional[C.c_void_p]:
    if t is None:
        return None
    if isinstance(t, int):
        return C.c_void_p(t)
    return C.c_void_p(t.data_ptr())


# torch.use_deterministic_algorithms(True), read at call time: the weight / bias gradients, the warp backward and the loss
# and metric sums then run their *_det entry points (fixed summation order), and ops without one alert as torch's do.
def deterministic() -> bool:
    return torch.are_deterministic_algorithms_enabled()


_alerted = set()


def nondeterministic_alert(op: str) -> None:
    """torch's behaviour for an op without a deterministic implementation: raise, or warn once under warn_only=True."""
    msg = (f"{op} does not have a deterministic implementation, but you set 'torch.use_deterministic_algorithms(True)'. "
           "You can turn off determinism just for this operation, or you can use the 'warn_only=True' option, if that's "
           "acceptable for your application.")
    if not torch.is_deterministic_algorithms_warn_only_enabled():
        raise RuntimeError(msg)
    if op not in _alerted:
        _alerted.add(op)
        warnings.warn(msg, UserWarning, stacklevel=3)


def _workspace(nbytes: int, what: str, device) -> torch.Tensor:
    if nbytes == 0:
        raise L.VsrbError(f"{what}: {L.load().vsrb_last_error().decode()}")
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


def require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise L.VsrbError(f"{what} lives on {t.device}: vsrlab_b200 runs on CUDA (sm_100a) only; there is no CPU path")


def check_conv_module(c) -> None:
    """The kernels implement the convolutions of the hot path: stride 1, 'same' zero padding, no dilation, no groups
    (reference conv.py:19,86-87,98; upsampling.py:7; basicvsr.py:18-21).  Anything else must fail loudly rather than
    silently compute a different convolution."""
    if not isinstance(c, torch.nn.Conv2d):
        return
    kh, kw = c.kernel_size
    ok = (tuple(c.stride) == (1, 1) and tuple(c.dilation) == (1, 1) and c.groups == 1 and c.padding_mode == "zeros"
          and c.padding in ((kh // 2, kw // 2), "same"))
    if not ok:
        raise L.VsrbError(f"unsupported Conv2d for the sm_100a kernels: stride={c.stride} padding={c.padding} dilation={c.dilation} "
                          f"groups={c.groups} padding_mode={c.padding_mode}; the hot path needs stride 1, padding k//2, no dilation, "
                          "groups 1")


class PackedConv:
    """Device image of one convolution's weights (or of `groups` same-shaped convolutions)
    in the layout the kernels consume; see vsrb_pack_conv_weight in include/vsrb200.h."""

    def __init__(self, convs: Sequence[torch.nn.Conv2d], segs: Sequence[Tuple[int, int]], dtype: int, pixshuf: int = 0):
        lib = L.load()
        w0 = convs[0].weight
        require_cuda(w0, "conv weight")
        cout, cin, kh, kw = w0.shape
        for c in convs:
            check_conv_module(c)
        self.split = dtype == BF16X2
        self.real_segs = tuple(segs)
        w = torch.stack([c.weight.detach().to(torch.float32) for c in convs]).contiguous()
        if self.split:
            # fp32-accurate mode: W = W_hi + W_lo (both bf16); every real segment becomes two weight segments
            # [W_hi | W_lo]; the launcher feeds (x_hi, W_hi), (x_lo, W_hi), (x_hi, W_lo) - the lo*lo term is dropped
            parts, new_segs, o = [], [], 0
            for off, c in segs:
                ws = w[:, :, off:off + c]
                hi = ws.to(torch.bfloat16).to(torch.float32)
                parts += [hi, ws - hi]
                new_segs += [(o, c), (o + c, c)]
                o += 2 * c
            w = torch.cat(parts, 2).contiguous()
            segs, cin, dtype = new_segs, o, BF16
        g = L.ConvGeom()
        g.kh, g.kw, g.n_seg = kh, kw, len(segs)
        for i, (off, c) in enumerate(segs):
            g.seg_off[i], g.seg_c[i] = off, c
        g.cout, g.pixshuf, g.groups, g.dtype, g.transpose = cout, pixshuf, len(convs), dtype, 0
        self.geom = g
        self.cout, self.cin, self.kh, self.kw = cout, cin, kh, kw
        self.cout_pad = (cout + 15) // 16 * 16
        self.dtype = dtype
        self.stamp = self.stamp_of(convs)
        self.uses = 0            # launches since packing; PDL is enabled from the second one on
        b = None
        if convs[0].bias is not None:
            b = torch.stack([c.bias.detach().to(torch.float32) for c in convs]).contiguous()
        nbytes = lib.vsrb_packed_weight_bytes(C.byref(g))
        if nbytes == 0:
            raise L.VsrbError(f"unsupported conv geometry: {lib.vsrb_last_error().decode()}")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        L.check(lib.vsrb_pack_conv_weight(C.byref(g), _p(w), cin, _p(b), _p(self.buf), _stream()), "vsrb_pack_conv_weight")

    @staticmethod
    def stamp_of(convs) -> tuple:
        """Identity + version of the parameters a packed image was built from.  In-place updates through `param.data`
        bypass `_version`: code that writes weights that way must call `functional.clear_caches()` afterwards
        (optimizers, `load_state_dict` and `.to()` all bump the version or replace the storage)."""
        return tuple((c.weight.data_ptr(), c.weight._version, 0 if c.bias is None else c.bias._version) for c in convs)


def conv2d_fwd(pc: PackedConv, ins: Sequence, in_c: Sequence[int], batch: int, h: int, w: int, *,
               imgs_per_group: Optional[int] = None, act: int = ACT_NONE, slope: float = 0.1, epilogue: int = EPI_NHWC,
               out=None, out_c: int = 0, out_img_stride: int = 0, out_group_stride: int = 0, residual=None, res_c: int = 0,
               f32_io=None, f32_in=None, aux_hw: Tuple[int, int] = (0, 0), max_ctas: int = 0, extra_flags: int = 0,
               patch=None, patch_img_stride: int = 0, patch_group_stride: int = 0):
    """Enqueue one fused convolution.  `ins`, `out`, `residual`, `f32_io`, `f32_in` are tensors
    (or raw int device addresses) that the caller keeps alive."""
    a = L.ConvArgs()
    a.geom = pc.geom
    if pc.split:
        # inputs are split-bf16 tensors [hi Cp | lo Cp]; three operands per real segment share two weight segments
        k = 0
        for i, t in enumerate(ins):
            ptr = t if isinstance(t, int) else t.data_ptr()
            cp = in_c[i] // 2
            for c0, wseg in ((0, 2 * i), (cp, 2 * i), (0, 2 * i + 1)):
                a.inp[k], a.in_c[k], a.in_c0[k], a.in_wseg[k] = ptr, in_c[i], c0, wseg
                k += 1
        a.n_in = k
        a.split = 1 if epilogue in (EPI_NHWC, EPI_CLEAN) else 0
    else:
        for i, t in enumerate(ins):
            a.inp[i] = t if isinstance(t, int) else t.data_ptr()
            a.in_c[i] = in_c[i]
    a.batch, a.h, a.w = batch, h, w
    a.imgs_per_group = imgs_per_group if imgs_per_group is not None else batch // pc.geom.groups
    a.packed = pc.buf.data_ptr()
    a.act, a.slope, a.epilogue = act, slope, epilogue
    a.out = _p(out)
    a.out_c = out_c
    a.out_img_stride, a.out_group_stride = out_img_stride, out_group_stride
    a.residual = _p(residual)
    a.res_c = res_c
    a.f32_io = _p(f32_io)
    a.f32_in = _p(f32_in)
    a.aux_h, a.aux_w = aux_hw
    a.max_ctas = max_ctas
    if patch is not None:
        a.patch = _p(patch)
        a.patch_img_stride, a.patch_group_stride = patch_img_stride, patch_group_stride
    a.flags = (L.CONV_PDL if (pc.uses > 0 and PDL) else 0) | extra_flags
    pc.uses += 1
    if PROFILE is None:                            # the common case: no per-launch bookkeeping
        L.check(L.load().vsrb_conv2d_fwd(C.byref(a), _stream()), "vsrb_conv2d_fwd")
        return
    g = pc.geom
    flops = 2.0 * batch * h * w * pc.cout * sum(c for _, c in pc.real_segs) * pc.kh * pc.kw   # algorithmic (not x3)
    kind = ("conv_tc_x3" if pc.split else "conv_tc") if pc.dtype == BF16 else "conv_f32"
    if PROFILE_SHAPES:
        cin = "+".join(str(c) for _, c in pc.real_segs)
        kind += f"[{pc.kh}x{pc.kw} {cin}->{pc.cout} n{batch} {h}x{w} g{g.groups} epi{epilogue}{' res' if residual is not None else ''}]"
    with _Timed(kind, flops):
        L.check(L.load().vsrb_conv2d_fwd(C.byref(a), _stream()), "vsrb_conv2d_fwd")


def flow_warp(x, flow, out, n: int, h: int, w: int, c: int, dtype: int, padding: int = PAD_ZEROS,
              x_img_stride: int = 0, flow_img_stride: int = 0) -> None:
    with _Timed("flow_warp", float(n) * h * w * (2 * c * ESIZE[dtype] + 8)):
        L.check(L.load().vsrb_flow_warp(_p(x), x_img_stride, _p(flow), flow_img_stride, _p(out), n, h, w, c, dtype, padding,
                                        _stream()), "vsrb_flow_warp")


def flow_warp_ex(x, flow, out, n: int, h: int, w: int, c: int, dtype: int, interp: int = INTERP_BILINEAR, padding: int = PAD_ZEROS,
                 align_corners: bool = True, x_img_stride: int = 0, flow_img_stride: int = 0) -> None:
    """flow_warp with any grid_sample mode (INTERP_*, PAD_* incl. reflection, align_corners)."""
    with _Timed("flow_warp_ex", float(n) * h * w * (2 * c * ESIZE[dtype] + 8)):
        L.check(L.load().vsrb_flow_warp_ex(_p(x), x_img_stride, _p(flow), flow_img_stride, _p(out), n, h, w, c, dtype, interp, padding,
                                           int(bool(align_corners)), _stream()), "vsrb_flow_warp_ex")


def flow_warp_groups(x, x_strides: Tuple[int, int], flow, flow_strides: Tuple[int, int], out, imgs_per_group: int, groups: int, h: int,
                     w: int, c: int, dtype: int, padding: int = PAD_ZEROS) -> None:
    """One launch for `groups` sets of images that read different bases (x / flow: raw addresses + (image, group) strides)."""
    with _Timed("flow_warp", float(imgs_per_group * groups) * h * w * (2 * c * ESIZE[dtype] + 8)):
        L.check(L.load().vsrb_flow_warp_groups(_p(x), x_strides[0], x_strides[1], _p(flow), flow_strides[0], flow_strides[1], _p(out),
                                               imgs_per_group, groups, h, w, c, dtype, padding, _stream()), "vsrb_flow_warp_groups")


def nchw_to_nhwc(src: torch.Tensor, dst: torch.Tensor, n: int, c: int, h: int, w: int, c_dst: int, dtype: int) -> None:
    L.check(L.load().vsrb_nchw_to_nhwc(_p(src), _p(dst), n, c, h, w, c_dst, dtype, _stream()), "vsrb_nchw_to_nhwc")


def nhwc_to_nchw(src: torch.Tensor, dst: torch.Tensor, n: int, c: int, h: int, w: int, c_src: int, dtype: int) -> None:
    L.check(L.load().vsrb_nhwc_to_nchw(_p(src), _p(dst), n, c, h, w, c_src, dtype, _stream()), "vsrb_nhwc_to_nchw")


def spynet_pyramid_base(frames, lvl, F: int, h: int, w: int, Hp: int, Wp: int, mean, std) -> None:
    m = (C.c_float * 3)(*mean)
    s = (C.c_float * 3)(*std)
    L.check(L.load().vsrb_spynet_pyramid_base(_p(frames), _p(lvl), F, h, w, Hp, Wp, m, s, _stream()), "vsrb_spynet_pyramid_base")


def avgpool2_c4(src, dst, F: int, H: int, W: int) -> None:
    L.check(L.load().vsrb_avgpool2_c4(_p(src), _p(dst), F, H, W, _stream()), "vsrb_avgpool2_c4")


def spynet_level_input(lvl, ref_idx, supp_idx, flow_prev, flow_up, conv_in, P: int, Hl: int, Wl: int, c_in: int, dtype: int) -> None:
    with _Timed("spynet_glue", float(P) * Hl * Wl * (16 + 4 * 16 + 8 + 8 + c_in * ESIZE[dtype])):
        L.check(L.load().vsrb_spynet_level_input(_p(lvl), _p(ref_idx), _p(supp_idx), _p(flow_prev), _p(flow_up), _p(conv_in),
                                                 P, Hl, Wl, c_in, dtype, _stream()), "vsrb_spynet_level_input")


def flow_resize(fin, fout, P: int, Hp: int, Wp: int, h: int, w: int) -> None:
    L.check(L.load().vsrb_flow_resize(_p(fin), _p(fout), P, Hp, Wp, h, w, _stream()), "vsrb_flow_resize")


def im2col3x3(frames: torch.Tensor, patches: torch.Tensor, n: int, h: int, w: int) -> None:
    """fp32 NCHW [n,3,h,w] -> bf16 [n,h,w,32] 3x3 neighbourhoods (the K = 32 operand of the image stems)."""
    L.check(L.load().vsrb_im2col3x3_c3(_p(frames), _p(patches), n, h, w, _stream()), "vsrb_im2col3x3_c3")


def pixel_unshuffle2(src: torch.Tensor, dst: torch.Tensor, n: int, h: int, w: int, c: int) -> None:
    """bf16 NHWC [n,2h,2w,c] -> [n,h,w,4c] (inverse PixelShuffle(2), PyTorch channel order)."""
    L.check(L.load().vsrb_pixel_unshuffle2(_p(src), _p(dst), n, h, w, c, _stream()), "vsrb_pixel_unshuffle2")


def launch_count() -> int:
    return int(L.load().vsrb_launch_count())


def debug_status() -> int:
    return int(L.load().vsrb_debug_status(_stream()))


def device_info() -> Tuple[int, int, int]:
    a, b, c = C.c_int32(), C.c_int32(), C.c_int32()
    L.check(L.load().vsrb_device_info(C.byref(a), C.byref(b), C.byref(c)), "vsrb_device_info")
    return a.value, b.value, c.value


# --------------------------------------------------------------------------------------
# training kernels
# --------------------------------------------------------------------------------------
class PackedConvT(PackedConv):
    """Weights packed for the INPUT-GRADIENT convolution (transposed + flipped, geom.transpose = 1).  A list of convs of
    one shape packs as weight groups (the two propagation directions run as one launch)."""

    def __init__(self, conv, dtype: int):
        lib = L.load()
        convs = list(conv) if isinstance(conv, (list, tuple)) else [conv]
        for c in convs:
            check_conv_module(c)
        w0 = convs[0].weight
        require_cuda(w0, "conv weight")
        cout, cin, kh, kw = w0.shape
        g = L.ConvGeom()
        g.kh, g.kw, g.n_seg = kh, kw, 1
        g.seg_off[0], g.seg_c[0] = 0, cout
        g.cout, g.pixshuf, g.groups, g.dtype, g.transpose = cin, 0, len(convs), dtype, 1
        self.geom = g
        self.cout, self.cin, self.kh, self.kw = cin, cout, kh, kw      # of the gradient conv
        self.cout_pad = (cin + 15) // 16 * 16
        self.dtype = dtype
        self.stamp = self.stamp_of(convs)
        self.uses = 0
        self.split = False
        self.real_segs = ((0, cout),)
        w = torch.stack([c.weight.detach().to(torch.float32) for c in convs]).contiguous()
        nbytes = lib.vsrb_packed_weight_bytes(C.byref(g))
        if nbytes == 0:
            raise L.VsrbError(f"unsupported conv geometry: {lib.vsrb_last_error().decode()}")
        self.buf = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        L.check(lib.vsrb_pack_conv_weight(C.byref(g), _p(w), cout, None, _p(self.buf), _stream()), "vsrb_pack_conv_weight")


def conv2d_wgrad(geom: "L.ConvGeom", ins: Sequence[torch.Tensor], in_c: Sequence[int], dz: torch.Tensor, dz_c: int, batch: int,
                 h: int, w: int, cin_total: int, dw: torch.Tensor, db: Optional[torch.Tensor]) -> None:
    """dw (fp32 OIHW) += sum_pixels dz (x) x ;  db += sum_pixels dz.  `geom` = forward geometry without pixshuf."""
    if deterministic():
        if geom.dtype == BF16 and geom.kh == geom.kw:
            return conv2d_wgrad_det(geom, ins, in_c, dz, dz_c, batch, h, w, cin_total, dw, db)
        nondeterministic_alert(f"vsrlab_b200 conv weight gradient ({geom.kh}x{geom.kw} filter, FFMA kernel)")
    n = len(ins)
    ptrs = (C.c_void_p * 2)(*[t.data_ptr() for t in ins], *([None] * (2 - n)))
    cs = (C.c_int32 * 2)(*in_c, *([0] * (2 - n)))
    flops = 2.0 * batch * h * w * geom.cout * sum(geom.seg_c[i] for i in range(geom.n_seg)) * geom.kh * geom.kw
    cin = sum(geom.seg_c[i] for i in range(geom.n_seg))
    with _Timed(f"conv_wgrad[{geom.kh}x{geom.kw} {cin}->{geom.cout} {h}x{w}]" if PROFILE_SHAPES else "conv_wgrad", flops):
        L.check(L.load().vsrb_conv2d_wgrad(C.byref(geom), ptrs, cs, _p(dz), dz_c, batch, h, w, batch // geom.groups, cin_total,
                                           _p(dw), _p(db), _stream()), "vsrb_conv2d_wgrad")


def conv2d_wgrad_multi(geom: "L.ConvGeom", chunks: Sequence[Tuple[Sequence[torch.Tensor], torch.Tensor]], in_c: Sequence[int],
                       dz_c: int, batch: int, h: int, w: int, cin_total: int, dw: torch.Tensor, db: Optional[torch.Tensor]) -> None:
    """dw / db += the gradient summed over `chunks` = [(inputs of one use, its dz), ...] of one shape, without concatenating
    them (tensor-core path: bf16 3x3 convs whose input segments have a multiple of 64 channels)."""
    if deterministic():
        return conv2d_wgrad_multi_det(geom, chunks, in_c, dz_c, batch, h, w, cin_total, dw, db)
    n, ns = len(chunks), geom.n_seg
    ptrs = (C.c_void_p * (n * ns))(*[t.data_ptr() for ins, _ in chunks for t in ins])
    dzs = (C.c_void_p * n)(*[dz.data_ptr() for _, dz in chunks])
    cs = (C.c_int32 * ns)(*in_c)
    cin = sum(geom.seg_c[i] for i in range(ns))
    flops = 2.0 * n * batch * h * w * geom.cout * cin * geom.kh * geom.kw
    with _Timed(f"conv_wgrad[{geom.kh}x{geom.kw} {cin}->{geom.cout} {h}x{w} x{n}]" if PROFILE_SHAPES else "conv_wgrad", flops):
        L.check(L.load().vsrb_conv2d_wgrad_multi(C.byref(geom), n, ptrs, cs, dzs, dz_c, batch, h, w, cin_total, _p(dw), _p(db),
                                                 _stream()), "vsrb_conv2d_wgrad_multi")


def flow_warp_bwd(x, flow, dout, dx, dflow, n: int, h: int, w: int, c: int, dtype: int, padding: int = PAD_ZEROS) -> None:
    """dx = the gradient wrt x, dflow = the gradient wrt the flow (either may be None).  `dx` must be a ZEROED fp32 buffer:
    the default kernel adds into it with atomics, the deterministic one (torch.use_deterministic_algorithms) overwrites
    it, so a buffer that already holds a gradient would be accumulated in one mode and lost in the other.  To sum several
    warp gradients, add the results."""
    if deterministic():
        tpp = c // (8 if dtype == BF16 else 4)
        if dflow is None or (tpp <= 32 and tpp & (tpp - 1) == 0):
            return flow_warp_bwd_det(x, flow, dout, dx, dflow, n, h, w, c, dtype, padding)
        nondeterministic_alert(f"vsrlab_b200 flow_warp backward ({c} channels)")
    with _Timed("flow_warp_bwd", float(n) * h * w * (3 * c * ESIZE[dtype] + 4 * c * 4)):
        L.check(L.load().vsrb_flow_warp_bwd(_p(x), _p(flow), _p(dout), _p(dx), _p(dflow), n, h, w, c, dtype, padding, _stream()),
                "vsrb_flow_warp_bwd")


def flow_warp_ex_bwd(x, flow, dout, dx, dflow, n: int, h: int, w: int, c: int, dtype: int, interp: int = INTERP_BILINEAR,
                     padding: int = PAD_ZEROS, align_corners: bool = True) -> None:
    """flow_warp_bwd for every grid_sample mode; the same contract for `dx` (a zeroed buffer that receives the gradient)."""
    if deterministic():
        if interp == INTERP_BILINEAR and align_corners and padding in (PAD_ZEROS, PAD_BORDER):
            return flow_warp_bwd(x, flow, dout, dx, dflow, n, h, w, c, dtype, padding)
        nondeterministic_alert("vsrlab_b200 flow_warp backward (nearest / bicubic, reflection or align_corners=False; as "
                               "grid_sampler_2d_backward_cuda)")
    with _Timed("flow_warp_ex_bwd", float(n) * h * w * (3 * c * ESIZE[dtype] + 4 * c * 4)):
        L.check(L.load().vsrb_flow_warp_ex_bwd(_p(x), _p(flow), _p(dout), _p(dx), _p(dflow), n, h, w, c, dtype, interp, padding,
                                               int(bool(align_corners)), _stream()), "vsrb_flow_warp_ex_bwd")


# ---- deterministic variants (torch.use_deterministic_algorithms; see deterministic()) ----
def conv2d_wgrad_det(geom: "L.ConvGeom", ins: Sequence[torch.Tensor], in_c: Sequence[int], dz: torch.Tensor, dz_c: int, batch: int,
                     h: int, w: int, cin_total: int, dw: torch.Tensor, db: Optional[torch.Tensor]) -> None:
    """conv2d_wgrad with a fixed summation order (bf16 square filters)."""
    lib = L.load()
    n = len(ins)
    ptrs = (C.c_void_p * 2)(*[t.data_ptr() for t in ins], *([None] * (2 - n)))
    cs = (C.c_int32 * 2)(*in_c, *([0] * (2 - n)))
    ws = _workspace(lib.vsrb_conv2d_wgrad_det_workspace_bytes(C.byref(geom), 1, batch, h, w, int(db is not None)), "wgrad_det", dz.device)
    with _Timed("conv_wgrad_det", 2.0 * batch * h * w * geom.cout * sum(geom.seg_c[i] for i in range(geom.n_seg)) * geom.kh * geom.kw):
        L.check(lib.vsrb_conv2d_wgrad_det(C.byref(geom), ptrs, cs, _p(dz), dz_c, batch, h, w, batch // geom.groups, cin_total, _p(dw),
                                          _p(db), _p(ws), ws.numel(), _stream()), "vsrb_conv2d_wgrad_det")


def conv2d_wgrad_multi_det(geom: "L.ConvGeom", chunks: Sequence[Tuple[Sequence[torch.Tensor], torch.Tensor]], in_c: Sequence[int],
                           dz_c: int, batch: int, h: int, w: int, cin_total: int, dw: torch.Tensor, db: Optional[torch.Tensor]) -> None:
    """conv2d_wgrad_multi with a fixed summation order."""
    lib = L.load()
    n, ns = len(chunks), geom.n_seg
    ptrs = (C.c_void_p * (n * ns))(*[t.data_ptr() for ins, _ in chunks for t in ins])
    dzs = (C.c_void_p * n)(*[dz.data_ptr() for _, dz in chunks])
    cs = (C.c_int32 * ns)(*in_c)
    ws = _workspace(lib.vsrb_conv2d_wgrad_det_workspace_bytes(C.byref(geom), n, batch, h, w, int(db is not None)), "wgrad_multi_det",
                    dw.device)
    with _Timed("conv_wgrad_det", 2.0 * n * batch * h * w * geom.cout * sum(geom.seg_c[i] for i in range(ns)) * geom.kh * geom.kw):
        L.check(lib.vsrb_conv2d_wgrad_multi_det(C.byref(geom), n, ptrs, cs, dzs, dz_c, batch, h, w, cin_total, _p(dw), _p(db), _p(ws),
                                                ws.numel(), _stream()), "vsrb_conv2d_wgrad_multi_det")


def flow_warp_bwd_det(x, flow, dout, dx, dflow, n: int, h: int, w: int, c: int, dtype: int, padding: int = PAD_ZEROS) -> None:
    """flow_warp_bwd with dx OVERWRITTEN (fixed-point sums) and the default kernel's dflow."""
    lib = L.load()
    ws = _workspace(lib.vsrb_flow_warp_bwd_det_workspace_bytes(n, h, w, c), "flow_warp_bwd_det", dout.device) if dx is not None else None
    with _Timed("flow_warp_bwd_det", float(n) * h * w * (3 * c * ESIZE[dtype] + 4 * c * 4)):
        L.check(lib.vsrb_flow_warp_bwd_det(_p(x), _p(flow), _p(dout), _p(dx), _p(dflow), n, h, w, c, dtype, padding, _p(ws),
                                           0 if ws is None else ws.numel(), _stream()), "vsrb_flow_warp_bwd_det")


def loss_sums(name: str, query: Sequence, *args) -> None:
    """vsrb_<name>(*args) of loss.cu (charbonnier, charbonnier_resized, psnr_sums, ssim_sums); `query` = the shape arguments of its
    workspace query.  Deterministic mode: loss_sums_det."""
    if deterministic():
        return loss_sums_det(name, query, *args)
    L.check(getattr(L.load(), "vsrb_" + name)(*args, _stream()), "vsrb_" + name)


def loss_sums_det(name: str, query: Sequence, *args) -> None:
    lib = L.load()
    dev = torch.device("cuda", torch.cuda.current_device())
    ws = _workspace(getattr(lib, f"vsrb_{name}_det_workspace_bytes")(*query), name + "_det", dev)
    L.check(getattr(lib, f"vsrb_{name}_det")(*args, _p(ws), ws.numel(), _stream()), f"vsrb_{name}_det")
