"""Training path: the same modules under torch autograd.

Every convolution (forward, input gradient, weight/bias gradient) and every feature warp (forward,
backward wrt features and flow) runs in libvsrb200.so; torch autograd only records the graph and
differentiates the cheap glue around them (concats, the fp32 residue/flow additions, pyramid
resampling, the bilinear skip).  Activations are bf16 `channels_last` tensors, i.e. exactly the NHWC
buffers the kernels consume, so there is no layout copy between torch and the kernels.

Reference: train.py:90-101 drives `model(lr)` under autocast and calls `.backward()` on the
Charbonnier losses (core/utils.py:235-280); this module is what makes that work on the drop-in.
"""
from __future__ import annotations

import weakref
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from . import ops
from ._lib import ACT_LRELU, ACT_NONE, ACT_RELU, BF16, F32, PAD_BORDER, PAD_ZEROS, VsrbError
from . import _lib as L
import ctypes as C

CL = torch.channels_last
_packed_t = {}
_ACT = {"none": ACT_NONE, "relu": ACT_RELU, "lrelu": ACT_LRELU}


def _cl(t: torch.Tensor) -> torch.Tensor:
    return t if t.is_contiguous(memory_format=CL) else t.contiguous(memory_format=CL)


def _packed_transposed(conv) -> ops.PackedConvT:
    """`conv`: one module, or a tuple of same-shaped modules (weight groups)."""
    convs = tuple(conv) if isinstance(conv, (list, tuple)) else (conv,)
    key = tuple(id(c) for c in convs)
    from . import functional as VF
    if VF.REPACK_IN_CAPTURE and torch.cuda.is_current_stream_capturing():
        return ops.PackedConvT(convs, BF16)                     # weights change between replays: the pack kernels are part of the graph
    pc = _packed_t.get(key)
    if pc is None or pc.stamp != ops.PackedConv.stamp_of(convs) or any(r() is not c for r, c in zip(pc.owners_t, convs)):
        pc = ops.PackedConvT(convs, BF16)                       # (ids are recycled: the owners must be the same live modules)
        pc.owners_t = [weakref.ref(c, lambda _r, k=key: _packed_t.pop(k, None)) for c in convs]
        _packed_t[key] = pc
    return pc


def _wgrad_geom(conv, segs):
    g = L.ConvGeom()
    g.kh, g.kw, g.n_seg = conv.kernel_size[0], conv.kernel_size[1], len(segs)
    for i, (off, c) in enumerate(segs):
        g.seg_off[i], g.seg_c[i] = off, c
    g.cout, g.pixshuf, g.groups, g.dtype, g.transpose = conv.out_channels, 0, 1, BF16, 0
    return g


# Weight gradients of a recurrent layer: the propagation resblocks apply the same conv at every time step on a small
# batch (N images), so a weight-gradient launch per use runs on a handful of CTAs (measured: 64 us each on 16 CTAs, 330
# launches = 17 % of the cfg4 step).  Inside `batched_wgrad()` every conv of a forward pass gets ONE `_WeightNode`: the
# uses' backward passes only park (inputs, dz) in its box, and the node's own backward - which autograd runs after the
# last use - concatenates them along the batch dimension and launches the weight/bias gradient once.  The parameter
# still receives its gradient from a single autograd node, so hooks (DDP's reducer) see nothing unusual.
_WGRAD_SCOPE: Optional[dict] = None
_BATCH_PIXELS = 1 << 18      # uses with fewer pixels than this are batched; larger ones already fill the GPU


class batched_wgrad:
    def __enter__(self):
        global _WGRAD_SCOPE
        self.prev, _WGRAD_SCOPE = _WGRAD_SCOPE, {}
        return self

    def __exit__(self, *exc):
        global _WGRAD_SCOPE
        _WGRAD_SCOPE = self.prev
        return False


class _WeightNode(torch.autograd.Function):
    @staticmethod
    def forward(ctx, weight, bias, conv, segs, box):
        ctx.conv, ctx.segs, ctx.box, ctx.has_bias = conv, segs, box, bias is not None
        ctx.shape, ctx.device = weight.shape, weight.device
        return weight.new_zeros(1)

    @staticmethod
    def backward(ctx, _dtoken):
        conv, segs, box = ctx.conv, ctx.segs, ctx.box
        dw = torch.zeros(ctx.shape, dtype=torch.float32, device=ctx.device)
        db = torch.zeros(conv.out_channels, dtype=torch.float32, device=ctx.device) if ctx.has_bias else None
        g = _wgrad_geom(conv, segs)
        groups = {}
        for ins, dz in box:
            key = (tuple(ins[0].shape[2:]), tuple(t.shape[1] for t in ins), dz.shape[1])
            groups.setdefault(key, []).append((ins, dz))
        box.clear()
        for (hw, in_c, dz_c), items in groups.items():
            h, w = hw
            small = [it for it in items if it[1].shape[0] * h * w < _BATCH_PIXELS]
            big = [it for it in items if it[1].shape[0] * h * w >= _BATCH_PIXELS]
            tc = (conv.kernel_size == (3, 3) and all(c % 64 == 0 for _, c in segs) and len({it[1].shape[0] for it in small}) == 1
                  and all(t.is_contiguous(memory_format=CL) and t.data_ptr() % 16 == 0 for it in small for t in (*it[0], it[1])))
            if len(small) > 1 and tc:
                # tensor-core path: one launch walks the list of (inputs, dz) pairs, no concatenation
                ops.conv2d_wgrad_multi(g, small, list(in_c), dz_c, small[0][1].shape[0], h, w, conv.in_channels, dw, db)
            elif len(small) > 1:
                ins = [torch.cat([it[0][i] for it in small], 0) for i in range(len(in_c))]
                big.append((ins, torch.cat([it[1] for it in small], 0)))
            else:
                big += small
            for ins, dz in big:
                ops.conv2d_wgrad(g, ins, list(in_c), dz, dz_c, dz.shape[0], h, w, conv.in_channels, dw, db)
        return dw, db, None, None, None


def _weight_token(mod, segs):
    """(token, box) of `mod` in the current batched_wgrad scope, or (None, None) outside one / for frozen weights."""
    if _WGRAD_SCOPE is None or not mod.weight.requires_grad:
        return None, None
    ent = _WGRAD_SCOPE.get(id(mod))
    if ent is None or ent[2] is not mod or ent[3] != tuple(segs):
        box: list = []
        ent = (_WeightNode.apply(mod.weight, mod.bias, mod, tuple(segs), box), box, mod, tuple(segs))
        _WGRAD_SCOPE[id(mod)] = ent
    return ent[0], ent[1]


class ConvFn(torch.autograd.Function):
    """act(conv(cat(inputs))) [+ residual] [pixel-shuffled], bf16 channels_last in and out."""

    @staticmethod
    def forward(ctx, weight, bias, token, box, conv, segs, act, slope, pixshuf, residual, *inputs):
        from .functional import packed
        pc = packed([conv], segs, BF16, pixshuf)
        ins = [_cl(t) for t in inputs]
        b, _, h, w = ins[0].shape
        r = pixshuf or 1
        co = conv.out_channels // (r * r)
        oc = (co + 15) // 16 * 16
        out = torch.empty((b, oc, h * r, w * r), dtype=torch.bfloat16, device=ins[0].device, memory_format=CL)
        res = _cl(residual) if residual is not None else None
        if res is not None and act != "none":
            raise VsrbError("ConvFn: a fused residual needs act='none' (reference conv.py:89-92)")
        ops.conv2d_fwd(pc, ins, [t.shape[1] for t in ins], b, h, w, act=_ACT[act], slope=slope, out=out, out_c=oc,
                       residual=res, res_c=0 if res is None else res.shape[1])
        ctx.conv, ctx.segs, ctx.act, ctx.slope, ctx.pixshuf, ctx.box = conv, segs, act, slope, pixshuf, box
        ctx.has_res = res is not None
        ctx.save_for_backward(weight, out if act != "none" else None, *ins)
        return out

    @staticmethod
    def backward(ctx, dy):
        weight, out = ctx.saved_tensors[0], ctx.saved_tensors[1]
        ins = list(ctx.saved_tensors[2:])
        conv, segs = ctx.conv, ctx.segs
        dy = _cl(dy)
        d_res = dy if ctx.has_res else None
        dz = dy
        # one fused elementwise kernel each (compare + multiply + select were three passes: 7 GB of traffic on the HR
        # LeakyReLU of conv_last.0 alone)
        if ctx.act == "relu":
            dz = torch.ops.aten.threshold_backward(dy, out, 0)
        elif ctx.act == "lrelu":
            dz = torch.ops.aten.leaky_relu_backward(dy, out, ctx.slope, True)
        cout = conv.out_channels
        if ctx.pixshuf:
            cq = cout // (ctx.pixshuf ** 2)
            if ctx.pixshuf == 2 and dz.shape[1] == cq and cq % 8 == 0 and dz.dtype == torch.bfloat16:
                # the library's un-shuffle: one HBM-bound pass instead of torch's reshape/permute/contiguous chain
                src = _cl(dz)
                bb, _, hh, ww = src.shape
                dz = torch.empty((bb, cout, hh // 2, ww // 2), dtype=torch.bfloat16, device=src.device, memory_format=CL)
                ops.pixel_unshuffle2(src, dz, bb, hh // 2, ww // 2, cq)
            else:
                dz = F.pixel_unshuffle(dz[:, :cq], ctx.pixshuf)
        dz = _cl(dz)
        dz_c = dz.shape[1]
        b, _, h, w = ins[0].shape
        # weight / bias gradient: parked for the conv's _WeightNode inside batched_wgrad(), else computed here
        dw = db = None
        if ctx.box is not None:
            ctx.box.append((ins, dz))
        elif ctx.needs_input_grad[0]:
            g = _wgrad_geom(conv, segs)
            dw = torch.zeros_like(weight, dtype=torch.float32)
            db = torch.zeros(cout, dtype=torch.float32, device=weight.device) if conv.bias is not None else None
            ops.conv2d_wgrad(g, ins, [t.shape[1] for t in ins], dz, dz_c, b, h, w, conv.in_channels, dw, db)
        # input gradient: the forward kernel on dz with transposed + flipped weights
        d_ins: List[Optional[torch.Tensor]] = [None] * len(ins)
        if any(ctx.needs_input_grad[10 + i] for i in range(len(ins))):
            pt = _packed_transposed(conv)
            dx = torch.empty((b, pt.cout_pad, h, w), dtype=torch.bfloat16, device=dz.device, memory_format=CL)
            ops.conv2d_fwd(pt, [dz], [dz_c], b, h, w, act=ACT_NONE, out=dx, out_c=pt.cout_pad)
            for i, (off, c) in enumerate(segs):
                if not ctx.needs_input_grad[10 + i]:
                    continue
                ca = ins[i].shape[1]
                if len(segs) == 1 and ca == pt.cout_pad:
                    d_ins[i] = dx
                else:
                    d_ins[i] = F.pad(dx[:, off:off + c], (0, 0, 0, 0, 0, ca - c))
        return (dw, db if (conv.bias is not None and ctx.needs_input_grad[1]) else None, None, None, None, None, None, None, None, d_res,
                *d_ins)


class SrTailFn(torch.autograd.Function):
    """sr = conv_last.2(x) + bilinear_up(lq) (basicvsr.py:81-82) with the inference path's image epilogue (EPI_SR): the conv
    writes the fp32 NCHW frames with the skip term added.  (As separate torch ops the slice of the 3 real channels, its fp32
    copy, the upsampling, the sum and - in the backward - a zero-filled 16-channel HR gradient were seven passes over HR maps.)
    Backward: dz = the 3-channel gradient repacked to 16-channel NHWC bf16 by the library's layout kernel; weight / bias /
    input gradients as in ConvFn; d lq = the bilinear kernel's transpose (aten)."""

    @staticmethod
    def forward(ctx, weight, bias, token, box, conv, x, lq):
        from .functional import packed
        from ._lib import EPI_SR
        x = _cl(x)
        n, xc, hh, ww = x.shape
        pc = packed([conv], [(0, conv.in_channels)], BF16, 0)
        lqc = lq.detach().to(torch.float32).contiguous()
        sr = torch.empty((n, conv.out_channels, hh, ww), dtype=torch.float32, device=x.device)
        ops.conv2d_fwd(pc, [x], [xc], n, hh, ww, act=ACT_NONE, epilogue=EPI_SR, f32_io=sr, f32_in=lqc, aux_hw=tuple(lq.shape[-2:]))
        ctx.conv, ctx.box, ctx.lq_shape = conv, box, tuple(lq.shape)
        ctx.save_for_backward(weight, x)
        return sr

    @staticmethod
    def backward(ctx, dsr):
        weight, x = ctx.saved_tensors
        conv = ctx.conv
        n, xc, hh, ww = x.shape
        dsr = dsr.contiguous()
        dz = torch.empty((n, 16, hh, ww), dtype=torch.bfloat16, device=x.device, memory_format=CL)
        ops.nchw_to_nhwc(dsr, dz, n, conv.out_channels, hh, ww, 16, BF16)
        segs = ((0, conv.in_channels),)
        dw = db = None
        if ctx.box is not None:
            ctx.box.append(([x], dz))
        elif ctx.needs_input_grad[0]:
            dw = torch.zeros_like(weight, dtype=torch.float32)
            db = torch.zeros(conv.out_channels, dtype=torch.float32, device=weight.device) if conv.bias is not None else None
            ops.conv2d_wgrad(_wgrad_geom(conv, segs), [x], [xc], dz, 16, n, hh, ww, conv.in_channels, dw, db)
        dx = None
        if ctx.needs_input_grad[5]:
            pt = _packed_transposed(conv)
            dx = torch.empty((n, pt.cout_pad, hh, ww), dtype=torch.bfloat16, device=x.device, memory_format=CL)
            ops.conv2d_fwd(pt, [dz], [16], n, hh, ww, act=ACT_NONE, out=dx, out_c=pt.cout_pad)
            if pt.cout_pad != xc:
                dx = F.pad(dx[:, :conv.in_channels], (0, 0, 0, 0, 0, xc - conv.in_channels))
        dlq = None
        if ctx.needs_input_grad[6]:
            if ops.deterministic():
                dlq = _resize_bilinear_backward(dsr, ctx.lq_shape[-2:], False)
            else:
                dlq = torch.ops.aten.upsample_bilinear2d_backward(dsr, [hh, ww], list(ctx.lq_shape), False, None, None)
        return dw, (db if (conv.bias is not None and ctx.needs_input_grad[1]) else None), None, None, None, dx, dlq


def sr_tail(mod, x: torch.Tensor, lq: torch.Tensor) -> torch.Tensor:
    """conv_last.2 + skip; `lq` [N,3,h,w] fp32, the output is H / h times larger."""
    token, box = _weight_token(mod, ((0, mod.in_channels),))
    if token is not None:
        return SrTailFn.apply(mod.weight.detach(), None if mod.bias is None else mod.bias.detach(), token, box, mod, x, lq)
    return SrTailFn.apply(mod.weight, mod.bias, None, None, mod, x, lq)


class WarpFn(torch.autograd.Function):
    """flow_warp on a channels_last tensor (bf16 or fp32); flow [B,h,w,2] fp32."""

    @staticmethod
    def forward(ctx, x, flow, border):
        x = _cl(x)
        flow = flow.contiguous()
        b, c, h, w = x.shape
        dt = BF16 if x.dtype == torch.bfloat16 else F32
        out = torch.empty_like(x, memory_format=CL)
        ops.flow_warp(x, flow, out, b, h, w, c, dt, PAD_BORDER if border else PAD_ZEROS)
        ctx.border, ctx.dt = border, dt
        ctx.save_for_backward(x, flow)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, flow = ctx.saved_tensors
        dout = _cl(dout)
        b, c, h, w = x.shape
        dx32 = torch.zeros((b, h, w, c), dtype=torch.float32, device=x.device) if ctx.needs_input_grad[0] else None
        dflow = torch.empty_like(flow) if ctx.needs_input_grad[1] else None
        ops.flow_warp_bwd(x, flow, dout, dx32, dflow, b, h, w, c, ctx.dt, PAD_BORDER if ctx.border else PAD_ZEROS)
        dx = dx32.to(x.dtype).permute(0, 3, 1, 2) if dx32 is not None else None
        return dx, dflow, None


class WarpExFn(torch.autograd.Function):
    """WarpFn with any grid_sample mode: interp INTERP_*, padding PAD_* (reflection included), align_corners."""

    @staticmethod
    def forward(ctx, x, flow, interp, padding, align_corners):
        x = _cl(x)
        flow = flow.contiguous()
        b, c, h, w = x.shape
        dt = BF16 if x.dtype == torch.bfloat16 else F32
        out = torch.empty_like(x, memory_format=CL)
        ops.flow_warp_ex(x, flow, out, b, h, w, c, dt, interp, padding, align_corners)
        ctx.mode, ctx.dt = (interp, padding, align_corners), dt
        ctx.save_for_backward(x, flow)
        return out

    @staticmethod
    def backward(ctx, dout):
        x, flow = ctx.saved_tensors
        dout = _cl(dout)
        b, c, h, w = x.shape
        dx32 = torch.zeros((b, h, w, c), dtype=torch.float32, device=x.device) if ctx.needs_input_grad[0] else None
        dflow = torch.empty_like(flow) if ctx.needs_input_grad[1] else None
        ops.flow_warp_ex_bwd(x, flow, dout, dx32, dflow, b, h, w, c, ctx.dt, *ctx.mode)
        dx = dx32.to(x.dtype).permute(0, 3, 1, 2) if dx32 is not None else None
        return dx, dflow, None, None, None


# --------------------------------------------------------------------------------------
# the modules, differentiable
# --------------------------------------------------------------------------------------
def conv(mod, inputs: Sequence[torch.Tensor], segs, act="none", slope=0.1, pixshuf=0, residual=None) -> torch.Tensor:
    for t in (*inputs, *([] if residual is None else [residual])):
        if t.dtype != torch.bfloat16:      # e.g. a torch op in between ran under autocast, whose fp32 list includes upsampling
            raise VsrbError(f"autograd.conv: activations must be bf16, got {t.dtype}")
    token, box = _weight_token(mod, segs)
    if token is not None:      # the weight's gradient flows through the token's node; this use sees the weight as a constant
        return ConvFn.apply(mod.weight.detach(), None if mod.bias is None else mod.bias.detach(), token, box, mod, tuple(segs), act, slope,
                            pixshuf, residual, *inputs)
    return ConvFn.apply(mod.weight, mod.bias, None, None, mod, tuple(segs), act, slope, pixshuf, residual, *inputs)


def to_cl16(x: torch.Tensor) -> torch.Tensor:
    """[B,c,h,w] -> bf16 channels_last, channels zero-padded to a multiple of 16."""
    c = x.shape[1]
    pad = (-c) % 16
    x = x.to(torch.bfloat16)
    if pad:
        x = F.pad(x, (0, 0, 0, 0, 0, pad))
    return _cl(x)


class ResBlockFn(torch.autograd.Function):
    """A whole ResidualBlock (conv.py:94-103: stem conv + LeakyReLU, then B x [conv, ReLU, conv, + identity]) as ONE autograd
    node.  The recurrent propagation calls it 2T times per clip on small batches, where the per-node cost of torch autograd
    and of `Function.apply` (~50 us per conv, forward + backward) exceeded the kernels' run time; here the 1 + 2B forward
    launches and the backward (input-gradient convs with the skip connection fused as their residual, ReLU masks as one
    threshold_backward each, weight gradients parked for the convs' _WeightNodes) are plain loops."""

    @staticmethod
    def forward(ctx, rbs, segs, n_in, boxes, *tensors):
        """`rbs`: tuple of G same-shaped ResidualBlocks = weight groups; images [g*B/G, (g+1)*B/G) belong to group g (the two
        propagation directions run as one launch per layer).  `boxes[layer][g]`: where that conv's (inputs, dz) are parked."""
        from .functional import packed
        ins = [_cl(t) for t in tensors[:n_in]]
        per_g = [[rb.conv[0]] + [c for blk in rb.res_block for c in (blk.conv1, blk.conv2)] for rb in rbs]
        layers = [tuple(cg[j] for cg in per_g) for j in range(len(per_g[0]))]          # layer j = its conv in every group
        mid = layers[0][0].out_channels
        b, _, h, w = ins[0].shape
        dev = ins[0].device

        def new():
            return torch.empty((b, mid, h, w), dtype=torch.bfloat16, device=dev, memory_format=CL)
        x = new()
        ops.conv2d_fwd(packed(list(layers[0]), segs, BF16, 0), ins, [t.shape[1] for t in ins], b, h, w, act=ACT_LRELU, slope=0.1, out=x,
                       out_c=mid)
        saved = [x]
        one = ((0, mid),)
        for j in range(1, len(layers), 2):
            t = new()
            ops.conv2d_fwd(packed(list(layers[j]), one, BF16, 0), [x], [mid], b, h, w, act=ACT_RELU, out=t, out_c=mid)
            y = new()
            ops.conv2d_fwd(packed(list(layers[j + 1]), one, BF16, 0), [t], [mid], b, h, w, act=ACT_NONE, out=y, out_c=mid, residual=x,
                           res_c=mid)
            saved += [t, y]
            x = y
        ctx.segs, ctx.n_in, ctx.layers, ctx.boxes = segs, n_in, layers, boxes
        ctx.save_for_backward(*ins, *saved[:-1])
        return x

    @staticmethod
    def backward(ctx, dy):
        n_in, layers, segs, boxes = ctx.n_in, ctx.layers, ctx.segs, ctx.boxes
        ins = list(ctx.saved_tensors[:n_in])
        acts = list(ctx.saved_tensors[n_in:])          # x0, t1, x1, t2, x2, ... (the last block's output is not needed)
        b, _, h, w = ins[0].shape
        G = len(layers[0])
        n = b // G

        def park(j, xs, dz):
            for gi in range(G):
                if boxes[j][gi] is not None:
                    boxes[j][gi].append(([t[gi * n:(gi + 1) * n] for t in xs], dz[gi * n:(gi + 1) * n]))

        def dgrad(j, dz, residual=None):
            pt = _packed_transposed(layers[j])
            dx = torch.empty((b, pt.cout_pad, h, w), dtype=torch.bfloat16, device=dz.device, memory_format=CL)
            ops.conv2d_fwd(pt, [dz], [dz.shape[1]], b, h, w, act=ACT_NONE, out=dx, out_c=pt.cout_pad, residual=residual,
                           res_c=0 if residual is None else residual.shape[1])
            return dx
        g = _cl(dy)
        nb = (len(layers) - 1) // 2
        for i in range(nb - 1, -1, -1):
            x_in, t = acts[2 * i], acts[2 * i + 1]
            park(2 + 2 * i, [t], g)                                   # conv2: no activation, dz = g
            dt = dgrad(2 + 2 * i, g)
            dz1 = torch.ops.aten.threshold_backward(dt, t, 0)        # ReLU mask of conv1's output
            park(1 + 2 * i, [x_in], dz1)
            g = dgrad(1 + 2 * i, dz1, residual=g)                     # + the skip connection's gradient, fused
        x0 = acts[0]
        dz0 = torch.ops.aten.leaky_relu_backward(g, x0, 0.1, True)   # LeakyReLU(0.1) of the stem, from its output
        park(0, ins, dz0)
        d_ins: List[Optional[torch.Tensor]] = [None] * n_in
        if any(ctx.needs_input_grad[4 + i] for i in range(n_in)):
            dx = dgrad(0, dz0)
            for i, (off, c) in enumerate(segs):
                if ctx.needs_input_grad[4 + i]:
                    ca = ins[i].shape[1]
                    d_ins[i] = dx if (n_in == 1 and ca == dx.shape[1]) else F.pad(dx[:, off:off + c], (0, 0, 0, 0, 0, ca - c))
        return (None, None, None, None, *d_ins, *([None] * (len(ctx.needs_input_grad) - 4 - n_in)))


def resblock(rb, inputs, segs) -> torch.Tensor:
    """ResidualBlock.forward (conv.py:101-103) on bf16 channels_last tensors.  `rb` may be a tuple of same-shaped blocks:
    weight groups over equal slices of the batch (needs a batched_wgrad scope)."""
    rbs = tuple(rb) if isinstance(rb, (list, tuple)) else (rb,)
    mid = rbs[0].conv[0].out_channels
    if mid % 16:
        raise VsrbError(f"training path: mid_channels={mid} must be a multiple of 16 (bf16 NHWC activations are stored in "
                        "16-channel groups); the inference path pads, the differentiable path does not")
    per_g = [[r.conv[0]] + [c for blk in r.res_block for c in (blk.conv1, blk.conv2)] for r in rbs]
    if _WGRAD_SCOPE is not None and all(c.kernel_size == (3, 3) for cg in per_g for c in cg):
        # fused node; the weights' gradients flow through the convs' tokens (inputs of the node), parked per use
        toks, boxes = [], []
        for j in range(len(per_g[0])):
            row = []
            for cg in per_g:
                tok, box = _weight_token(cg[j], tuple(segs) if j == 0 else ((0, mid),))
                row.append(box)
                if tok is not None:
                    toks.append(tok)
            boxes.append(row)
        return ResBlockFn.apply(rbs, tuple(segs), len(inputs), boxes, *inputs, *toks)
    if len(rbs) != 1:
        raise VsrbError("grouped residual blocks need a batched_wgrad() scope and 3x3 convs")
    rb = rbs[0]
    x = conv(rb.conv[0], inputs, segs, "lrelu")
    for blk in rb.res_block:
        t = conv(blk.conv1, [x], [(0, mid)], "relu")
        x = conv(blk.conv2, [t], [(0, mid)], "none", residual=x)
    return x


def cleaner(cl, x: torch.Tensor) -> torch.Tensor:
    """IterativeRefinement on [B,3,h,w] fp32 (realbasicvsr.py:24-30), out of place under autograd."""
    mid = cl.resblock.conv[0].out_channels
    for _ in range(cl.steps):
        f = resblock(cl.resblock, [to_cl16(x)], [(0, 3)])
        x = x + conv(cl.conv, [f], [(0, mid)], "none")[:, :3].float()
    return x


_resize_mats: dict = {}


def _resize_matrix(size: int, out: int, align_corners: bool, device) -> torch.Tensor:
    """[out, size] fp32: the weights of F.interpolate's bilinear resize (no antialias) along one axis."""
    key = (size, out, bool(align_corners), str(device))
    m = _resize_mats.get(key)
    if m is None:
        o = torch.arange(out, dtype=torch.float64)
        if align_corners:
            pos = o * ((size - 1) / (out - 1) if out > 1 else 0.0)
        else:
            pos = ((o + 0.5) * (size / out) - 0.5).clamp_(min=0.0)
        i0 = pos.floor().clamp_(0, size - 1).long()
        i1 = (i0 + 1).clamp_(max=size - 1)
        f = (pos - i0.double()).float()
        m = torch.zeros(out, size)
        m[torch.arange(out), i0] += 1.0 - f
        m[torch.arange(out), i1] += f
        m = m.to(device)
        _resize_mats[key] = m
    return m


def _resize_bilinear(x: torch.Tensor, size, align_corners: bool) -> torch.Tensor:
    """F.interpolate(x, size, mode="bilinear", align_corners) as matrix products A_h @ x @ A_w^T (fp32), differentiable as
    is.  An axis that keeps its size is not multiplied, so a same-size resize is an exact identity.  torch's bilinear
    kernel parallelises over the output pixels only and loops over n * c inside each thread (0.08 - 0.2 ms per level on the
    224 x 2 flow maps of SPyNet's x2 upsampling), and its backward has no deterministic CUDA implementation."""
    n, c, h, w = x.shape
    oh, ow = size
    with torch.autocast("cuda", enabled=False):                           # flows stay fp32 (autocast would run the products in half)
        y = x.float().reshape(n * c, h, w)
        if oh != h:
            y = torch.matmul(_resize_matrix(h, oh, align_corners, x.device), y)          # rows
        if ow != w:
            y = torch.matmul(y, _resize_matrix(w, ow, align_corners, x.device).t())      # columns
        return y.view(n, c, oh, ow)


def _resize_bilinear_backward(g: torch.Tensor, size, align_corners: bool) -> torch.Tensor:
    """The gradient of _resize_bilinear wrt its [n, c, *size] input: A_h^T @ g @ A_w."""
    n, c, oh, ow = g.shape
    h, w = size
    y = g.float().reshape(n * c, oh, ow)
    if oh != h:
        y = torch.matmul(_resize_matrix(h, oh, align_corners, g.device).t(), y)
    if ow != w:
        y = torch.matmul(y, _resize_matrix(w, ow, align_corners, g.device))
    return y.reshape(n, c, h, w)


def _bilinear(x: torch.Tensor, size, align_corners: bool = False) -> torch.Tensor:
    """F.interpolate(x, size, mode="bilinear"); under torch.use_deterministic_algorithms the matrix products of
    _resize_bilinear, whose backward is deterministic."""
    if ops.deterministic():
        return _resize_bilinear(x, size, align_corners)
    return F.interpolate(x, size=size, mode="bilinear", align_corners=align_corners)


def _upsample2_aligned(x: torch.Tensor) -> torch.Tensor:
    """F.interpolate(x, scale_factor=2, mode="bilinear", align_corners=True) (spynet.py:64-66)."""
    return _resize_bilinear(x, (2 * x.shape[2], 2 * x.shape[3]), True)


def spynet(sp, ref: torch.Tensor, supp: torch.Tensor) -> torch.Tensor:
    """Spynet.forward with gradients (spynet.py:38-93); resampling glue in torch fp32, convs + warps native."""
    h, w = ref.shape[-2:]
    hp, wp = (h + 31) // 32 * 32, (w + 31) // 32 * 32
    ref = _bilinear(ref, (hp, wp))
    supp = _bilinear(supp, (hp, wp))
    refs, supps = [(ref - sp.mean) / sp.std], [(supp - sp.mean) / sp.std]
    for _ in range(5):
        refs.append(F.avg_pool2d(refs[-1], 2, 2))
        supps.append(F.avg_pool2d(supps[-1], 2, 2))
    refs, supps = refs[::-1], supps[::-1]
    flow = ref.new_zeros(ref.shape[0], 2, hp // 32, wp // 32)
    for level in range(6):
        flow_up = flow if level == 0 else _upsample2_aligned(flow) * 2.0
        s4 = _cl(F.pad(supps[level], (0, 0, 0, 0, 0, 1)))                       # fp32, 4 channels
        warped = WarpFn.apply(s4, flow_up.permute(0, 2, 3, 1).contiguous(), True)[:, :3]
        x = to_cl16(torch.cat([refs[level], warped, flow_up], 1))
        mods = sp.basic_module[level].basic_module
        for j in range(5):
            cv = mods[j].conv[0]
            x = conv(cv, [x], [(0, cv.in_channels)], "relu")
        flow = flow_up + x[:, :2].float()
    flow = _bilinear(flow, (h, w))
    # per-axis rescale without a host-built tensor (keeps the step capturable in a CUDA graph)
    return torch.cat([flow[:, :1] * (float(w) / float(wp)), flow[:, 1:] * (float(h) / float(hp))], 1)


_gather_idx: dict = {}


def _gather_indices(n: int, t: int, device):
    """(perm, inverse): row r of [backward frames (nn, i) | forward frames (nn, i)] comes from row perm[r] of the
    concatenated steps; every row is taken exactly once, so the gradient is the inverse gather - no scatter-add."""
    key = (n, t, str(device))
    if key not in _gather_idx:
        ib = [(t - 1 - i) * 2 * n + nn for nn in range(n) for i in range(t)]
        jf = [i * 2 * n + n + nn for nn in range(n) for i in range(t)]
        perm = torch.tensor(ib + jf)
        _gather_idx[key] = (perm.to(device), torch.argsort(perm).to(device))
    return _gather_idx[key]


class _GatherFramesFn(torch.autograd.Function):
    """rows [t * 2n, h, w, C] of the propagation steps -> (backward features, forward features) in the output's (n, t)
    order.  The row selection is a permutation: forward one gather, backward one concatenation + the inverse gather
    (torch's index_select backward is an atomic index_add_: 0.44 ms per step on 240 maps of 64x64x64)."""

    @staticmethod
    def forward(ctx, rows, perm, inv):
        ctx.save_for_backward(inv)
        out = rows.index_select(0, perm)
        half = out.shape[0] // 2
        return out[:half], out[half:]

    @staticmethod
    def backward(ctx, g_bk, g_fw):
        inv, = ctx.saved_tensors
        return torch.cat([g_bk, g_fw], 0).index_select(0, inv), None, None


class _GatherStepsFn(torch.autograd.Function):
    """rows [R, ...] -> one tensor per propagation step (rows idx[k * per : (k + 1) * per] each), made by ONE gather; the
    gradient is one stack + one index_add_ on a small tensor.  (Slicing the frames / flows of a step out of their clip
    tensors inside the loop cost a zero-fill of the whole clip tensor plus an add per step in the backward pass.)"""

    @staticmethod
    def forward(ctx, rows, idx, steps):
        ctx.save_for_backward(idx)
        ctx.n_rows = rows.shape[0]
        out = rows.index_select(0, idx)
        return tuple(out.view(steps, -1, *rows.shape[1:]).unbind(0))

    @staticmethod
    def backward(ctx, *gs):
        idx, = ctx.saved_tensors
        ref = next(g for g in gs if g is not None)
        g = torch.stack([torch.zeros_like(ref) if x is None else x for x in gs], 0).flatten(0, 1)
        out = torch.zeros((ctx.n_rows, *g.shape[1:]), dtype=g.dtype, device=g.device)
        return out.index_add_(0, idx, g), None, None


_step_idx: dict = {}


def _step_indices(n: int, t: int, device):
    """(frame rows, flow rows) per step: step k runs frame t-1-k of the backward chain (images [0, n)) and frame k of the
    forward chain (images [n, 2n)); from step 1 on it warps with backward flow t-1-k and forward flow k-1."""
    key = (n, t, str(device))
    if key not in _step_idx:
        fr = [v for k in range(t) for v in ([nn * t + (t - 1 - k) for nn in range(n)] + [nn * t + k for nn in range(n)])]
        m = n * (t - 1)
        fw = [v for k in range(1, t) for v in ([nn * (t - 1) + (t - 1 - k) for nn in range(n)] + [m + nn * (t - 1) + (k - 1) for nn in range(n)])]
        _step_idx[key] = (torch.tensor(fr).to(device), torch.tensor(fw, dtype=torch.long).to(device))
    return _step_idx[key]


def basicvsr(bv, lrs: torch.Tensor) -> torch.Tensor:
    """BasicVSR.forward with gradients (basicvsr.py:39-83)."""
    from . import functional as VF
    n, t, c, h, w = lrs.shape
    mid = bv.mid_channels
    train_flow = any(p.requires_grad for p in bv.spynet.parameters())
    a = lrs[:, :-1].reshape(-1, c, h, w)
    b = lrs[:, 1:].reshape(-1, c, h, w)
    if train_flow:
        # both directions as one batch (first the backward pairs, then the forward pairs), like the inference path
        fl = spynet(bv.spynet, torch.cat([a, b], 0), torch.cat([b, a], 0))
        flows = fl.permute(0, 2, 3, 1).contiguous()                          # [2m, h, w, 2]: backward pairs, then forward pairs
    else:
        with torch.no_grad():
            ref, supp = VF._pair_indices(n, t, lrs.device)
            flows = VF._spynet_run(bv.spynet, lrs.detach().reshape(n * t, c, h, w).contiguous(), ref, supp, BF16)
    idx_frames, idx_flows = _step_indices(n, t, lrs.device)
    lr_rows = to_cl16(lrs.reshape(n * t, c, h, w)).permute(0, 2, 3, 1)       # [n * t, h, w, 16], plain contiguous view
    lr_steps = _GatherStepsFn.apply(lr_rows, idx_frames, t)
    flow_steps = _GatherStepsFn.apply(flows, idx_flows, t - 1) if t > 1 else ()
    segs = [(3, mid), (0, 3)]
    # both directions advance together: step k runs frame t-1-k of the backward chain and frame k of the forward chain as
    # the two weight groups of one launch per layer (images [0, n) backward, [n, 2n) forward)
    feats: List[torch.Tensor] = []
    feat = torch.zeros((2 * n, mid, h, w), dtype=torch.bfloat16, device=lrs.device).contiguous(memory_format=CL)
    for k in range(t):
        if k > 0:
            feat = WarpFn.apply(feat, flow_steps[k - 1], False)
        feat = resblock((bv.backward_resblocks, bv.forward_resblocks), [feat, lr_steps[k].permute(0, 3, 1, 2)], segs)
        feats.append(feat)
    # fusion + reconstruction, batched over frames in the output's (n, t) order: one gather per direction out of the
    # concatenated steps (slicing every step's `feat` in two cost five slow strided kernels per step in the backward pass)
    allf = torch.cat(feats, 0).permute(0, 2, 3, 1)                           # [t * 2n, h, w, C]: plain contiguous view
    perm, inv = _gather_indices(n, t, lrs.device)
    bk, fw = _GatherFramesFn.apply(allf, perm, inv)
    bk = bk.permute(0, 3, 1, 2)                                              # frame (nn, i) = step t-1-i, image nn
    fw = fw.permute(0, 3, 1, 2)                                              # frame (nn, i) = step i, image n + nn
    x = conv(bv.point_conv[0], [bk, fw], [(0, mid), (mid, mid)], "lrelu")
    for up in bv.upsample:
        x = conv(up.upconv, [x], [(0, mid)], "none", pixshuf=2)
    x = conv(bv.conv_last[0], [x], [(0, mid)], "lrelu")
    scale = 2 ** len(bv.upsample)
    last = bv.conv_last[2]
    if last.out_channels == 3 and c == 3 and last.kernel_size == (3, 3) and last.in_channels % 16 == 0:
        sr = sr_tail(last, x, lrs.reshape(n * t, c, h, w))                   # conv + bilinear skip in one kernel
    else:
        x = conv(last, [x], [(0, last.in_channels)], "none")[:, :c].float()
        lq = lrs.reshape(n * t, c, h, w)
        if ops.deterministic():
            sr = x + _resize_bilinear(lq, (h * scale, w * scale), False)
        else:
            sr = x + F.interpolate(lq, scale_factor=scale, mode="bilinear", align_corners=False)
    return sr.view(n, t, c, h * scale, w * scale)


def realbasicvsr(model, lr: torch.Tensor, write_back: bool = True):
    """(sr, lq) with gradients.  The cleaned clip is also written back into the caller's `lr`, which is what the
    reference's in-place refinement leaves there (realbasicvsr.py:26-29); `write_back=False` leaves that to the caller
    (graphs.py replays this body on a static copy of the input)."""
    n, t, c, h, w = lr.shape
    with batched_wgrad():
        lq = cleaner(model.cleaner, lr.reshape(n * t, c, h, w).float()).view(n, t, c, h, w)
        sr = basicvsr(model.basicvsr, lq)
    if write_back:
        with torch.no_grad():
            lr.copy_(lq)
    return sr, lq


# --------------------------------------------------------------------------------------
# GAN discriminator (SURVEY §8f row 4): SpectralConv / UNetDiscriminator on the same conv kernels
# --------------------------------------------------------------------------------------
class _DerivedConv:
    """What ConvFn / PackedConv read from an nn.Conv2d, for a weight that is DERIVED from the module's parameters (spectral
    normalisation; the 3x3 re-layout of a 4x4 stride-2 filter).  Under autograd every forward call gets its OWN holder: the
    node keeps it alive until its backward has run, so a second forward before that backward (train_gan.py:52-53 calls the
    discriminator on hr and on sr, then backpropagates both) cannot swap the weight under the first one's input-gradient
    conv.  The packed-weight caches drop an entry when its holder dies."""

    def __init__(self):
        self.weight = self.bias = None
        self.kernel_size = (3, 3)
        self.in_channels = self.out_channels = 0
        self.stamp = None

    def set(self, weight):
        self.weight = weight
        self.out_channels, self.in_channels = weight.shape[0], weight.shape[1]
        return self


def _holder(sc, conv, w: torch.Tensor, derive):
    """Holder of derive(w): per call when a graph is recorded or the module is in training mode (u / v move every call);
    otherwise one per module, rebuilt when the parameters or the power-iteration vectors changed."""
    if conv.training or (torch.is_grad_enabled() and w.requires_grad):
        return _DerivedConv().set(derive(w))
    stamp = tuple((t.data_ptr(), t._version) for t in (conv.weight_orig, conv.weight_u, conv.weight_v))
    h = sc.__dict__.get("_vsrb_holder")
    if h is None or h.stamp != stamp:
        h = _DerivedConv().set(derive(w))
        h.stamp = stamp
        sc.__dict__["_vsrb_holder"] = h
    return h


def _normalised_weight(conv):
    """The weight `torch.nn.utils.spectral_norm` would hand to F.conv2d: its forward pre-hook recomputes `conv.weight` from
    weight_orig / u / v (one power iteration in training mode, like a real forward)."""
    for hook in conv._forward_pre_hooks.values():
        hook(conv, None)
    return conv.weight


_S2_IDX = None


def _stride2_as_3x3(w: torch.Tensor) -> torch.Tensor:
    """A 4x4, stride-2, pad-1 filter [co, ci, 4, 4] as the equivalent 3x3, stride-1, pad-1 filter [co, 4 ci, 3, 3] on the
    pixel-unshuffled input (channel 4c + 2dy + dx = input pixel (2Y+dy, 2X+dx)): output (Y, X) reads input row 2Y + ky - 1,
    i.e. unshuffled row Y + t - 1 with (t, dy) = (0,1), (1,0), (1,1), (2,0) for ky = 0..3; 20 of the 36 taps are zero."""
    global _S2_IDX
    if _S2_IDX is None or _S2_IDX[0].device != w.device:
        k_of = {(0, 1): 0, (1, 0): 1, (1, 1): 2, (2, 0): 3}
        idx = torch.zeros(2, 2, 3, 3, dtype=torch.long)
        msk = torch.zeros(2, 2, 3, 3)
        for (ty, dy), ky in k_of.items():
            for (tx, dx), kx in k_of.items():
                idx[dy, dx, ty, tx] = ky * 4 + kx
                msk[dy, dx, ty, tx] = 1.0
        _S2_IDX = (idx.flatten().to(w.device), msk.flatten().to(w.device))
    idx, msk = _S2_IDX
    co, ci = w.shape[:2]
    w3 = w.flatten(2)[:, :, idx] * msk.to(w.dtype)                       # [co, ci, 36] ordered (dy, dx, ty, tx)
    return w3.view(co, ci * 4, 3, 3)


def spectral_conv(sc, x: torch.Tensor, act: str, slope: float) -> torch.Tensor:
    """act(SpectralConv(x)) on a bf16 channels_last tensor (channels padded to 16): 3x3 stride 1, or 4x4 stride 2 as
    pixel-unshuffle + 3x3 (exact)."""
    conv = sc.conv
    w = _normalised_weight(conv)
    cin = conv.in_channels
    if conv.kernel_size == (3, 3) and conv.stride == (1, 1) and conv.padding == (1, 1):
        return globals()["conv"](_holder(sc, conv, w, lambda t: t), [x], [(0, cin)], act, slope)
    if conv.kernel_size == (4, 4) and conv.stride == (2, 2) and conv.padding == (1, 1):
        if cin % 4:
            raise VsrbError("4x4 stride-2 SpectralConv: in_channels must be a multiple of 4 on this path")
        xs = _cl(F.pixel_unshuffle(x[:, :cin], 2))
        return globals()["conv"](_holder(sc, conv, w, _stride2_as_3x3), [xs], [(0, 4 * cin)], act, slope)
    raise VsrbError(f"SpectralConv geometry k={conv.kernel_size} stride={conv.stride} pad={conv.padding} is not implemented "
                    "(3x3 s1 p1 and 4x4 s2 p1 are)")


def unet_discriminator(D, img: torch.Tensor) -> torch.Tensor:
    """UNetDiscriminator.forward (unet-discriminator.py:19-31)."""
    def up(t):     # (autocast lists upsampling as an fp32 op: back to bf16 for the next conv)
        return _cl(F.interpolate(t, scale_factor=2, mode="bilinear", align_corners=False).to(torch.bfloat16))
    mid = D.conv_0.out_channels
    f0 = conv(D.conv_0, [to_cl16(img)], [(0, img.shape[1])], "lrelu", 0.2)
    f1 = spectral_conv(D.conv_1, f0, "lrelu", 0.2)
    f2 = spectral_conv(D.conv_2, f1, "lrelu", 0.2)
    f3 = spectral_conv(D.conv_3, f2, "lrelu", 0.2)
    f3 = up(f3)
    f4 = up(spectral_conv(D.conv_4, f3, "lrelu", 0.2) + f2)
    f5 = up(spectral_conv(D.conv_5, f4, "lrelu", 0.2) + f1)
    f6 = spectral_conv(D.conv_6, f5, "lrelu", 0.2) + f0
    out = spectral_conv(D.conv_7, f6, "lrelu", 0.2)
    out = spectral_conv(D.conv_8, out, "lrelu", 0.2)
    return conv(D.conv_9, [out], [(0, mid)], "none")[:, :1].float().contiguous()
