"""Fused training objective and on-device metrics for the callers of the hot path (SURVEY §8f row 2).

The reference computes `CharbonnierLoss(sr, hr) + CharbonnierLoss(lq, resize(hr, (h, w)))` with a dozen elementwise
torch kernels and then synchronises the host twice per step for `.item()` of PSNR / SSIM (train.py:93-101,
core/utils.py:235-252, core/metrics.py:13).  Here each loss term is ONE kernel forward (read x, y; reduce) and ONE
kernel backward (read x, y; write the gradient, scaled by the upstream gradient taken from device memory), the resize
of `hr` is computed inside the second term's kernel, and the metrics return device tensors.

* `CharbonnierLoss`          drop-in for `vsrlab.core.losses.CharbonnierLoss` (same constructor, same forward(x, y))
* `realbasicvsr_loss`        both terms of `compute_loss` (core/utils.py:235-240) in two launches
* `PerceptualLoss`, `AdversarialLoss`   the GAN recipe's two extra terms (core/losses.py:29-74; SURVEY §8f row 4): the VGG19
                             feature stack runs on the conv kernels (frozen weights: input gradients only)
* `PSNR`, `SSIM`             modules with piqa's call signature (defaults of piqa.PSNR / piqa.SSIM), results stay on
                             the device; `MetricCollection.forward` of the reference calls `.item()` on them, which works.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib as L
from .ops import _p, loss_sums, require_cuda


def _f32c(t: torch.Tensor) -> torch.Tensor:
    return t.detach().to(torch.float32).contiguous()


class _CharbonnierFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, eps):
        require_cuda(x, "charbonnier input")
        xc, yc = _f32c(x), _f32c(y)
        if xc.shape != yc.shape:
            raise L.VsrbError(f"CharbonnierLoss: shapes differ {tuple(xc.shape)} vs {tuple(yc.shape)}")
        acc = torch.zeros(1, dtype=torch.float64, device=x.device)
        loss_sums("charbonnier", (xc.numel(),), _p(xc), _p(yc), xc.numel(), eps, _p(acc), None, None, 1.0)
        ctx.save_for_backward(xc, yc)
        ctx.eps, ctx.x_dtype, ctx.y_dtype = eps, x.dtype, y.dtype
        return (acc / xc.numel()).to(torch.float32).squeeze(0)

    @staticmethod
    def backward(ctx, g):
        xc, yc = ctx.saved_tensors
        gx = torch.empty_like(xc)
        acc = torch.zeros(1, dtype=torch.float64, device=xc.device)
        gs = g.detach().to(torch.float32).contiguous()
        loss_sums("charbonnier", (xc.numel(),), _p(xc), _p(yc), xc.numel(), ctx.eps, _p(acc), _p(gx), _p(gs), 1.0 / xc.numel())
        gy = -gx if ctx.needs_input_grad[1] else None
        return (gx.to(ctx.x_dtype) if ctx.needs_input_grad[0] else None), (gy.to(ctx.y_dtype) if gy is not None else None), None


class _CharbonnierResizedFn(torch.autograd.Function):
    """mean(sqrt((lq - resize(hr, lq.shape[-2:]))^2 + eps)); gradient wrt lq only (hr is data)."""

    @staticmethod
    def forward(ctx, lq, hr, eps):
        require_cuda(lq, "charbonnier input")
        lc, hc = _f32c(lq), _f32c(hr)
        h, w = lc.shape[-2:]
        H, W = hc.shape[-2:]
        planes = lc.numel() // (h * w)
        if hc.numel() // (H * W) != planes:
            raise L.VsrbError("charbonnier_resized: lq and hr must have the same leading dimensions")
        acc = torch.zeros(1, dtype=torch.float64, device=lq.device)
        loss_sums("charbonnier_resized", (planes, h, w), _p(lc), _p(hc), planes, h, w, H, W, eps, _p(acc), None, None, 1.0)
        ctx.save_for_backward(lc, hc)
        ctx.eps, ctx.dtype = eps, lq.dtype
        return (acc / lc.numel()).to(torch.float32).squeeze(0)

    @staticmethod
    def backward(ctx, g):
        lc, hc = ctx.saved_tensors
        h, w = lc.shape[-2:]
        H, W = hc.shape[-2:]
        planes = lc.numel() // (h * w)
        gl = torch.empty_like(lc)
        acc = torch.zeros(1, dtype=torch.float64, device=lc.device)
        gs = g.detach().to(torch.float32).contiguous()
        loss_sums("charbonnier_resized", (planes, h, w), _p(lc), _p(hc), planes, h, w, H, W, ctx.eps, _p(acc), _p(gl), _p(gs),
                  1.0 / lc.numel())
        return gl.to(ctx.dtype), None, None


class CharbonnierLoss(torch.nn.Module):
    """Drop-in for the reference's CharbonnierLoss (core/losses.py:10-18): forward(x, y) = mean(sqrt((x-y)^2 + eps))."""

    def __init__(self, eps: float = 1e-9):
        super().__init__()
        self.eps = eps

    def forward(self, x, y):
        return _CharbonnierFn.apply(x, y, self.eps)


def realbasicvsr_loss(sr: torch.Tensor, hr: torch.Tensor, lq: Optional[torch.Tensor] = None, eps: float = 1e-9) -> torch.Tensor:
    """compute_loss of the reference (core/utils.py:235-240) with its Charbonnier loss: the resize of `hr` to lq's
    size happens inside the second term's kernel instead of materialising the resized clip."""
    loss = _CharbonnierFn.apply(sr, hr, eps)
    if lq is not None:
        loss = loss + _CharbonnierResizedFn.apply(lq, hr, eps)
    return loss


LAYER_WEIGHTS = {"2": 0.1, "7": 0.1, "16": 0.8, "25": 0.9, "34": 1.0}        # core/losses.py:8


class PerceptualLoss(torch.nn.Module):
    """`vsrlab.core.losses.PerceptualLoss` (core/losses.py:29-64) with the VGG19 feature stack on the sm_100a conv kernels:
    weight * sum_k layer_weights[k] * L1(features_k(yhat), features_k(y)).  Same constructor (`weight`); `vgg_layers` lets
    a caller hand in the `torchvision` feature stack (the default, like the reference, asks torchvision for the
    ImageNet-pretrained one, which needs a download).  Notes on fidelity: the reference stores `output[name] = x` and then
    runs the next `ReLU(inplace=True)` ON THAT TENSOR, so the features of layers 2, 7, 16 and 25 are post-ReLU and only
    layer 34 (the last of the slice) is a raw conv output - reproduced here by fusing each ReLU into its conv.  VGG
    parameters are frozen (core/losses.py:36-37): the backward computes input gradients only."""

    def __init__(self, weight=1, vgg_layers=None, layer_weights=None):
        super().__init__()
        self.weight = weight
        self.layer_weights = dict(layer_weights or LAYER_WEIGHTS)
        if vgg_layers is None:
            from torchvision import models
            vgg_layers = models.vgg19(weights="IMAGENET1K_V1").features[:max(map(int, self.layer_weights)) + 1]
        self.vgg_layers = vgg_layers
        for p in self.vgg_layers.parameters():
            p.requires_grad = False

    def features(self, x: torch.Tensor) -> dict:
        """x [N,3,h,w] -> {layer name: bf16 channels_last feature map}"""
        import torch.nn.functional as F
        from . import autograd as A
        require_cuda(x, "perceptual loss input")
        t = A.to_cl16(x)
        out = {}
        layers = list(self.vgg_layers.named_children())
        taps = self.layer_weights
        i = 0
        while i < len(layers):
            name, m = layers[i]
            if isinstance(m, torch.nn.Conv2d):
                nxt = layers[i + 1] if i + 1 < len(layers) else None
                relu = nxt is not None and isinstance(nxt[1], torch.nn.ReLU)
                # a tapped conv followed by an out-of-place ReLU keeps its raw output: do not fuse in that case
                fuse = relu and (nxt[1].inplace or name not in taps)
                t = A.conv(m, [t], [(0, m.in_channels)], "relu" if fuse else "none")
                if name in taps:
                    out[name] = t
                if fuse:
                    if nxt[0] in taps:
                        out[nxt[0]] = t
                    i += 1
            elif isinstance(m, torch.nn.MaxPool2d):
                t = A._cl(F.max_pool2d(t, m.kernel_size, m.stride, m.padding))
            elif isinstance(m, torch.nn.ReLU):
                t = F.relu(t)
            else:
                raise L.VsrbError(f"PerceptualLoss: layer {name} ({type(m).__name__}) is not part of a VGG feature stack")
            if name in taps and name not in out:
                out[name] = t
            i += 1
        return out

    def forward(self, yhat: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
        h, w = y.shape[-2:]
        fx = self.features(yhat.reshape(-1, 3, h, w))
        with torch.no_grad():
            fy = self.features(y.detach().reshape(-1, 3, h, w))
        loss = 0
        for k, wk in self.layer_weights.items():
            loss = loss + (fx[k].float() - fy[k].float()).abs().mean() * wk
        return loss * self.weight


class AdversarialLoss(torch.nn.Module):
    """`vsrlab.core.losses.AdversarialLoss` (core/losses.py:66-74): BCE-with-logits against a constant target; the weight
    applies to the generator's term only."""

    def __init__(self, weight=2e-5):
        super().__init__()
        self.weight = weight

    def forward(self, x, target, is_disc=False):
        import torch.nn.functional as F
        loss = F.binary_cross_entropy_with_logits(x, torch.full_like(x, float(target)))
        return loss if is_disc else loss * self.weight


class PSNR(torch.nn.Module):
    """piqa.PSNR semantics (epsilon 1e-8, value_range 1, reduction 'mean') on [N,C,H,W]; `x` is clamped to [0,1] inside the
    kernel (what core/utils.py:244 does before the call - clamping twice changes nothing)."""

    def __init__(self, epsilon: float = 1e-8, value_range: float = 1.0, reduction: str = "mean"):
        super().__init__()
        if value_range != 1.0:
            raise L.VsrbError("PSNR: value_range 1 only (frames are [0,1]-scaled on this path)")
        self.epsilon, self.reduction = epsilon, reduction

    def forward(self, x, y):
        require_cuda(x, "metric input")
        xc, yc = _f32c(x), _f32c(y)
        n = xc.shape[0]
        per = xc.numel() // n
        sums = torch.zeros(n, dtype=torch.float64, device=x.device)
        loss_sums("psnr_sums", (n, per), _p(xc), _p(yc), n, per, _p(sums))
        v = (10.0 * torch.log10(1.0 / (sums / per + self.epsilon))).to(torch.float32)
        return v.mean() if self.reduction == "mean" else (v.sum() if self.reduction == "sum" else v)


class SSIM(torch.nn.Module):
    """piqa.SSIM defaults (window 11, sigma 1.5, k1 0.01, k2 0.03, value_range 1, per-channel Gaussian filter with 'valid'
    borders, reduction 'mean') on [N,C,H,W], H, W >= 11."""

    def __init__(self, window_size: int = 11, sigma: float = 1.5, n_channels: int = 3, reduction: str = "mean", **kwargs):
        super().__init__()
        if window_size != 11 or sigma != 1.5 or kwargs.get("value_range", 1.0) != 1.0:
            raise L.VsrbError("SSIM: the fused kernel implements piqa's defaults (window 11, sigma 1.5, value_range 1)")
        self.reduction = reduction

    def forward(self, x, y):
        require_cuda(x, "metric input")
        xc, yc = _f32c(x), _f32c(y)
        n, c, h, w = xc.shape
        sums = torch.zeros(n, dtype=torch.float64, device=x.device)
        loss_sums("ssim_sums", (n, c, h, w), _p(xc), _p(yc), n, c, h, w, 1, _p(sums))
        v = (sums / (c * (h - 10) * (w - 10))).to(torch.float32)
        return v.mean() if self.reduction == "mean" else (v.sum() if self.reduction == "sum" else v)


def running_metrics_on_device(sr: torch.Tensor, hr: torch.Tensor):
    """compute_metric of the reference (core/utils.py:242-247) without host synchronisation: {'PSNR': t, 'SSIM': t}."""
    x = sr.detach().flatten(0, 1) if sr.dim() == 5 else sr.detach()
    y = hr.detach().flatten(0, 1) if hr.dim() == 5 else hr.detach()
    return {"PSNR": PSNR()(x, y), "SSIM": SSIM()(x, y)}
