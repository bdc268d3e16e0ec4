"""SPyNet + flow_warp with the reference's names
(reference src/vsr/models/RealBasicVSR/modules/spynet.py:13-21 SpynetModule,
:23-93 Spynet, :95-106 flow_warp)."""
from collections import OrderedDict

import torch
from torch import nn

from vsrlab.core import PROJECT_ROOT
from vsrlab.core.modules.conv import ConvReLU
from vsrlab_b200 import functional as VF


class SpynetModule(nn.Module):
    """8 -> 32 -> 64 -> 32 -> 16 -> 2, 7x7, ReLU after every conv (spynet.py:13-21)."""

    def __init__(self):
        super().__init__()
        widths = (8, 32, 64, 32, 16, 2)     # [ref rgb, warped rgb, flow xy] -> flow residue
        self.basic_module = nn.Sequential(*[ConvReLU(ci, co, 7, 1, 3) for ci, co in zip(widths[:-1], widths[1:])])

    def forward(self, x):
        return VF.conv_chain(x, [m.conv[0] for m in self.basic_module], act="relu")


class Spynet(nn.Module):
    def __init__(self, pretrained: bool = False):
        super().__init__()
        self.basic_module = nn.ModuleList(SpynetModule() for _ in range(6))      # six pyramid levels, coarse to fine
        for name, rgb in (("mean", (0.485, 0.456, 0.406)), ("std", (0.229, 0.224, 0.225))):   # ImageNet statistics
            self.register_buffer(name, torch.tensor(rgb, dtype=torch.float32).view(1, 3, 1, 1))
        if pretrained:
            # the reference's blob location and key remap (spynet.py:32-36): "basic_module.N.basic_module.M" + ".0" + rest
            blob = torch.load(f"{PROJECT_ROOT}/src/optical_flow/weights/spynet-sintel.pth")
            self.basic_module.load_state_dict(OrderedDict((k[13:34] + ".0" + k[34:], v) for k, v in blob.items()))

    def compute_flow(self, ref, supp):
        """Flow on inputs whose sides are multiples of 32 (spynet.py:38-67)."""
        return VF.spynet_flow(self, ref, supp, resize=False)

    def forward(self, ref, supp):
        """Flow from `ref` to `supp`, [T,2,h,w] fp32 (spynet.py:69-93)."""
        return VF.spynet_flow(self, ref, supp, resize=True)


def flow_warp(x, flow, interpolation="bilinear", padding_mode="zeros", align_corners=True):
    """Backward warp; `flow` is channels-last [T,h,w,2] (spynet.py:95-106).  Every F.grid_sample mode: interpolation
    bilinear / nearest / bicubic, padding_mode zeros / border / reflection, align_corners True / False."""
    return VF.flow_warp(x, flow, padding_mode, interpolation, align_corners)
