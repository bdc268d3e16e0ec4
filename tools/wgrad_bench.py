"""Weight-gradient kernels on the shapes of the cfg4 training step: time per launch (CUDA events, L2 flushed between
launches) of the kernel the library's dispatch picks (csrc/wgrad_taps.cu or csrc/wgrad_tc.cu), with the VSRB_WG_DEBUG
decomposition (1 = no final atomics, 2 = no MMAs, 4 = no loads).

    python tools/wgrad_bench.py [--images 224]
"""
import argparse
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from vsrlab_b200 import _lib as L, load, ops  # noqa: E402
from vsrlab_b200._lib import BF16  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=224)
    ap.add_argument("--modes", default="default,default:1,default:2,default:3,default:4",
                    help="default (the library's dispatch), optionally :<VSRB_WG_DEBUG bits>")
    ap.add_argument("--sides", default="64,32,16")
    ap.add_argument("--shapes", default="", help="K,cin,x_channels,cout;... instead of the cfg4 list")
    a = ap.parse_args()
    if any(m.partition(":")[0] != "default" for m in a.modes.split(",")):
        ap.error(f"modes are default[:<VSRB_WG_DEBUG bits>], got {a.modes!r}")
    load()
    dev = torch.device("cuda:0")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    CL = torch.channels_last
    shapes = [(7, 8, 16, 32), (7, 32, 32, 64), (7, 64, 64, 32), (7, 32, 32, 16), (7, 16, 16, 2), (3, 3, 16, 64), (1, 128, 128, 64), (3, 64, 64, 64)]
    if a.shapes:
        shapes = [tuple(int(v) for v in sh.split(",")) for sh in a.shapes.split(";")]
    for side in [int(v) for v in a.sides.split(",")]:
        for K, cin, xc, cout in shapes:
            B = a.images
            zc = (cout + 15) // 16 * 16
            x = torch.randn(B, xc, side, side, device=dev).to(torch.bfloat16).contiguous(memory_format=CL)
            dz = torch.randn(B, zc, side, side, device=dev).to(torch.bfloat16).contiguous(memory_format=CL)
            geom = L.ConvGeom()
            geom.kh = geom.kw = K
            geom.n_seg, geom.cout, geom.pixshuf, geom.groups, geom.dtype, geom.transpose = 1, cout, 0, 1, BF16, 0
            geom.seg_off[0], geom.seg_c[0] = 0, cin
            dw = torch.zeros(cout, cin, K, K, dtype=torch.float32, device=dev)
            flops = 2.0 * B * side * side * cin * cout * K * K
            row = []
            for mode in a.modes.split(","):
                dbg = mode.partition(":")[2]
                os.environ.pop("VSRB_WG_DEBUG", None)
                if dbg:
                    os.environ["VSRB_WG_DEBUG"] = dbg
                ts = []
                for i in range(6):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    ops.conv2d_wgrad(geom, [x], [xc], dz, zc, B, side, side, cin, dw, None)
                    e1.record()
                    torch.cuda.synchronize()
                    if i >= 2:
                        ts.append(e0.elapsed_time(e1) * 1e3)
                us = sorted(ts)[len(ts) // 2]
                row.append(f"{mode} {us:7.1f} us ({flops / us / 1e6:6.1f} TF/s)")
            print(f"{K}x{K} {cin:3d}->{cout:3d} {B}x{side}x{side}: " + " | ".join(row), flush=True)
    os.environ.pop("VSRB_WG_DEBUG", None)


if __name__ == "__main__":
    main()
