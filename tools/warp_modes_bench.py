"""flow_warp_ex (every grid_sample mode) next to the default flow_warp kernel, in the method of warp_bench.py: a working
set larger than L2 (64 feature maps of 180 x 320 x 64: 472 MB in + 472 MB out in bf16, twice that in fp32), L2 flushed
before every timed launch, CUDA events.  Rate = algorithmic bytes (C x elem read + 8 B flow + C x elem written per
pixel, the same count for every mode) over the median kernel time; min and max of the repetitions show the spread.

    python tools/warp_modes_bench.py [--reps 20] [--n 64] [--mag 8]
"""
import argparse
import itertools
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from vsrlab_b200 import ops  # noqa: E402
from vsrlab_b200._lib import (BF16, F32, INTERP_BICUBIC, INTERP_BILINEAR, INTERP_NEAREST, PAD_BORDER,  # noqa: E402
                              PAD_REFLECTION, PAD_ZEROS)

dev = torch.device("cuda:0")
INTERPS = {"bilinear": INTERP_BILINEAR, "nearest": INTERP_NEAREST, "bicubic": INTERP_BICUBIC}
PADS = {"zeros": PAD_ZEROS, "border": PAD_BORDER, "reflection": PAD_REFLECTION}


def time_launch(fn, flush, reps):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], ts[0], ts[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--mag", type=float, default=8.0, help="flows uniform in +-mag px")
    a = ap.parse_args()
    n, h, w, c = a.n, 180, 320, 64
    print(f"# {torch.cuda.get_device_name(dev)}; n={n} {h}x{w}x{c}, flows +-{a.mag} px, {a.reps} reps, L2 flushed", flush=True)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev).manual_seed(0)
    fl = (torch.rand(n, h, w, 2, device=dev, generator=g) - 0.5) * 2 * a.mag
    print(f"{'dtype':5s} {'kernel':8s} {'interp':8s} {'padding':10s} {'align':5s} {'us':>8s} {'TB/s':>6s} {'min-max us':>17s}")
    for dt in (BF16, F32):
        x = torch.randn(n, h, w, c, device=dev, generator=g).to(ops.TORCH_DT[dt])
        out = torch.empty_like(x)
        byt = n * h * w * (2 * c * ops.ESIZE[dt] + 8)
        name = "bf16" if dt == BF16 else "fp32"
        ms, lo, hi = time_launch(lambda: ops.flow_warp(x, fl, out, n, h, w, c, dt, PAD_ZEROS), flush, a.reps)
        print(f"{name:5s} {'default':8s} {'bilinear':8s} {'zeros':10s} {'True':5s} {ms * 1e3:8.1f} {byt / ms / 1e9:6.2f} "
              f"{lo * 1e3:8.1f}-{hi * 1e3:<8.1f}", flush=True)
        for (iname, interp), (pname, pad), align in itertools.product(INTERPS.items(), PADS.items(), (True, False)):
            kern = "default" if interp == INTERP_BILINEAR and pad != PAD_REFLECTION and align else "ex"
            ms, lo, hi = time_launch(lambda: ops.flow_warp_ex(x, fl, out, n, h, w, c, dt, interp, pad, align), flush, a.reps)
            print(f"{name:5s} {kern:8s} {iname:8s} {pname:10s} {str(align):5s} {ms * 1e3:8.1f} {byt / ms / 1e9:6.2f} "
                  f"{lo * 1e3:8.1f}-{hi * 1e3:<8.1f}", flush=True)
        del x, out
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
