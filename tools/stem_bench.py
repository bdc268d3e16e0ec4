"""Propagation stem: [stem conv] alone and [flow_warp x2 + stem conv], two weight groups x `imgs` images, replayed from a CUDA
graph between two ordinary resblock convs (so launch overlap is realistic).  With VSRB_RING_DEBUG=64 it prints the ring-walk
kernel's cycle counters for the stem instead.
    python tools/stem_bench.py [--imgs 2]
"""
import argparse
import os
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
from vsrlab_b200 import ops  # noqa: E402
from vsrlab_b200._lib import ACT_LRELU, ACT_RELU, BF16, PAD_ZEROS  # noqa: E402

dev = torch.device("cuda:0")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--imgs", type=int, default=2)
    ap.add_argument("--h", type=int, default=180)
    ap.add_argument("--w", type=int, default=320)
    ap.add_argument("--reps", type=int, default=30)
    a = ap.parse_args()
    n, h, w = a.imgs, a.h, a.w
    B = 2 * n
    stem = ops.PackedConv([torch.nn.Conv2d(67, 64, 3, 1, 1).to(dev) for _ in range(2)], [(3, 64), (0, 3)], BF16)
    body = ops.PackedConv([torch.nn.Conv2d(64, 64, 3, 1, 1).to(dev) for _ in range(2)], [(0, 64)], BF16)
    feat = torch.randn(B, h, w, 64, device=dev).to(torch.bfloat16)
    flow = (torch.rand(B, h, w, 2, device=dev) - 0.5) * 3.0
    lr = torch.rand(B, h, w, 16, device=dev).to(torch.bfloat16)
    patches = torch.randn(B, h, w, 32, device=dev).to(torch.bfloat16)
    warped, x1, x2 = (torch.empty_like(feat) for _ in range(3))

    def separate():
        ops.flow_warp(feat[:n], flow[:n], warped[:n], n, h, w, 64, BF16, PAD_ZEROS)
        ops.flow_warp(feat[n:], flow[n:], warped[n:], n, h, w, 64, BF16, PAD_ZEROS)
        ops.conv2d_fwd(stem, [warped, lr], [64, 16], B, h, w, act=ACT_LRELU, out=x1, out_c=64, patch=patches)

    def stem_only():
        ops.conv2d_fwd(stem, [feat, lr], [64, 16], B, h, w, act=ACT_LRELU, out=x1, out_c=64, patch=patches)

    def body_only():
        pass

    def run(fn):
        def chain():
            for _ in range(a.reps):
                fn()
                ops.conv2d_fwd(body, [x1], [64], B, h, w, act=ACT_RELU, out=x2, out_c=64)
                ops.conv2d_fwd(body, [x2], [64], B, h, w, act=ACT_RELU, out=feat, out_c=64)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            chain()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            chain()
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        assert ops.debug_status() == 0
        return ts[len(ts) // 2] * 1e3 / a.reps

    if os.environ.get("VSRB_RING_DEBUG") and int(os.environ["VSRB_RING_DEBUG"]) & 64:
        import ctypes as C
        from vsrlab_b200 import _lib as L
        buf = (C.c_uint64 * 8)()
        stem_only()
        L.load().vsrb_ring_debug_stats(buf, 1)
        for _ in range(20):
            stem_only()
        L.load().vsrb_ring_debug_stats(buf, 1)
        v = [x / 20 for x in buf]
        print(f"stem only: per launch: issuer wait acc-slot {v[0]:.0f} cyc, wait rows {v[1]:.0f} cyc, steps {v[2]:.1f}; warp4: "
              f"wait finished rows {v[3]:.0f}, epilogue {v[4]:.0f} cyc")
        return
    base = run(body_only)
    for name, fn in (("stem only (no warp)", stem_only), ("warp x2 + stem", separate)):
        t = run(fn)
        print(f"{name:22s}: {t - base:7.2f} us on top of the two body convs ({base:.2f} us)", flush=True)


if __name__ == "__main__":
    main()
