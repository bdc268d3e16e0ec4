"""BASELINE cfg4: Real-BasicVSR (experiment=basic, 5/5 blocks) training step on 15-frame 64x64 LR patches,
batch 8 per GPU, Adam, Charbonnier losses as reference train.py / core/utils.py:235-280, DDP over NCCL when
launched with torchrun.  Prints one JSON line (rank 0)."""
import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

import torch
import torch.nn.functional as F

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))


def charbonnier(a, b):
    return torch.sqrt((a - b) ** 2 + 1e-9).mean()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--frames", type=int, default=15)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--train-flow", type=int, default=1)
    ap.add_argument("--graph", action="store_true",
                    help="additionally capture forward + backward + clip + Adam in ONE CUDA graph (torch whole-network capture, "
                         "single GPU) and time its replay: what the step costs once the host is out of the loop")
    ap.add_argument("--host-profile", action="store_true", help="cProfile one step on the host (stderr)")
    ap.add_argument("--kernel-profile", action="store_true", help="torch.profiler (CUPTI) table of every kernel of one step (stderr)")
    ap.add_argument("--deterministic", action="store_true",
                    help="also time the step under torch.use_deterministic_algorithms(True), alternating with the default mode "
                         "in rounds of --steps steps (single GPU)")
    a = ap.parse_args()
    if a.deterministic:
        os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")     # torch's condition for deterministic cuBLAS products
    import torch.distributed as dist
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    from vsrlab_b200 import ops
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(0)
    model = RealBasicVSR(cleaning_blocks=a.blocks, mid_channels=64, upscale=4, res_blocks=a.blocks, pretrained_flow=False,
                         train_flow=bool(a.train_flow)).to(dev).train()
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local]) if world > 1 else model
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.99), capturable=bool(a.graph and world == 1))
    g = torch.Generator().manual_seed(rank)
    lr = torch.rand(a.batch, a.frames, 3, 64, 64, generator=g).to(dev)
    hr = torch.rand(a.batch, a.frames, 3, 256, 256, generator=g).to(dev)

    def step():
        x = lr.clone()
        with torch.autocast("cuda", dtype=torch.bfloat16):
            sr, lq = net(x)
        loss = charbonnier(sr, hr) + charbonnier(lq, F.interpolate(hr.flatten(0, 1), size=(64, 64), mode="bilinear").view_as(lq))
        opt.zero_grad(set_to_none=True)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
        opt.step()
        return loss.detach()      # (a live `loss` would keep the graph and the parameters' grad accumulators alive)

    losses = []
    for _ in range(a.warmup):
        losses.append(step().item())
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        losses.append(step())
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / a.steps
    ms_graph = None
    if a.graph and world == 1:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                step()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        opt.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()

        def graph_body():
            x = lr.clone()
            with torch.autocast("cuda", dtype=torch.bfloat16):
                sr, lq = net(x)
            loss = charbonnier(sr, hr) + charbonnier(lq, F.interpolate(hr.flatten(0, 1), size=(64, 64), mode="bilinear").view_as(lq))
            loss.backward()
            torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
            opt.step()
            return loss
        with torch.cuda.graph(graph, stream=side):     # same stream as the warm-up: the parameters' grad accumulators live on it
            static_loss = graph_body()
        torch.cuda.synchronize()
        for _ in range(2):
            graph.replay()
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(a.steps):
            graph.replay()
        g1.record()
        torch.cuda.synchronize()
        ms_graph = g0.elapsed_time(g1) / a.steps
        print(f"graph replay: {ms_graph:.2f} ms per step, loss {float(static_loss):.5f}", file=sys.stderr)
    if a.kernel_profile and rank == 0:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof_k:
            step()
            torch.cuda.synchronize()
        print(prof_k.key_averages().table(sort_by="cuda_time_total", row_limit=40, max_name_column_width=70), file=sys.stderr)
        with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA], record_shapes=True) as prof_o:
            step()
            torch.cuda.synchronize()
        print(prof_o.key_averages(group_by_input_shape=True).table(sort_by="self_cuda_time_total", row_limit=30, max_name_column_width=40,
                                                                    max_shapes_column_width=70), file=sys.stderr)
        # the torch glue between the library's kernels: aten ops by input shape
        rows = [e for e in prof_o.key_averages(group_by_input_shape=True) if e.key.startswith("aten::") and e.device_time_total > 0]
        rows.sort(key=lambda e: -e.self_device_time_total)
        print("aten ops by self CUDA time:", file=sys.stderr)
        for e in rows[:45]:
            print(f"  {e.self_device_time_total / 1e3:8.3f} ms {e.count:4d}x  {e.key:34s} {str(e.input_shapes)[:110]}", file=sys.stderr)
    if a.host_profile and rank == 0:
        import cProfile
        import pstats
        pr = cProfile.Profile()
        t0 = time.perf_counter()
        pr.enable()
        step()
        pr.disable()
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        print(f"host time of one step {1e3 * (t1 - t0):.1f} ms (profiler on), +{1e3 * (time.perf_counter() - t1):.1f} ms GPU drain", file=sys.stderr)
        pstats.Stats(pr, stream=sys.stderr).sort_stats("tottime").print_stats(28)
    ops.PROFILE = []
    step()
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    fam = {}
    for kind, ev0, ev1, work, tag in prof:
        d = fam.setdefault(kind, [0.0, 0.0, 0])
        d[0] += ev0.elapsed_time(ev1)
        d[1] += work
        d[2] += 1
    det_ms = None
    if a.deterministic and world == 1:
        # both modes warmed up (each captures its own training graphs), then alternating rounds: the median per mode
        def timed(mode, n):
            torch.use_deterministic_algorithms(mode)
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            ev0.record()
            for _ in range(n):
                step()
            ev1.record()
            torch.cuda.synchronize()
            return ev0.elapsed_time(ev1) / n
        for mode in (False, True):
            timed(mode, a.warmup + 4)
        rounds = {False: [], True: []}
        for _ in range(5):
            for mode in (False, True):
                rounds[mode].append(timed(mode, a.steps))
        torch.use_deterministic_algorithms(False)
        med = {m: sorted(v)[len(v) // 2] for m, v in rounds.items()}
        try:
            power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(local)],
                                   capture_output=True, text=True, timeout=30).stdout.strip()
        except (OSError, subprocess.SubprocessError):
            power = "unknown"
        det_ms = {"gpu": torch.cuda.get_device_name(dev), "power_limit": power, "ms_default": round(med[False], 3),
                  "ms_deterministic": round(med[True], 3), "rounds_ms": {"default": [round(v, 3) for v in rounds[False]],
                                                                         "deterministic": [round(v, 3) for v in rounds[True]]},
                  "cost": f"{100.0 * (med[True] / med[False] - 1.0):+.1f} %"}
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        # replicas must hold identical weights after the all-reduced steps
        w0 = torch.cat([p.detach().flatten() for p in model.parameters()])
        ref = w0.clone()
        dist.broadcast(ref, 0)
        same = bool(torch.equal(w0, ref))
    else:
        same = True
    if rank == 0:
        print(json.dumps({
            "workload": f"cfg4 training step: batch {a.batch}/GPU x {a.frames} frames 64x64, {a.blocks}/{a.blocks} blocks, train_flow={a.train_flow}",
            "n_gpus": world, "ms_per_step": t.item(), "ms_per_step_cuda_graph": ms_graph, "clips_per_sec": world * a.batch / (t.item() * 1e-3),
            "loss_first": float(losses[0]), "loss_last": float(losses[-1]), "replicas_identical": same,
            **({"deterministic": det_ms} if det_ms is not None else {}),
            "kernels_ms": {k: {"ms": round(v[0], 2), "launches": v[2], "tflops_or_gbs": round(v[1] / max(v[0], 1e-9) / 1e9, 1)}
                           for k, v in fam.items()},
        }), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
