"""Benchmark of the Real-BasicVSR x4 hot path (BASELINE.json: output frames/s, 720p out).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one `model(lr)` pass of the drop-in `vsrlab...RealBasicVSR` over `--clips`
synthetic 30-frame 180x320 clips per GPU (cfg3 of BASELINE.json, experiment=basic 5/5 blocks
unless --blocks is given), bf16 mode.  Prints ONE JSON line (rank 0).

--dump-outputs DIR writes the `sr` and `lq` that the last timed step returned (rank 0's clips) as
DIR/sr.npy and DIR/lq.npy, float32.  Inputs and weights are seeded, so two builds run with the same
arguments can be compared output for output.  An output larger than DUMP_ELEMS elements is written
as the 1-D sample at DUMP_ELEMS seeded flat indices (sorted, drawn with replacement), the same
indices on every run with the same arguments.

* value        frames/s, all ranks, inputs already resident in HBM (CUDA events, max over ranks)
* e2e          same metric through the public nn.Module call with pinned HOST buffers: H2D of the
               clip and D2H of sr/lq inside the timed region (`e2e_narrow`: the same with the opt-in
               uint8 `sr` output the reference's PNG dump consumes)
* roofline     the dominant kernel family (tcgen05 implicit-GEMM convs): algorithmic conv FLOPs / CUDA-event
               time of those launches, against MEASURED_PEAKS.json
* parity       the same 6 frames of one 180x320 clip through the reference's own modules on the CPU
               (oracle/_ref, else the oracle port) and through the GPU path: fp32-mode max-abs error,
               bf16-mode PSNR delta, flow error.  A broken gate fails the benchmark.
* cpu_baseline that reference run, timed (frames/s on this box's host cores)
* blocks20     the model-file default 20/20-block configuration (conf/train/model/basicvsr.yaml:2,5)
* train_cfg4   BASELINE cfg4: training step (fp16-requesting autocast + GradScaler + Adam, batch 8 x 15 frames
               64x64 per GPU), DDP over NCCL when N > 1
* --impl reference: the reference's own CPU implementation (oracle/_ref; else the oracle port) on all
               host cores, bounded sample per step.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "realbasicvsr_x4_output_frames_per_sec_720p"
UNIT = "frames/s"
T_FRAMES, LR_H, LR_W = 30, 180, 320
CFG4_FWD_GFLOP = {5: 3824.66, 20: 9260.48}        # SURVEY.md §8d: forward conv FLOPs of one cfg4 micro-batch; training ~ 3x
DUMP_ELEMS = 1 << 22                              # 16 MB of float32 per dumped array: sr + lq stay under 64 MB


def peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return {"hbm": d["hbm_gbs"], "tf_burst": d["bf16_tflops"], "tf_sust": d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                "src": "measured"}
    return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sust": 1400.0, "src": "fallback"}


def build_model(blocks: int, device, train_flow: bool = False):
    from vsrlab.vsr.models.RealBasicVSR.realbasicvsr import RealBasicVSR
    torch.manual_seed(0)
    m = RealBasicVSR(cleaning_blocks=blocks, mid_channels=64, upscale=4, res_blocks=blocks, pretrained_flow=False,
                     train_flow=train_flow)
    return m.to(device)


class ClockSampler(threading.Thread):
    """nvidia-smi-equivalent (NVML) clocks and throttle reasons during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.reasons, self.max_mhz = index, False, [], set(), None
        self.power_w, self.power_limit_w = [], None

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
                     0x80: "hw_power_brake_slowdown"}
            try:
                self.power_limit_w = nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0
            except Exception:  # noqa: BLE001
                pass
            while not self.stop_flag:
                self.sm.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    self.power_w.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception:  # noqa: BLE001
                    pass
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
                time.sleep(0.05)
        except Exception as e:  # noqa: BLE001
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def summary(self):
        sm = sorted(self.sm)
        pw = sorted(self.power_w)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "power_w": pw[len(pw) // 2] if pw else None, "power_limit_w": self.power_limit_w}


def bind_to_gpu_numa_node(index: int) -> str:
    """Host placement for the end-to-end leg, per rank: (1) run on the CPUs NVML reports as local to GPU `index` when the
    container's cpuset contains them, (2) ask the kernel to place this process's new pages - the pinned host buffers
    allocated afterwards - on the GPU's own NUMA node (set_mempolicy(MPOL_PREFERRED)), which also works when those
    CPUs are outside the cpuset.  Every step moves ~0.75 GB per rank between pinned host memory and the GPU; with the
    buffers of all ranks on one node the 8-GPU run is bound by that node's memory / inter-socket path."""
    notes = []
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        try:
            words = nv.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
            cpus = [64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1]
            allowed = [c for c in cpus if c in os.sched_getaffinity(0)]
            if allowed:
                os.sched_setaffinity(0, allowed)
                notes.append(f"{len(allowed)} cpus local to gpu {index}")
            else:
                notes.append(f"cpus local to gpu {index} outside cpuset")
        except Exception as e:  # noqa: BLE001
            notes.append(f"affinity unchanged ({type(e).__name__})")
        bus = nv.nvmlDeviceGetPciInfo(h).busId
        bus = bus.decode() if isinstance(bus, bytes) else bus
        node_file = Path("/sys/bus/pci/devices") / bus[-12:].lower() / "numa_node"
        node = int(node_file.read_text()) if node_file.exists() else -1
        if node >= 0:
            mask = (ctypes.c_ulong * 16)()
            mask[node // 64] = 1 << (node % 64)
            libc = ctypes.CDLL(None, use_errno=True)
            rc = libc.syscall(238, 1, ctypes.byref(mask), 1024)          # x86-64 set_mempolicy(MPOL_PREFERRED, mask, maxnode)
            notes.append(f"mempolicy prefer node {node}" if rc == 0 else f"mempolicy node {node} refused (errno {ctypes.get_errno()})")
        else:
            notes.append("numa node unknown")
    except Exception as e:  # noqa: BLE001
        notes.append(f"nvml unavailable ({type(e).__name__})")
    return "; ".join(notes)


# ---------------------------------------------------------------------------------------------
# the reference on the CPU: its own modules (oracle/_ref, byte-compiled by oracle/make_ref.py) in a process of
# their own - they call themselves `vsrlab`, like the drop-in - or, where those are absent, the oracle port.
# ---------------------------------------------------------------------------------------------
def reference_available() -> bool:
    from oracle import make_ref
    return make_ref.available()


def run_reference_process(blocks: int, frames: int, threads: int, steps: int = 1, warmup: int = 1, dump: str = "", seed: int = 0):
    cmd = [sys.executable, "-m", "oracle.ref_runner", "--blocks", str(blocks), "--frames", str(frames), "--threads", str(threads),
           "--steps", str(steps), "--warmup", str(warmup), "--seed", str(seed), "--height", str(LR_H), "--width", str(LR_W)]
    if dump:
        cmd += ["--dump", dump]
    out = subprocess.run(cmd, cwd=str(ROOT), check=True, capture_output=True, text=True).stdout
    return json.loads(out.strip().splitlines()[-1])


def oracle_port_sample(blocks: int, frames: int, threads: int, steps: int = 1, warmup: int = 1, seed: int = 0):
    """CPU restatement of the reference path (oracle/vsr_oracle.py) on `frames` frames of one 180x320 clip."""
    from oracle import vsr_oracle as O
    torch.set_num_threads(threads)
    sd = {k: v.detach().cpu() for k, v in build_model(blocks, "cpu").state_dict().items()}
    x = torch.rand(1, frames, 3, LR_H, LR_W, generator=torch.Generator().manual_seed(seed))
    with torch.no_grad():
        for _ in range(warmup):
            O.realbasicvsr(x[:, :2].clone(), sd)
        t0 = time.perf_counter()
        for _ in range(steps):
            sr, lq, ff, fb = O.realbasicvsr(x.clone(), sd, return_flows=True)
        dt = time.perf_counter() - t0
    n = steps * frames
    return {"frames": n, "seconds": dt, "frames_per_s": n / dt, "kind": "port", "threads": threads}, (sr, lq, ff, fb)


def run_reference(a):
    """--impl reference: the reference's CPU implementation on the host cores, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    total = a.steps + a.warmup
    frames = T_FRAMES if total <= 2 else max(3, min(T_FRAMES, 96 // max(total, 1)))      # whole run: a few minutes at most
    if reference_available():
        r = run_reference_process(a.blocks, frames, cores, steps=a.steps, warmup=a.warmup)
        what = "the reference's own modules (oracle/_ref, byte-compiled from the reference sources), torch CPU fp32"
    else:
        r, _ = oracle_port_sample(a.blocks, frames, cores, steps=a.steps, warmup=a.warmup)
        what = "oracle port (oracle/vsr_oracle.py; oracle/_ref was not built), torch CPU fp32"
    v = r["frames_per_s"]
    full = frames == T_FRAMES
    sample = (f"{frames} frames of one {LR_H}x{LR_W} clip per step" + ("" if full else " (a bounded sample of the 30-frame clip: "
              "frames/s is NOT extrapolated, the per-clip fixed work of a shorter clip is included)") + f"; {what}")
    cfg = workload_config(a, 1)
    cfg.update({"clips_per_gpu_per_step": 1, "frames_per_clip": frames, "precision": "fp32 (torch CPU, oneDNN)",
                "cuda_graph": "n/a (CPU)", "parallelism": f"{cores} host threads, no GPU", "l2": "n/a"})
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": r["seconds"] / max(a.steps, 1) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": r["kind"], "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def workload_config(a, clips):
    return {"workload": f"cfg3: Real-BasicVSR x4 inference, {T_FRAMES}-frame {LR_H}x{LR_W}->{4*LR_H}x{4*LR_W} clips, "
                        f"{a.blocks}/{a.blocks} blocks", "clips_per_gpu_per_step": clips, "frames_per_clip": T_FRAMES,
            "precision": "bf16 activations, fp32 accumulate", "cuda_graph": "whole forward captured once, replayed per step",
            "parallelism": f"clips sharded over {a.gpus} GPU(s), no collective",
            "l2": "per-step working set (GBs of activations) exceeds the 126 MB L2; no explicit flush"}


def dump_outputs(path: str, outputs: dict) -> None:
    """`outputs` name -> device tensor; see the module docstring for what is written."""
    import numpy as np
    out = Path(path)
    out.mkdir(parents=True, exist_ok=True)
    for name, t in outputs.items():
        if t.numel() > DUMP_ELEMS:
            idx = torch.randint(t.numel(), (DUMP_ELEMS,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(out / f"{name}.npy", t.float().cpu().numpy())


def emit(line: dict) -> None:
    """The ONE JSON line goes to the real stdout; everything else a library prints to stdout while the
    benchmark runs (e.g. NCCL's version banner) has been redirected to stderr by main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


# ---------------------------------------------------------------------------------------------
# parity at the benchmark's own shape + the CPU baseline (rank 0, N = 1)
# ---------------------------------------------------------------------------------------------
def parity_and_cpu_baseline(a, dev, frames: int = 6):
    from oracle import vsr_oracle as O
    from vsrlab_b200 import functional as VF
    import numpy as np
    cores = os.cpu_count() or 1
    if reference_available():
        with tempfile.TemporaryDirectory() as td:
            dump = str(Path(td) / "ref.npz")
            r = run_reference_process(a.blocks, frames, cores, steps=1, warmup=1, dump=dump)
            d = np.load(dump)
            sr_ref, lq_ref = torch.from_numpy(d["sr"]), torch.from_numpy(d["lq"])
            ff_ref, fb_ref = torch.from_numpy(d["flow_forward"]), torch.from_numpy(d["flow_backward"])
        what = "the reference's own modules (oracle/_ref)"
    else:
        r, (sr_ref, lq_ref, ff_ref, fb_ref) = oracle_port_sample(a.blocks, frames, cores)
        ff_ref, fb_ref = ff_ref.reshape(-1, 2, LR_H, LR_W), fb_ref.reshape(-1, 2, LR_H, LR_W)
        what = "oracle port (oracle/vsr_oracle.py)"
    model = build_model(a.blocks, dev).eval()                 # same seed, same constructor order => the reference's weights
    x = torch.rand(1, frames, 3, LR_H, LR_W, generator=torch.Generator().manual_seed(0))
    with torch.no_grad(), VF.precision("fp32"):
        xin = x.clone().to(dev)
        sr32, lq32 = model(xin)
        ff, fb = model.basicvsr.compute_flow(lq32)
    with torch.no_grad(), VF.precision("bf16"):
        sr16, _ = model(x.clone().to(dev))
        ff16, fb16 = model.basicvsr.compute_flow(lq32)
    hr = torch.rand(sr_ref.shape, generator=torch.Generator().manual_seed(9))
    par = {
        "against": what, "sample": f"{frames} frames of one {LR_H}x{LR_W} clip, {a.blocks}/{a.blocks} blocks, seed 0",
        "fp32_max_abs": max((sr32.cpu() - sr_ref).abs().max().item(), (lq32.cpu() - lq_ref).abs().max().item()),
        "bf16_psnr_delta_db": abs(O.psnr(sr16.cpu(), hr) - O.psnr(sr_ref, hr)),
        "bf16_psnr_vs_reference_db": O.psnr(sr16.cpu(), sr_ref),
        "flow_max_px": max((ff.cpu() - ff_ref).abs().max().item(), (fb.cpu() - fb_ref).abs().max().item()),
        "flow_max_px_bf16": max((ff16.cpu() - ff_ref).abs().max().item(), (fb16.cpu() - fb_ref).abs().max().item()),
        "gates": {"fp32_max_abs": 1e-4, "bf16_psnr_delta_db": 0.05, "flow_max_px": 1e-2},
    }
    par["ok"] = bool(par["fp32_max_abs"] <= 1e-4 and par["bf16_psnr_delta_db"] <= 0.05 and par["flow_max_px"] <= 1e-2
                     and par["flow_max_px_bf16"] <= 1e-2)
    base = {"value": r["frames_per_s"], "unit": UNIT, "cores": cores, "kind": r["kind"],
            "sample": f"{frames} frames of one {LR_H}x{LR_W} clip ({r['seconds']:.1f} s after one warm-up pass), full forward, {what}"}
    del model
    return par, base


# ---------------------------------------------------------------------------------------------
# BASELINE cfg4: the training step, on the reference's recipe (train.py:74,90-98; core/utils.py:147-151,235-240,270-280)
# ---------------------------------------------------------------------------------------------
def train_cfg4(a, dev, world, rank, local, steps: int = 8, warmup: int = 4, batch: int = 8, frames: int = 15, num_grad_acc: int = 4):
    import warnings
    import torch.distributed as dist
    import torch.nn.functional as F
    from vsrlab_b200 import functional as VF
    VF.set_precision(None)                                   # follow autocast, as train.py does
    model = build_model(a.blocks, dev, train_flow=True).train()
    net = torch.nn.parallel.DistributedDataParallel(model, device_ids=[local]) if world > 1 else model
    opt = torch.optim.Adam(net.parameters(), lr=1e-4, betas=(0.9, 0.99))
    sched = torch.optim.lr_scheduler.CosineAnnealingLR(opt, T_max=600000, eta_min=1e-7)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        scaler = torch.cuda.amp.GradScaler()
    g = torch.Generator().manual_seed(rank)
    lr = torch.rand(batch, frames, 3, 64, 64, generator=g).to(dev)
    hr = torch.rand(batch, frames, 3, 256, 256, generator=g).to(dev)

    def charbonnier(x, y):
        return torch.sqrt((x - y) ** 2 + 1e-9).mean()

    def micro_step(i):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ctx = torch.cuda.amp.autocast()
        with ctx:
            sr, lq = net(lr.clone())
            loss = charbonnier(sr, hr) + charbonnier(lq, F.interpolate(hr.flatten(0, 1), size=(64, 64), mode="bilinear").view_as(lq))
        scaler.scale(loss / num_grad_acc).backward()         # under DDP the gradient all-reduce fires here, every micro-step
        if (i + 1) % num_grad_acc == 0:
            scaler.unscale_(opt)
            torch.nn.utils.clip_grad_norm_(net.parameters(), 1.0)
            scaler.step(opt)
            scaler.update()
            sched.step()
            opt.zero_grad()
        return loss.detach()

    losses = [micro_step(i) for i in range(warmup)]
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    losses += [micro_step(i) for i in range(steps)]
    e1.record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    same = True
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        w0 = torch.cat([p.detach().flatten() for p in model.parameters()])
        ref = w0.clone()
        dist.broadcast(ref, 0)
        same = bool(torch.equal(w0, ref))
        flag = torch.tensor([1.0 if same else 0.0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        same = bool(flag.item() == 1.0)
    ms = t.item()
    tf = 3.0 * CFG4_FWD_GFLOP.get(a.blocks, float("nan")) * world / ms              # GFLOP / ms = TFLOP/s, whole job
    pk = peaks()
    out = {"workload": f"cfg4: Real-BasicVSR training micro-step, batch {batch}/GPU x {frames} frames 64x64 LR, {a.blocks}/{a.blocks} blocks, "
                       f"train_flow=true, fp16-requesting autocast + GradScaler, num_grad_acc={num_grad_acc}, Adam, clip 1.0",
           "n_gpus": world, "parallelism": "DDP, NCCL all-reduce on every micro-step (no no_sync, as the reference)" if world > 1 else "single GPU",
           "ms_per_step": ms, "clips_per_s": world * batch / (ms * 1e-3), "tflops": tf, "frac_of_sustained_peak": tf / world / pk["tf_sust"],
           "loss_first": float(losses[0]), "loss_last": float(losses[-1]), "replicas_identical": same,
           "grad_scale": float(scaler.get_scale()), "steps": steps, "warmup": warmup}
    from vsrlab_b200 import graphs as _graphs

    # after three eager calls the model's forward / backward replay from CUDA graphs inside this unchanged loop
    # (vsrlab_b200.graphs.training_forward), under DDP too
    out["fwd_bwd_graphed"] = _graphs.graphed_patterns(model) > 0
    if world == 1:
        # the opt-in whole-step graph (vsrlab_b200.graphs.GraphedTrainStep: forward + backward + clip + Adam in ONE CUDA graph,
        # bf16 autocast, no GradScaler): what the same kernels cost when the host is out of the way.  The eager number above
        # is bound by Python launch overhead and varies with the box's host (42 - 57 ms seen for the same 35 ms of kernels).
        from vsrlab_b200.graphs import GraphedTrainStep
        del opt
        opt_g = torch.optim.Adam(model.parameters(), lr=1e-4, betas=(0.9, 0.99), capturable=True)

        def loss_fn(outs, hr_):
            sr, lq = outs
            return charbonnier(sr, hr_) + charbonnier(lq, F.interpolate(hr_.flatten(0, 1), size=(64, 64), mode="bilinear").view_as(lq))
        gstep = GraphedTrainStep(model, opt_g, loss_fn, (lr, hr), clip_grad_norm=1.0, warmup=3)
        for _ in range(2):
            gstep(lr, hr)
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(steps):
            gl = gstep(lr, hr)
        g1.record()
        torch.cuda.synchronize()
        gms = g0.elapsed_time(g1) / steps
        out["cuda_graph"] = {"ms_per_step": gms, "clips_per_s": batch / (gms * 1e-3), "tflops": 3.0 * CFG4_FWD_GFLOP.get(a.blocks, float("nan")) / gms,
                             "loss": float(gl), "recipe": "GraphedTrainStep: bf16 autocast, Adam(capturable), clip 1.0, optimizer step every replay"}
        del gstep, opt_g
    del net, model
    VF.set_precision(a.precision)
    return out


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--clips", type=int, default=2, help="clips per GPU per step")
    ap.add_argument("--streams", type=int, default=1,
                    help="process the step's clips on this many CUDA streams (fills the fill/drain bubbles of the "
                         "sequential propagation kernels with another clip's work)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "fp32_ffma"],
                    help="bf16 (headline) | fp32 = fp32-accurate split-bf16 on the tensor cores | fp32_ffma = FFMA kernel")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the reference CPU run and the parity record")
    ap.add_argument("--no-extras", action="store_true", help="skip the blocks20 / train_cfg4 / e2e_narrow legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the sr / lq of the last timed step to DIR/<name>.npy (float32, see the module docstring)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs dumps the GPU path's outputs; it does not apply to --impl reference")
    a.warmup = max(a.warmup, 3) if a.impl != "reference" else a.warmup
    if a.impl == "reference":
        return run_reference(a)

    import torch.distributed as dist
    from vsrlab_b200 import functional as VF
    from vsrlab_b200 import ops, shard
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa = bind_to_gpu_numa_node(local)       # pinned host buffers are then placed next to the GPU's PCIe root
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    VF.set_precision(a.precision)
    model = build_model(a.blocks, dev).eval()
    clips = a.clips
    # clip sharding (SURVEY §8e): a global queue of world*clips clips per step, rank r takes clips r, r+W, ...
    my_clips = shard.shard_clips(world * clips, rank, world)
    gen = torch.Generator().manual_seed(1000 + rank)
    host_lr = torch.rand(len(my_clips), T_FRAMES, 3, LR_H, LR_W, generator=gen).pin_memory()
    lr_dev = host_lr.to(dev)
    work = torch.empty_like(lr_dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    side = [torch.cuda.Stream(device=dev) for _ in range(max(0, a.streams - 1))]

    def step(m=model):
        work.copy_(lr_dev)                       # the model refines its input in place (reference contract)
        if a.streams <= 1:
            with torch.no_grad():
                return m(work)
        # clips are independent: split them over the streams (same public call, one per stream)
        cur = torch.cuda.current_stream(dev)
        parts = work.chunk(a.streams, dim=0)
        outs = []
        for i, part in enumerate(parts):
            st = cur if i == 0 else side[i - 1]
            st.wait_stream(cur) if i else None
            with torch.cuda.stream(st), torch.no_grad():
                outs.append(m(part))
        for st in side:
            cur.wait_stream(st)
        return outs

    for _ in range(a.warmup):
        step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0, r0 = ops.launch_count(), VF.replayed_launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(a.steps - 1):
        step()
    out = step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = ops.launch_count() - l0 + VF.replayed_launches() - r0      # direct launches + kernel nodes of graph replays
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if a.dump_outputs and rank == 0:
        # dumped before anything else runs: `lq` is `work`, which the next step() overwrites in place
        sr, lq = [torch.cat(o) for o in zip(*out)] if a.streams > 1 else out
        dump_outputs(a.dump_outputs, {"sr": sr, "lq": lq})
        del sr, lq
    del out

    # ---- end to end: pinned host -> device -> model -> pinned host --------------------------
    # What a user of the drop-in does for a stream of clips: H2D of clip k+1 and D2H of clip k-1 run on a copy
    # stream while `model(lr)` of clip k runs on the compute stream.  Every step's H2D and D2H are inside the
    # timed region; the region ends when the last result has landed in pinned host memory.
    copy_stream = torch.cuda.Stream(device=dev)
    main_stream = torch.cuda.current_stream(dev)

    def e2e_leg(sr_dtype, out_kind):
        host_sr = [torch.empty(len(my_clips), T_FRAMES, 3, 4 * LR_H, 4 * LR_W, dtype=sr_dtype).pin_memory() for _ in range(2)]
        host_lq = [torch.empty_like(host_lr).pin_memory() for _ in range(2)]

        def e2e_run(n_steps):
            nxt = None
            with torch.cuda.stream(copy_stream):
                nxt = host_lr.to(dev, non_blocking=True)
                up = torch.cuda.Event()
                up.record(copy_stream)
            for k in range(n_steps):
                x, ready = nxt, up
                main_stream.wait_event(ready)
                x.record_stream(main_stream)
                with torch.no_grad(), VF.output_dtype(out_kind):
                    sr, lq = model(x)
                done = torch.cuda.Event()
                done.record(main_stream)
                with torch.cuda.stream(copy_stream):
                    if k + 1 < n_steps:                       # prefetch the next clip batch
                        nxt = host_lr.to(dev, non_blocking=True)
                        up = torch.cuda.Event()
                        up.record(copy_stream)
                    copy_stream.wait_event(done)
                    sr.record_stream(copy_stream)
                    lq.record_stream(copy_stream)
                    host_sr[k % 2].copy_(sr, non_blocking=True)
                    host_lq[k % 2].copy_(lq, non_blocking=True)
            main_stream.wait_stream(copy_stream)

        e2e_run(4)    # warm-up long enough for the caching allocator to own every output block the steady state needs
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        e2e_run(a.steps)
        f1.record()
        barrier()
        return f0.elapsed_time(f1), (host_sr[0].numel() * host_sr[0].element_size() + host_lq[0].numel() * 4)

    ms_e2e, d2h_bytes = e2e_leg(torch.float32, None)
    ms_e2e_u8, d2h_bytes_u8 = (0.0, 0) if a.no_extras else e2e_leg(torch.uint8, "uint8")

    # ---- per-kernel roofline: CUDA events around every launch of one more step --------------
    # The timed region replays a CUDA graph, so the per-launch pass must not be paced by the host either: a spin kernel
    # holds the stream while the step's launches and event records are queued, then the GPU runs them back to back and the
    # events see device-side durations (kernel + the GPU's own launch latency), not waits for Python.
    torch.cuda.synchronize()
    torch.cuda._sleep(int(0.15 * 1.9e9))
    ops.PROFILE = []
    step()
    torch.cuda.synchronize()
    prof, ops.PROFILE = ops.PROFILE, None
    fam, parts = {}, {}
    shapes = {}
    for kind, ev0, ev1, work_units, tag in prof:
        sec = ev0.elapsed_time(ev1) * 1e-3
        if "[" in kind:                                   # VSRB_PROFILE_SHAPES=1: per-shape table, family key without the shape
            q = shapes.setdefault(tag + " " + kind, [0.0, 0.0, 0])
            q[0] += sec
            q[1] += work_units
            q[2] += 1
            kind = kind.split("[")[0]
        d = fam.setdefault(kind, [0.0, 0.0, 0])
        d[0] += sec
        d[1] += work_units
        d[2] += 1
        if kind.startswith("conv_"):
            q = parts.setdefault(tag, [0.0, 0.0, 0])
            q[0] += sec
            q[1] += work_units
            q[2] += 1
    step_s_prof = sum(d[0] for d in fam.values())

    # ---- flow_warp on a working set far larger than L2 (256 feature maps, 1.9 GB in + 1.9 GB out), L2 flushed ----
    def warp_standalone():
        from vsrlab_b200._lib import BF16, PAD_ZEROS
        n = 256
        xw = torch.randn(n, LR_H, LR_W, 64, device=dev).to(torch.bfloat16)
        fw = (torch.rand(n, LR_H, LR_W, 2, device=dev) - 0.5) * 4.0
        ow = torch.empty_like(xw)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        ts = []
        for i in range(8):
            flush.zero_()
            w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            w0.record()
            ops.flow_warp(xw, fw, ow, n, LR_H, LR_W, 64, BF16, PAD_ZEROS)
            w1.record()
            torch.cuda.synchronize()
            if i >= 3:
                ts.append(w0.elapsed_time(w1) * 1e-3)
        return n * LR_H * LR_W * 264 / (sorted(ts)[len(ts) // 2]) / 1e9

    warp_big = warp_standalone() if rank == 0 else 0.0

    # ---- the model-file default 20/20 blocks (conf/train/model/basicvsr.yaml:2,5): "report both" (SURVEY §8) ----
    blocks20 = None
    if world == 1 and not a.no_extras and a.blocks != 20:
        VF.clear_caches()
        m20 = build_model(20, dev).eval()
        for _ in range(3):
            step(m20)
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        n20 = max(3, min(a.steps, 5))
        for _ in range(n20):
            step(m20)
        g1.record()
        torch.cuda.synchronize()
        ms20 = g0.elapsed_time(g1) / n20
        blocks20 = {"workload": "cfg3 with 20/20 blocks (model-file defaults)", "value": clips * T_FRAMES / (ms20 * 1e-3), "unit": UNIT,
                    "ms_per_step": ms20, "steps": n20, "conv_tflops": clips * 32772.49 / ms20}
        del m20
        VF.clear_caches()

    if ops.debug_status() != 0:                     # a kernel gave up on a pipeline barrier: the numbers would be meaningless
        raise RuntimeError("libvsrb200 reported a pipeline time-out during the benchmark")

    train = None
    if not a.no_extras:
        VF.clear_caches()
        torch.cuda.empty_cache()
        train = train_cfg4(a, dev, world, rank, local)
        VF.clear_caches()

    t = torch.tensor([ms, ms_e2e, ms_e2e_u8], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e, ms_e2e_u8 = t.tolist()
    frames_step, _ = shard.reduce_throughput(len(my_clips) * T_FRAMES, 0.0, dev)          # sum of frames over ranks
    value = frames_step * a.steps / (ms * 1e-3)
    e2e = frames_step * a.steps / (ms_e2e * 1e-3)
    affinities = [numa]
    if world > 1:
        affinities = [None] * world
        dist.all_gather_object(affinities, numa)
    if rank == 0:
        pk = peaks()
        traffic = {}
        tp = ROOT / "profiles" / "traffic.json"            # dram bytes per launch from `ncu --set full` captures
        if tp.exists():
            traffic = json.loads(tp.read_text())
        conv = fam.get("conv_tc") or fam.get("conv_tc_x3") or fam.get("conv_f32") or [1e-9, 0.0, 0]
        warp = fam.get("flow_warp", [1e-9, 0.0, 0])
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "fp32": "bf16x3 (split-bf16, fp32-accurate)", "fp32_ffma": "f32"}[a.precision],
            "data": "synthetic", "config": workload_config(a, clips),
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": host_lr.numel() * 4,
                    "d2h_bytes_per_step": d2h_bytes,
                    "pipeline": "copies on a second stream overlap the next step's compute; all copies are inside the timed region",
                    "host_affinity": affinities},
            "gpu_launches": launches,
            "clocks": sampler.summary(),
            "roofline": {"kernel": "conv_tc_kernel + conv_ring_kernel (tcgen05 implicit-GEMM convs, all launches of a step)",
                         "bound": "tensor",
                         "achieved": conv[1] / conv[0] / 1e12, "peak": pk["tf_sust"], "unit": "TFLOP/s",
                         "frac": conv[1] / conv[0] / 1e12 / pk["tf_sust"],
                         "traffic": (traffic.get("conv_tc") or {}).get("dram_bytes_per_launch"),
                         "traffic_source": traffic.get("conv_tc"),
                         "peak_source": pk["src"] + " (sustained)",
                         "launches_per_step": conv[2], "share_of_step": conv[0] / max(step_s_prof, 1e-9)},
            "roofline_warp": {"kernel": "flow_warp_kernel", "bound": "hbm", "achieved": warp[1] / warp[0] / 1e9, "peak": pk["hbm"],
                              "unit": "GB/s", "frac": warp[1] / warp[0] / 1e9 / pk["hbm"],
                              "traffic": (traffic.get("flow_warp") or {}).get("dram_bytes_per_launch"), "traffic_source": traffic.get("flow_warp"),
                              "launches_per_step": warp[2], "share_of_step": warp[0] / max(step_s_prof, 1e-9),
                              "note": "in-step calls move 30-60 MB each (L2 resident, launch-latency bound); `standalone` is the "
                                      "same kernel on 256 feature maps (3.9 GB moved, L2 flushed)",
                              "standalone": {"achieved": warp_big, "frac": warp_big / pk["hbm"], "unit": "GB/s"}},
            "kernel_time_share": {k: round(v[0] / max(step_s_prof, 1e-9), 4) for k, v in fam.items()},
            "conv_by_part": {k: {"ms": round(v[0] * 1e3, 3), "tflops": round(v[1] / v[0] / 1e12, 1), "launches": v[2]}
                             for k, v in parts.items()},
        }
        if ms_e2e_u8 > 0:
            line["e2e_narrow"] = {"value": frames_step * a.steps / (ms_e2e_u8 * 1e-3), "unit": UNIT,
                                  "h2d_bytes_per_step": host_lr.numel() * 4, "d2h_bytes_per_step": d2h_bytes_u8,
                                  "note": "opt-in vsrlab_b200.set_output_dtype('uint8'): sr leaves the last conv as the 8-bit values the "
                                          "reference's PNG dump stores (test.py:138-141); lq stays fp32.  The default (fp32 sr) is `e2e`."}
        if blocks20:
            line["blocks20"] = blocks20
        if train:
            line["train_cfg4"] = train
        if shapes:
            line["conv_by_shape"] = {k: {"ms": round(v[0] * 1e3, 3), "tflops": round(v[1] / v[0] / 1e12, 1), "launches": v[2]}
                                     for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][0])}
        if world == 1 and not a.no_cpu_baseline:
            VF.clear_caches()
            par, base = parity_and_cpu_baseline(a, dev)
            line["parity"], line["cpu_baseline"] = par, base
            if not par["ok"]:
                emit(line)
                raise RuntimeError(f"parity gate broken at the benchmark's shape: {par}")
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
