"""bench.py --dump-outputs: what the timed path returned, written so that two builds can be compared output for output."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

import bench

ROOT = Path(__file__).resolve().parents[1]


def test_dump_writes_small_outputs_whole_and_samples_large_ones(tmp_path):
    g = torch.Generator().manual_seed(3)
    small = torch.rand(1, 2, 3, 8, 8, generator=g)
    big = torch.rand(bench.DUMP_ELEMS + 1000, generator=g).to(torch.bfloat16)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"lq": small, "sr": big})
    lq, sr = np.load(tmp_path / "a" / "lq.npy"), np.load(tmp_path / "a" / "sr.npy")
    assert lq.dtype == sr.dtype == np.float32
    assert np.array_equal(lq, small.numpy())
    assert sr.shape == (bench.DUMP_ELEMS,)
    assert np.isin(sr, big.float().numpy()).all()
    assert np.array_equal(sr, np.load(tmp_path / "b" / "sr.npy"))          # the same seeded sample every time


@pytest.mark.gpu
def test_bench_steps_and_dumped_outputs(tmp_path):
    """--steps sets the timed work (kernel launches scale with it), and the last step's outputs do not depend on it."""
    runs = {}
    for steps in (1, 2):
        out = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "3", "--clips", "1",
                            "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                           cwd=str(tmp_path), capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        line = json.loads(r.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps
        runs[steps] = line, {n: np.load(out / f"{n}.npy") for n in ("sr", "lq")}
    assert runs[2][0]["gpu_launches"] == 2 * runs[1][0]["gpu_launches"] > 0
    total = 0
    for n in ("sr", "lq"):
        a, b = runs[1][1][n], runs[2][1][n]
        assert a.dtype == np.float32 and a.shape == (bench.DUMP_ELEMS,)  # 1 clip: 83 M sr / 5.2 M lq elements, sampled
        assert np.isfinite(a).all() and np.array_equal(a, b)
        total += a.nbytes
    assert total <= 64 << 20
