"""bench.py contract checks that need no GPU: the reference arm (`--impl reference`) prints one JSON line with the keys the driver reads,
non-zero ranks of a torchrun launch stay silent, and the product arm refuses to run without CUDA instead of falling back."""
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]


def _run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, str(ROOT / "bench.py")] + args, capture_output=True, text=True, timeout=timeout, env=e, cwd=str(ROOT))


def test_reference_arm_prints_the_contract_line():
    res = _run(["--impl", "reference", "--steps", "12", "--warmup", "1"])
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    baseline = json.loads((ROOT / "BASELINE.json").read_text())
    assert line["impl"] == "reference" and baseline["metric"].startswith(line["metric"]) and line["unit"] == "Mpixels/s"
    for key in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["steps"] == 12
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None and line["data"] == "synthetic"
    assert "workload" in line["config"] and "model" not in line["config"]
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_is_silent_on_other_ranks():
    res = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert res.returncode == 0 and res.stdout.strip() == ""


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        return                                   # on a GPU box the driver runs the real thing
    res = _run(["--steps", "1", "--warmup", "3", "--no-e2e", "--no-cpu-baseline"], timeout=300)
    assert res.returncode != 0 and res.stdout.strip() == ""      # no JSON line from a CPU fallback: there is none


@pytest.mark.gpu
def test_dump_outputs_is_the_blur_of_the_last_step_whatever_the_step_count(tmp_path):
    """--steps sets the timed launches, and --dump-outputs writes the same fixed sample of the blurred image on every run: rows of the
    oracle's blur of the benchmark's seeded input."""
    import torch

    import oracle_lib as zo
    from gpu_utils import rel_err
    dumps = []
    for steps in (1, 4):
        d = tmp_path / f"steps{steps}"
        res = _run(["--steps", str(steps), "--warmup", "3", "--no-e2e", "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(d)])
        assert res.returncode == 0, res.stderr[-2000:]
        line = json.loads(res.stdout.strip().splitlines()[-1])
        assert line["steps"] == steps and line["gpu_launches"] == steps
        files = sorted(d.iterdir())
        assert [f.name for f in files] == ["gaussian_blur.npy", "gaussian_blur_rows.npy"]
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        dumps.append((np.load(files[0]), np.load(files[1])))
    (a, rows), (b, rows_b) = dumps
    assert a.shape == (256, 8192, 4) and a.dtype == np.float32 and rows.dtype == np.float64
    assert np.array_equal(a, b) and np.array_equal(rows, rows_b)
    rows = rows.astype(np.int64)
    assert np.array_equal(rows[:8], np.arange(8)) and np.array_equal(rows[-8:], np.arange(8184, 8192)) and np.all(np.diff(rows) > 0)
    # the benchmark's input (N = 1: rank 0's seed), blurred by the oracle in strips that hold every row a checked row reads
    x = torch.rand(8192, 8192, 4, device="cuda", dtype=torch.float32, generator=torch.Generator(device="cuda").manual_seed(2))
    taps = zo.gaussian_taps(2.25)
    for lo, hi, check in [(0, 15, range(0, 8)), (8177, 8192, range(8184, 8192))] + [(r - 7, r + 8, [r]) for r in rows[8:-8:40]]:
        want = zo.conv_separable(x[lo:hi].cpu().numpy(), taps, taps, "mirror")
        for r in check:
            assert rel_err(a[np.searchsorted(rows, r)], want[r - lo]) <= 1e-5, r
