"""bench.py contract pieces: the `--impl reference` arm (CPU oracle port on the host cores) prints one JSON line with the keys a
consumer of the line reads; under a multi-rank launch only rank 0 prints; the GPU arm refuses to run without a device; on a GPU,
`--dump-outputs` writes the timed path's last outputs, identical from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASELINE = json.load(open(os.path.join(ROOT, "BASELINE.json"))) if os.path.exists(os.path.join(ROOT, "BASELINE.json")) else None


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, env=e, cwd=ROOT)


def test_reference_arm_line():
    out = _run(["--impl", "reference", "--gpus", "1", "--steps", "32", "--warmup", "2"])
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
                "config", "cpu_baseline", "e2e"):
        assert key in line, key
    assert line["impl"] == "reference" and line["higher_is_better"] is True and line["vs_baseline"] is None and line["steps"] == 32
    if BASELINE:
        assert line["metric"] == BASELINE["metric"]
    assert line["value"] > 1e5 and line["unit"] == "env-steps/s"
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == (os.cpu_count() or 1) and cb["value"] == line["value"] and "32 steps" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_reference_arm_other_ranks_stay_silent():
    out = _run(["--impl", "reference", "--gpus", "2", "--steps", "8", "--warmup", "1"], env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_gpu_arm_refuses_without_a_device():
    import torch

    if torch.cuda.is_available():
        return
    out = _run(["--steps", "2", "--warmup", "1"])
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path_are_reproducible(tmp_path):
    """--dump-outputs writes the last of the --steps timed steps as float32 .npy files; the same arguments give the same arrays"""
    lines = []
    for run in ("a", "b"):
        out = _run(["--gpus", "1", "--steps", "37", "--warmup", "3", "--envs-per-gpu", "4096", "--no-extra", "--no-cpu-baseline",
                    "--dump-outputs", str(tmp_path / run)])
        assert out.returncode == 0, out.stderr[-2000:]
        lines.append(json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1]))
    assert lines[0]["steps"] == 37 and lines[0]["gpu_launches"] == 2  # 32 + 5 fused steps
    shapes = {"obs": (4096, 14), "reference": (4096, 2), "reward": (4096,), "terminated": (4096,)}
    assert sorted(os.listdir(tmp_path / "a")) == sorted(f"{k}.npy" for k in shapes)
    for name, shape in shapes.items():
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all()
        assert np.array_equal(a, b), name
