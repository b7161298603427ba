"""CPU: the benchmark's reference arm runs without a GPU and prints the contract's JSON line; the CUDA arm
refuses to run without a device (no CPU fallback)."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[1]


def _run(args, **env):
    e = dict(os.environ, **env)
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, env=e,
                          timeout=600)


def test_reference_arm_json_line():
    p = _run(["--impl", "reference", "--config", "c3", "--steps", "1", "--warmup", "0", "--cpu-sample-stride", "16"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "ray_steps_per_s" and d["unit"] == "ray-steps/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["steps"] == 1
    assert d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "ray-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "config3" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_quietly():
    p = _run(["--impl", "reference", "--config", "c3", "--gpus", "2", "--steps", "1", "--warmup", "0"], RANK="1",
             WORLD_SIZE="2", LOCAL_RANK="1")
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_cuda_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    p = _run(["--config", "c3", "--steps", "1", "--warmup", "3"])
    assert p.returncode != 0
    assert "CUDA" in (p.stderr + p.stdout)


def test_steps_and_dump_outputs_are_checked(tmp_path):
    p = _run(["--impl", "reference", "--config", "c3", "--steps", "0"])
    assert p.returncode == 2 and "--steps must be at least 1" in p.stderr
    p = _run(["--impl", "reference", "--config", "c3", "--dump-outputs", str(tmp_path / "out")])
    assert p.returncode == 2 and "--dump-outputs" in p.stderr and not (tmp_path / "out").exists()


def test_dump_outputs_whole_map_and_seeded_sample(tmp_path):
    """--dump-outputs: a map within the budget is written whole; a larger one as the same seeded pixel sample of
    every plane, within the budget, identical from run to run."""
    import numpy as np
    import torch
    sys.path.insert(0, str(ROOT))
    import bench
    nf, ny, nx = 3, 40, 50
    image = torch.arange(2 * nf * ny * nx, dtype=torch.float64).reshape(2 * nf, ny, nx)
    assert bench.dump_outputs(image, nf, tmp_path / "whole") == ["tb", "vi"]
    np.testing.assert_array_equal(np.load(tmp_path / "whole" / "tb.npy"), image[:nf].numpy())
    np.testing.assert_array_equal(np.load(tmp_path / "whole" / "vi.npy"), image[nf:].numpy())
    budget = 20000
    for d in ("a", "b"):
        assert bench.dump_outputs(image, nf, tmp_path / d, max_bytes=budget) == ["pixel_index", "tb", "vi"]
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= budget
    files = {f.stem: np.load(f) for f in (tmp_path / "a").iterdir()}
    idx = files["pixel_index"].astype(np.int64)
    assert files["pixel_index"].dtype == np.float64 and len(np.unique(idx)) == len(idx) > 0
    flat = image.reshape(2 * nf, -1).numpy()
    np.testing.assert_array_equal(files["tb"], flat[:nf, idx])
    np.testing.assert_array_equal(files["vi"], flat[nf:, idx])
    for name, a in files.items():
        np.testing.assert_array_equal(np.load(tmp_path / "b" / f"{name}.npy"), a)


def test_reference_numpy_leg_runs_the_unmodified_reference():
    """bench.py's `extras.reference_numpy`: the UNMODIFIED reference package (baseline/_ref, installed by
    baseline/install_ref.sh) timed in a child process: ray_trace single-process and over a process pool, the CPU sampler."""
    import pytest
    sys.path.insert(0, str(ROOT))
    import bench
    if not (ROOT / "baseline" / "_ref" / "raytracingGRFF").is_dir():
        pytest.skip("the unmodified raytracingGRFF package is not part of the repository: install it into baseline/_ref "
                    "with `sh baseline/install_ref.sh <raytracingGRFF checkout>`")
    w = bench.workload("c3", 1)
    w["grid_n"] = 32
    d = bench.reference_numpy_timing(None, w, budget_rays=64, n_steps=12)
    assert "unavailable" not in d, d
    assert d["rays"] == 64 and d["ray_trace_single_process_ray_steps_per_s"] > 0
    assert d["ray_trace_process_pool_ray_steps_per_s"] > 0 and d["sampler_samples_per_s"] > 0
