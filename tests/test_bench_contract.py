"""bench.py prints exactly one JSON line with the keys the driver depends on (CPU plumbing run)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "clocks"}


def run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_bench_json_contract_single_rank():
    d = run(["--backend", "gloo", "--model", "resnet18", "--batch-size", "2", "--steps", "2", "--warmup", "1"])
    assert REQUIRED <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["e2e"]["h2d_bytes_per_step"] == 2 * 3 * 224 * 224 * 4 + 2 * 8 and d["e2e"]["d2h_bytes_per_step"] == 4
    assert d["config"]["global_batch"] == 2 and d["gpu_launches"] > 0


def test_bench_two_ranks_native_emulation():
    d = run(["--gpus", "2", "--backend", "emu", "--model", "resnet18", "--batch-size", "2", "--steps", "2", "--warmup", "1",
             "--no-e2e"])
    assert d["n_gpus"] == 2 and d["config"]["global_batch"] == 4 and d["config"]["backend"] == "emu"
    assert d["gpu_launches"] == 2 * 2 * d["config"]["buckets"]      # one RS + one AG per bucket per step


def test_dump_outputs_are_float32_bounded_and_reproducible(tmp_path):
    import numpy as np
    args = ["--backend", "gloo", "--model", "resnet18", "--batch-size", "2", "--warmup", "1", "--no-e2e"]
    dumps = []
    for name, steps in (("a", 2), ("b", 2), ("c", 3)):
        # on the CPU even where a GPU is present: cuDNN's autotuner may pick other algorithms from run to run
        run(args + ["--steps", str(steps), "--dump-outputs", str(tmp_path / name)], env={"CUDA_VISIBLE_DEVICES": ""})
        files = sorted(os.listdir(tmp_path / name))
        assert files == ["loss.npy", "model_state.npy"]
        arrays = {f: np.load(tmp_path / name / f) for f in files}
        assert all(a.dtype == np.float32 for a in arrays.values())
        assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
        assert arrays["loss.npy"].shape == (1,) and np.isfinite(arrays["loss.npy"]).all()
        dumps.append(arrays)
    for f in dumps[0]:
        np.testing.assert_array_equal(dumps[0][f], dumps[1][f])       # same arguments: same inputs, same outputs
        assert not np.array_equal(dumps[0][f], dumps[2][f])           # one more timed step: another loss and state


def test_reference_arm_reports_unavailable_without_gpu():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"], cwd=ROOT,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["impl"] == "reference"
    import torch
    if not torch.cuda.is_available():
        assert "unavailable" in d
