"""CPU: the contract of ``bench.py --impl reference`` (the driver runs it beside the GPU arm and divides the two lines):
one JSON line with the GPU arm's metric / unit / config, no transfers, the reference class on the host cores; ranks other
than 0 of a torchrun launch exit 0 without work or output; and the GPU arm refuses to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*argv, env=None, timeout=240):
    e = dict(os.environ)
    e.pop("RANK", None); e.pop("WORLD_SIZE", None); e.pop("LOCAL_RANK", None)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], cwd=ROOT, env=e, capture_output=True,
                          text=True, timeout=timeout)


def test_reference_arm_prints_one_line_with_the_gpu_arms_config():
    sys.path.insert(0, ROOT)
    import bench
    r = _bench("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == bench.UNIT and d["higher_is_better"] is True
    assert d["config"] == bench.workload(bench.B_PER_GPU)            # identical to the GPU arm's config (same_config)
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0 and d["vs_baseline"] is None
    assert d["e2e"] == {"value": d["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["value"] == d["value"] > 0 and cb["kind"] in ("reference", "port") and 1 <= cb["cores"] <= cb["usable_cpus"]
    assert "predictStream.py:154-157" in cb["sample"]
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "models.py")):
        assert cb["kind"] == "reference"                             # the unmodified class, not the restatement


def test_reference_arm_other_ranks_exit_quietly():
    r = _bench("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"},
               timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _bench("--steps", "1", timeout=120)
    assert r.returncode != 0 and "needs a GPU" in r.stderr


def test_argument_checks(tmp_path):
    r = _bench("--steps", "0", timeout=120)
    assert r.returncode == 2 and "--steps must be at least 1" in r.stderr
    r = _bench("--impl", "reference", "--dump-outputs", str(tmp_path), timeout=120)
    assert r.returncode == 2 and "--dump-outputs applies to the b200 arm" in r.stderr
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_is_reproducible(tmp_path):
    """--dump-outputs writes the last timed step's logits; two runs with the same arguments write the same array."""
    import numpy as np
    ys = []
    for i in range(2):
        out = tmp_path / str(i)
        r = _bench("--steps", "2", "--warmup", "3", "--batch", "256", "--sustained-seconds", "0", "--e2e-steps", "1",
                   "--parity-windows", "0", "--extra-steps", "0", "--no-cpu-baseline", "--dump-outputs", str(out), timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert d["steps"] == 2 and d["n_gpus"] == 1
        assert os.listdir(out) == ["logits.npy"]
        y = np.load(out / "logits.npy")
        assert y.dtype == np.float32 and y.shape == (256,) and np.isfinite(y).all()
        ys.append(y)
    assert np.array_equal(ys[0], ys[1])
