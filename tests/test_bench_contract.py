"""CPU: the reference arm of bench.py (``--impl reference``: the oracle port of the reference's eager CPU step, timed on the
host cores) runs without a GPU and prints ONE JSON line that carries the keys of the measurement contract.  Both arms write
the last timed step's arrays with ``--dump-outputs`` (the kernel arm's check needs the GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args, env=None):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600,
                       cwd=ROOT, env=dict(os.environ, **(env or {})))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    return json.loads(lines[0])


def _load_dump(d):
    arrays = {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}
    assert all(f.endswith(".npy") for f in os.listdir(d))
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    return arrays


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1", "--steps", "1",
                        "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "train images/sec" and d["unit"] == "img/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and abs(d["value"] - d["cpu_baseline"]["value"]) < 1e-9 and d["e2e"]["value"] == d["value"]
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0 and d["vs_baseline"] is None and "workload" in d["config"]


def test_reference_arm_dumps_the_last_step(tmp_path):
    d = _bench("--impl", "reference", "--config", "1", "--steps", "2", "--warmup", "0", "--dump-outputs", str(tmp_path),
               env=dict(CUDA_VISIBLE_DEVICES=""))
    a = _load_dump(tmp_path)
    assert sorted(a) == ["loss", "output", "params"]
    assert a["output"].shape == (8, 1000) and a["loss"].shape == ()
    assert a["params"].shape == (1 << 21,)                  # ViT-Ti has 5.7M parameters: a sample of 2M of them
    assert 0 < float(a["loss"]) < np.log(1000)              # the second step on the same batch is below chance
    assert d["steps"] == 2


@pytest.mark.gpu
def test_kernel_arm_dumps_the_same_arrays_for_the_same_arguments(cuda_device, tmp_path):
    """Seeded inputs, weights and DropPath masks: two runs differ only by the order of the GEMMs' split-K atomics (and an
    Adam update whose gradient sits at that rounding may flip sign, so the weights are held to their RMS error)."""
    args = ["--config", "1", "--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--no-e2e"]
    runs = []
    for k in range(2):
        d = _bench(*args, "--dump-outputs", str(tmp_path / str(k)), env=dict(VITK_BENCH_NO_SAMPLER="1"))
        assert d["steps"] == 3 and d["gpu_launches"] > 100
        runs.append(_load_dump(tmp_path / str(k)))
    a, b = runs
    assert sorted(a) == ["loss", "output", "params"] and a["output"].shape == (8, 1000)
    assert float(b["loss"]) == d["config"]["final_loss"]
    assert abs(float(a["loss"]) - float(b["loss"])) < 1e-3 * abs(float(b["loss"]))
    for k in ("output", "params"):
        x, y = a[k].astype(np.float64), b[k].astype(np.float64)
        assert np.sqrt(np.mean((x - y) ** 2) / np.mean(y ** 2)) < 1e-2, k
