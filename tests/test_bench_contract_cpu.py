"""bench.py's driver contract, on CPU: the reference arm prints ONE JSON line with the contract's keys (the unmodified reference
pipeline from the oracle/_ref snapshot when it is present, else the oracle port), our arm refuses to run without a CUDA device
(there is no CPU fallback), and both arms describe the workload with the same `config` object."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, timeout=900):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS=os.environ.get("OMP_NUM_THREADS", "8"))
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=env, timeout=timeout,
                          cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "scene-steps/s" and d["n_gpus"] == 1
    assert d["metric"] == "6-view 224x400 denoising-steps/sec" and d["value"] > 0 and d["ms_per_step"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["gpu_launches"] == 0
    # the workload description both arms print (the driver compares the `config` objects)
    cfg = d["config"]
    assert cfg["workload"].startswith("configs[2]: 6-view 224x400, full cond") and cfg["latent_hw"] == [28, 50]
    assert cfg["sharding"].startswith("scene-per-GPU replicas") and cfg["scheduler"] == "ddim"


def test_dump_outputs_caps_the_size_with_a_fixed_sample(tmp_path, monkeypatch):
    """--dump-outputs: float32 .npy files; over the size limit, the same seeded sample of positions on every run."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    x = torch.arange(1000, dtype=torch.float64).reshape(10, 100)
    bench.dump_outputs(str(tmp_path / "full"), {"latents": x})
    full = np.load(tmp_path / "full" / "latents.npy")
    assert full.dtype == np.float32 and full.shape == (10, 100) and (full == x.numpy()).all()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 400)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"latents": x})
    a, b = np.load(tmp_path / "a" / "latents.npy"), np.load(tmp_path / "b" / "latents.npy")
    assert a.nbytes <= 400 and a.size == 100 and (a == b).all()
    assert (np.diff(a) > 0).all() and np.isin(a, full).all()


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine WITHOUT a CUDA device")
def test_our_arm_has_no_cpu_fallback():
    r = _run("--steps", "1", "--warmup", "1", timeout=300)
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout)
