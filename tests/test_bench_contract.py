"""bench.py's contract, as far as it can be checked without a GPU: the reference arm (the reference's CPU path, timed
on the host cores) prints ONE well-formed JSON line with the keys the driver reads; the product arm refuses to run
without a CUDA device instead of falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=600, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    res = _run("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "patchnce_fwd_bwd_patches_per_s" and d["unit"] == "patches/s"
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e["value"] == d["value"] and e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0


def test_dump_outputs_writes_the_last_step_the_same_way_every_run(tmp_path):
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        res = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path / run))
        assert res.returncode == 0, res.stderr[-2000:]
        dumps.append({f[:-4]: np.load(tmp_path / run / f) for f in sorted(os.listdir(tmp_path / run))})
    a, b = dumps
    assert sorted(a) == sorted(b) and sum(x.nbytes for x in a.values()) <= 64 << 20
    assert all(x.dtype in (np.float32, np.float64) for x in a.values())
    for name in a:
        np.testing.assert_array_equal(a[name], b[name])
    assert a["loss"].shape == (1,) and np.isfinite(a["loss"]).all()
    layers = [(64, 256, 256), (256, 64, 64), (256, 64, 64), (128, 128, 128), (64, 256, 256)]     # --layers b5
    for l, (c, h, w) in enumerate(layers):
        ids = a[f"ids_l{l}"]
        assert ids.shape == (256,) and ids.min() >= 0 and ids.max() < h * w and (ids == np.round(ids)).all()
        assert a[f"grad_l{l}"].shape == (4, c, 256) and np.abs(a[f"grad_l{l}"]).max() > 0     # --cpu-batch 4
        assert a[f"grad_l{l}_flat"].shape == (65536,)


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a CUDA device is present")
    res = _run("--steps", "1", "--warmup", "1")
    assert res.returncode != 0 and "no CPU fallback" in res.stderr
    assert not res.stdout.strip()
