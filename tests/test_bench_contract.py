"""bench.py's contract with the driver, as far as it can be exercised without a GPU: the reference arm prints exactly
ONE JSON line with the contract's keys, and both arms describe the workload with the same `config` object."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_arm_prints_one_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                          "--warmup", "0", "--ref_sample", "1", "--rec_iters", "2"], stdout=subprocess.PIPE,
                         stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    line = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in line, key
    assert line["impl"] == "reference" and line["unit"] == "images/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    assert line["e2e"] == {"value": line["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == line["value"] and 1 <= cb["cores"] and cb["cores_present"] >= 1
    assert "workload" in line["config"] and "model" not in line["config"]
    # the same object the GPU arm prints for this command line
    assert line["config"] == _bench_module().arm_config("mnist", 256, 10, 2, 1, "fp16")


def test_config_names_the_baseline_configuration():
    b = _bench_module()
    assert b.arm_config("mnist", 256, 10, 200, 1, "fp16")["baseline_config"] == "configs[1]"
    assert b.arm_config("f-mnist", 256, 10, 200, 1, "fp16")["baseline_config"] == "configs[2]"
    assert b.arm_config("celeba", 128, 10, 200, 1, "fp16")["baseline_config"] == "configs[3]"
    c5 = b.arm_config("mnist", 512, 10, 200, 8, "fp16")
    assert c5["baseline_config"] == "configs[4]" and c5["global_batch"] == 4096 and c5["per_gpu_batch"] == 512
    assert b.arm_config("mnist", 256, 10, 20, 1, "fp16")["baseline_config"] == "custom"
    assert "192 MiB" in c5["l2"]                       # the timing rule: say how L2 is flushed, in `config`


def test_steps_below_one_is_refused():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 2 and "--steps" in res.stderr and not res.stdout.strip()


def test_dump_output_is_float32_and_samples_large_outputs(tmp_path, monkeypatch):
    b = _bench_module()
    small = torch.arange(2 * 3 * 4, dtype=torch.float32).reshape(2, 3, 4)
    got = np.load(b.dump_output(str(tmp_path / "small"), "reconstructions", small))
    assert got.dtype == np.float32 and np.array_equal(got, small.numpy())
    assert os.listdir(tmp_path / "small") == ["reconstructions.npy"]
    # over the size limit: a fixed sample of whole rows, the same on every call, and the indices of those rows
    monkeypatch.setattr(b, "DUMP_BYTES", 10 * (3 * 4 * 4 + 8))
    big = torch.randn(50, 3, 4, generator=torch.Generator().manual_seed(0))
    for d in ("big1", "big2"):
        b.dump_output(str(tmp_path / d), "reconstructions", big)
    rec, rows = np.load(tmp_path / "big1" / "reconstructions.npy"), np.load(tmp_path / "big1" / "reconstructions_rows.npy")
    assert rec.dtype == np.float32 and rows.dtype == np.float64 and rec.shape == (10, 3, 4)
    assert np.all(np.diff(rows) > 0) and np.array_equal(rec, big.numpy()[rows.astype(np.int64)])
    assert np.array_equal(rec, np.load(tmp_path / "big2" / "reconstructions.npy"))
    assert np.array_equal(rows, np.load(tmp_path / "big2" / "reconstructions_rows.npy"))


@pytest.mark.gpu
def test_dump_outputs_is_what_the_timed_path_returned(tmp_path):
    """--dump-outputs writes the reconstructions of the last timed step: the same for the same arguments whatever --steps
    is, and the result of the projection of the benchmark's own inputs."""
    args = ["--gpus", "1", "--warmup", "1", "--batch", "8", "--rec_iters", "3", "--no_extra", "--no_profile",
            "--cpu_sample", "0"]
    for steps in (1, 3):
        res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args +
                             ["--steps", str(steps), "--dump-outputs", str(tmp_path / str(steps))],
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600, cwd=ROOT)
        assert res.returncode == 0, res.stderr[-2000:]
        assert json.loads(res.stdout)["steps"] == steps
        assert os.listdir(tmp_path / str(steps)) == ["reconstructions.npy"]
    once, thrice = np.load(tmp_path / "1" / "reconstructions.npy"), np.load(tmp_path / "3" / "reconstructions.npy")
    assert once.dtype == np.float32 and once.shape == (8, 28, 28, 1) and np.array_equal(once, thrice)
    wl = _bench_module().Workload("mnist", 8, 10, 3, "fp16", torch.device("cuda", 0), 0, 1)
    assert np.array_equal(once, wl.step().cpu().numpy())
    wl.close()
