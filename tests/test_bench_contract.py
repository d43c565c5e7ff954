"""bench.py prints exactly ONE JSON line on stdout with the keys the driver reads -- for the reference arm (CPU,
checked here without a GPU) and for our arm (GPU, small step)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(*args, timeout=900, env=None):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                       timeout=timeout, cwd=ROOT, env=None if env is None else {**os.environ, **env})
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                       # nothing but the JSON line on stdout
    return json.loads(lines[0])


@pytest.mark.parametrize("arm", ["port"])
def test_reference_arm_line(arm):
    """`--impl reference` without a staged reference checkout: the census on the oracle port (kind "port");
    OMP_NUM_THREADS=1 as torchrun exports it must not shrink the thread count."""
    d = _run("--impl", "reference", "--steps", "1", "--warmup", "0", env={"HAIRFAST_CPU_ARM": arm,
                                                                          "OMP_NUM_THREADS": "1"})
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "hair_swap_triples_per_sec" and d["unit"] == "triples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["e2e"] == {"value": d["value"], "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == arm and cb["cores"] > 1 and cb["value"] == d["value"] and "sample" in cb
    assert "workload" in d["config"] and set(cb["per_call_s"]) >= {"gen_full", "e4e", "seg_1024"}


def test_dump_outputs_budget_and_sample(tmp_path):
    """bench.dump_outputs: nested outputs by name, float32, small arrays whole, large ones as the same seeded sample
    on every call, 64 MB in all."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    outs = {"small": torch.arange(12, dtype=torch.int64).reshape(3, 4),
            "nested": (torch.randn(40_000_000, generator=torch.Generator().manual_seed(0)), None,
                       [torch.ones(2, 2, dtype=torch.bfloat16)]),
            "absent": None}
    for d in ("a", "b"):
        bench.dump_outputs(outs, str(tmp_path / d))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == ["nested.0.npy", "nested.2.0.npy", "small.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= bench.DUMP_BYTES
    small = np.load(tmp_path / "a" / "small.npy")
    assert small.dtype == np.float32 and np.array_equal(small, np.arange(12).reshape(3, 4))
    big = np.load(tmp_path / "a" / "nested.0.npy")
    assert big.dtype == np.float32 and 0 < big.size < 40_000_000
    assert np.isin(big, outs["nested"][0].numpy()).all()
    for n in names:
        assert np.array_equal(np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)), n


@pytest.mark.gpu
def test_our_arm_line(tmp_path):
    d = _run("--steps", "2", "--warmup", "3", "--triples", "2", "--no-extras", "--dump-outputs", str(tmp_path))
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 3 and d["scaling"] == "weak"
    assert d["value"] > 0 and abs(d["value"] - 2 / (d["ms_per_step"] * 1e-3)) < 1e-2 * d["value"]
    e = d["e2e"]
    assert e["value"] > 0 and e["unit"] == "triples/s" and e["h2d_bytes_per_step"] > 0
    assert e["d2h_bytes_per_step"] == 2 * 3 * 1024 * 1024 * 4
    assert d["gpu_launches"] > 100                      # our kernels ran inside the timed region
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    r = d["roofline"]
    assert r["bound"] == "tensor" and r["unit"] == "TFLOP/s" and 0 < r["frac"] <= 1.05
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-3 and "traffic" in r
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] > 0
    assert d["config"]["triples_per_step_per_gpu"] == 2 and "workload" in d["config"]
    assert d["latency_T1"]["latency_ms_per_triple"] > 0
    dumped = {n: os.path.getsize(tmp_path / n) for n in os.listdir(tmp_path)}
    assert {"e4e_a.npy", "fse.0.npy", "gen7_5_8.0.npy", "pp_res.npy", "seg_1024_b.npy"} <= set(dumped)
    assert sum(dumped.values()) <= 64 << 20


@pytest.mark.gpu
def test_two_gpu_outputs_equal_single_gpu():
    """SURVEY 8d config 5: per-triple outputs of the N-GPU run equal the 1-GPU computation bit for bit (checked inside
    bench.py after the timed region; needs two devices)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", "29533", os.path.join(ROOT, "bench.py"), "--gpus", "2", "--steps", "1",
           "--warmup", "3", "--triples", "2", "--no-extras", "--no-cpu-baseline"]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([l for l in p.stdout.splitlines() if l.strip().startswith("{")][-1])
    assert d["n_gpus"] == 2 and d["shard_output_equality"]["bit_identical_to_single_gpu"] is True
