"""bench.py contract pieces that can be checked without a GPU."""
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]


def _run(*args, env=None):
    import os

    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=300, cwd=str(ROOT),
                          env={**os.environ, **(env or {})})


def test_reference_arm_prints_one_json_line_and_exits_zero():
    out = _run("--impl", "reference", "--gpus", "1", "--steps", "2", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-500:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    assert rec["impl"] == "reference" and ("unavailable" in rec or "value" in rec)
    # under torchrun only rank 0 speaks
    quiet = _run("--impl", "reference", "--gpus", "2", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert quiet.returncode == 0 and quiet.stdout.strip() == ""


def test_no_silent_cpu_fallback_and_launch_mismatch_is_reported():
    bad = _run("--gpus", "2")          # not launched under torchrun with 2 ranks
    assert bad.returncode != 0 and "WORLD_SIZE" in (bad.stderr + bad.stdout)
    if not torch.cuda.is_available():
        out = _run("--steps", "1", "--warmup", "1")
        assert out.returncode != 0 and "CUDA" in (out.stderr + out.stdout) and not out.stdout.strip().startswith("{")


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_steps_below_one_are_rejected():
    out = _run("--steps", "0")
    assert out.returncode != 0 and "--steps" in out.stderr and not out.stdout.strip()


def test_dump_outputs_writes_a_fixed_sample_within_budget(tmp_path, monkeypatch):
    """``--dump-outputs``: small parameter vectors are written whole, large ones as the same seeded sample every time; only float32 /
    float64 ``.npy`` files are written and a dump above the byte budget is refused."""
    import numpy as np
    import pytest

    bench = _bench_module()
    small = torch.arange(10, dtype=torch.float32)
    assert np.array_equal(bench.param_sample(small), small.numpy())
    monkeypatch.setattr(bench, "DUMP_PARAMS", 64)
    big = torch.randn(10_000)
    a, b = bench.param_sample(big), bench.param_sample(big.clone())
    assert a.dtype == np.float32 and 0 < a.size <= 64 and np.array_equal(a, b)
    assert np.isin(a, big.numpy()).all()
    bench.dump_outputs(str(tmp_path / "out"), {"global_params": a, "loss": np.ones(3)})
    assert np.array_equal(np.load(tmp_path / "out" / "global_params.npy"), a)
    assert np.load(tmp_path / "out" / "loss.npy").dtype == np.float64
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 8)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "over"), {"loss": np.ones(3)})
    assert not (tmp_path / "over").exists()


def test_ddp_config_follows_the_sharding_switch():
    """``--sharding``: plain DDP deletes ``fsdp_config`` (the launch scripts' choice), ``zero1`` / ``zero3`` keep it and name the scheme;
    ``auto`` shards the 7B config fully and leaves the small ones replicated; ``--global-batch`` reaches the trainer config."""
    import argparse

    bench = _bench_module()

    def cfg(model, sharding, impl="ours"):
        a = argparse.Namespace(model=model, precision="amp_bf16", attention="b200", sharding=sharding)
        return bench.ddp_cfg(a, impl, 8)

    c = cfg("mpt-125m", "auto")
    assert not c["llm_config"].get("fsdp_config") and c["kernels"]["param_sharding"] == "auto"
    c = cfg("mpt-7b", "auto")
    assert c["llm_config"]["fsdp_config"]["activation_checkpointing"] is True and c["kernels"]["param_sharding"] == "zero3"
    assert cfg("mpt-1b", "zero1")["kernels"]["param_sharding"] == "zero1" and cfg("mpt-1b", "zero1")["llm_config"].get("fsdp_config")
    assert not cfg("mpt-7b", "none")["llm_config"].get("fsdp_config")
    assert not cfg("mpt-7b", "zero3", impl="torch")["llm_config"].get("fsdp_config")      # the stock arm is always plain DDP
    bench.DDP_GLOBAL_BATCH = 32
    assert int(cfg("mpt-7b", "auto")["llm_config"]["global_train_batch_size"]) == 32
