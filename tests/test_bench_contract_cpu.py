"""bench.py's reference arm (the CPU leg the driver runs as `--impl reference`) prints ONE JSON line with the contract's
keys.  Runs the tiny workload so that it takes seconds; no GPU involved."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny", "--steps", "1",
                        "--warmup", "1", "--train-model", "tiny-qwen2-d128", "--train-seq", "64"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "e2e", "cpu_baseline", "gpu_launches"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["higher_is_better"] is True and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    hop = cb["reference_hop"]
    assert hop["decode"]["seconds"] > 0 and hop["prefill"]["payload_bytes"] > hop["decode"]["payload_bytes"]
    # the training half of BASELINE's metric travels on the same line
    tr = d["train"]
    assert tr["unit"] == "samples/s" and tr["value"] > 0 and tr["cpu_baseline"]["kind"] == "port" and tr["cpu_baseline"]["cores"] >= 1


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_dump_outputs_writes_float64_and_a_fixed_sample_over_the_limit(tmp_path, monkeypatch):
    bench = _bench()
    small, big = np.arange(12, dtype=np.int64).reshape(3, 4), np.arange(1000, dtype=np.int64).reshape(100, 10)
    bench.dump_outputs(str(tmp_path / "a"), {"small": small})
    got = np.load(tmp_path / "a" / "small.npy")
    assert got.dtype == np.float64 and np.array_equal(got, small)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4096 + 10 * big[0].nbytes)      # room for 10 rows of 10 float64
    for d in ("b", "c"):
        bench.dump_outputs(str(tmp_path / d), {"big": big})
    got = np.load(tmp_path / "b" / "big.npy")
    assert got.shape == (10, 10) and np.array_equal(got, np.load(tmp_path / "c" / "big.npy"))
    rows = got[:, 0].astype(np.int64) // 10
    assert np.all(np.diff(rows) > 0) and np.array_equal(got, big[rows])


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]], ids=["steps0", "dump_ref"])
def test_bench_rejects_arguments_it_cannot_honour(extra, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=120,
                       cwd=tmp_path)
    assert r.returncode == 2 and not r.stdout and not os.path.exists(tmp_path / "out"), r.stderr[-2000:]
