"""bench.py's reference arm (`--impl reference`) runs without a GPU: it must print ONE JSON line with the contract's keys,
and the committed round profile must carry the keys the driver and the judge read."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["value"] > 0 and d["unit"] == "matches/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_committed_round_profile_has_the_contract_keys():
    d = json.load(open(os.path.join(ROOT, "profiles", "r1_bench_n1.json")))
    assert BASE_KEYS | {"clocks", "roofline"} <= set(d)
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-12
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["value"] < d["value"]
    assert d["dtype"] == "u8" and d["data"] == "synthetic" and d["scaling"] == "weak"


def test_dump_outputs_writes_float_arrays_within_the_limit(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    arrays = {"response": np.linspace(0.0, 1.0, 7), "cells": np.array([[0, 100, 255]], dtype=np.uint8),
              "passes": np.array([3, 2 ** 31 + 1], dtype=np.uint32), "ids": np.arange(4, dtype=np.int32)}
    bench.dump_outputs(str(tmp_path / "out"), arrays)
    assert sorted(os.listdir(tmp_path / "out")) == ["cells.npy", "ids.npy", "passes.npy", "response.npy"]
    for name, a in arrays.items():
        b = np.load(tmp_path / "out" / f"{name}.npy")
        assert b.dtype == (np.float32 if a.dtype == np.uint8 else np.float64) and np.array_equal(a, b)
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_LIMIT_BYTES // 8 + 1)})
    assert not (tmp_path / "big").exists()


@pytest.mark.gpu
def test_dumped_outputs_repeat_exactly_between_runs(tmp_path):
    """Two runs with the same arguments: the same inputs, so the same outputs, bit for bit (the sweep is exact)."""
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--candidates", "64",
                            "--no-graph", "--no-map", "--no-cpu", "--no-rows", "--no-seq", "--no-replay", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
        assert line["steps"] == 2 and line["gpu_launches"] > 0
        assert sorted(os.listdir(d)) == ["covariance.npy", "mean.npy", "response.npy"]
        dumps.append({n: np.load(d / f"{n}.npy") for n in ("response", "mean", "covariance")})
    a, b = dumps
    assert a["response"].shape == (64,) and a["mean"].shape == (64, 3) and a["covariance"].shape == (64, 3, 3)
    assert all(v.dtype == np.float64 for v in a.values()) and a["response"].max() > 0
    for n in a:
        assert np.array_equal(a[n], b[n]), n
