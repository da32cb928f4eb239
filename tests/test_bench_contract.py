"""The driver-facing contract of ``bench.py --impl reference`` (the CPU arm runs without a GPU): ONE JSON line
with the keys the driver parses, on a corpus small enough for the CPU suite.  The b200 arm's line is checked on
the GPU box by the driver itself; the keys both arms share are listed once here."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]

SHARED_KEYS = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
               "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e")


def test_reference_arm_prints_one_contract_line():
    proc = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--movies", "3000",
                           "--vocab", "5000", "--steps", "2", "--warmup", "1"],
                          capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert proc.returncode == 0, proc.stderr[-2000:]
    lines = [l for l in proc.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in SHARED_KEYS:
        assert k in d, k
    assert d["metric"] == "hybrid queries/sec" and d["unit"] == "queries/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 2 and d["warmup"] == 1 and d["n_gpus"] == 1
    assert d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["workload"].startswith("configs[3]") and d["config"]["movies"] == 3000
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e2e = d["e2e"]
    assert e2e == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # value = queries of the timed steps / their time
    assert abs(d["value"] * d["ms_per_step"] / 1e3 - int(cb["sample"].split()[0])) < 1e-6 * max(1, d["value"])


def test_dump_outputs_writes_float_arrays_and_samples_above_the_cap(tmp_path, monkeypatch):
    import bench
    rng = np.random.default_rng(1)
    arrays = {"id": rng.integers(10, 2 ** 40, (300, 10)), "score": rng.standard_normal((300, 10)),
              "dist": rng.standard_normal((300, 10)).astype(np.float32), "count": rng.integers(0, 11, 300).astype(np.int32)}
    bench.dump_outputs(tmp_path / "all", arrays)
    for name, a in arrays.items():
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == (np.float32 if a.dtype == np.float32 else np.float64)
        assert (got == a).all()
    assert not (tmp_path / "all" / "query_index.npy").exists()
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 8000)
    for d in ("s1", "s2"):
        bench.dump_outputs(tmp_path / d, arrays)
    rows = np.load(tmp_path / "s1" / "query_index.npy").astype(np.int64)
    assert 0 < len(rows) < 300 and (np.diff(rows) > 0).all()
    assert sum((tmp_path / "s1" / f"{n}.npy").stat().st_size for n in list(arrays) + ["query_index"]) < 8000 + 5 * 256
    for name, a in arrays.items():
        got = np.load(tmp_path / "s1" / f"{name}.npy")
        assert (got == a[rows]).all() and (got == np.load(tmp_path / "s2" / f"{name}.npy")).all()
    with pytest.raises(ValueError):
        bench.dump_outputs(tmp_path / "big", {"id": np.array([2 ** 53 + 1], np.int64)})
