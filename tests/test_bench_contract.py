"""bench.py: the reference arm runs on host cores only, so its JSON contract can be checked without a GPU (one line, the
keys a reader of the line expects, the metric/config of BASELINE.json, a bounded CPU sample); --dump-outputs writes the
result of the timed path in an order and sample that do not depend on the run."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "3000000", "--groups", "50000",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert d["impl"] == "reference" and d["metric"] == "groupby-agg rows/sec" and d["unit"] == "rows/s"
    assert base["metric"].startswith("groupby-agg rows/sec")
    for k in ("value", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["dtype"] == "int64" and d["data"] == "synthetic"
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["value"] > 1e5   # rows/s: the multi-threaded port does tens of millions per second even on a small box


def test_write_outputs_orders_by_key_and_samples_the_same_rows(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    rng = np.random.default_rng(4)
    keys = rng.permutation(1000)
    cols = {"key": torch.from_numpy(keys), "val": torch.from_numpy(keys * 3 - 7), "val_count": torch.from_numpy(keys % 5)}
    bench.write_outputs(str(tmp_path / "all"), cols)
    for name, exp in (("key", np.arange(1000)), ("val", np.arange(1000) * 3 - 7), ("val_count", np.arange(1000) % 5)):
        got = np.load(tmp_path / "all" / f"{name}.npy")
        assert got.dtype == np.float64
        np.testing.assert_array_equal(got, exp)
    # above the size cap: a seeded sample of the key-ordered rows, independent of the row order the library returned
    monkeypatch.setattr(bench, "DUMP_BYTES", 3 * 8 * 100)
    shuffled = rng.permutation(1000)
    bench.write_outputs(str(tmp_path / "a"), cols)
    bench.write_outputs(str(tmp_path / "b"), {k: v[shuffled] for k, v in cols.items()})
    for name in cols:
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert len(a) == 100
        np.testing.assert_array_equal(a, b)
    k = np.load(tmp_path / "a" / "key.npy")
    assert (np.diff(k) > 0).all()
    np.testing.assert_array_equal(np.load(tmp_path / "a" / "val.npy"), k * 3 - 7)


@pytest.mark.gpu
def test_dump_outputs_writes_the_groupby_result_of_the_timed_path(gpu_lib, tmp_path):
    import numpy as np

    from bodo_b200 import synth

    rows, groups = 3_000_000, 50_000
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--rows", str(rows), "--groups", str(groups), "--steps", "2",
                        "--warmup", "1", "--no-e2e", "--no-cpu", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    k, v = synth.numpy_fill(0, rows, groups, 1)
    present = np.bincount(k, minlength=groups) > 0
    np.testing.assert_array_equal(np.load(tmp_path / "key.npy"), np.arange(groups)[present])
    np.testing.assert_array_equal(np.load(tmp_path / "val.npy"), np.bincount(k, weights=v, minlength=groups)[present])
    np.testing.assert_array_equal(np.load(tmp_path / "val_count.npy"), np.bincount(k, minlength=groups)[present])
