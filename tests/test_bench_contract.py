"""bench.py's contract, the parts that run without a GPU: the reference arm (`--impl reference`) prints ONE JSON line with the
keys the driver reads, on the CPU restatement only; the product arm refuses to run without a GPU (no CPU fallback)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=ROOT, timeout=600)


def test_reference_arm_line_has_the_contract_keys():
    out = _run("--impl", "reference", "--config", "C1", "--steps", "2", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                       # exactly one JSON line on stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "aligned CCS reads/sec pileup+call+phase" and d["unit"] == "reads/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert abs(d["value"] - d["config"]["total_reads"] / (d["ms_per_step"] / 1e3)) <= 1e-6 * d["value"]
    assert d["config"]["workload"].startswith("C1") and d["config"]["total_reads"] == 5000 and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bad_arguments_are_refused():
    out = _run("--impl", "reference", "--steps", "0")
    assert out.returncode != 0 and "--steps must be at least 1" in out.stderr and not out.stdout.strip()
    out = _run("--impl", "reference", "--dump-outputs", "unused")
    assert out.returncode != 0 and "needs --impl ours" in out.stderr and not os.path.exists(os.path.join(ROOT, "unused"))


def test_dump_outputs_stay_within_the_limit_and_repeat(tmp_path):
    """--dump-outputs: small outputs are written whole; oversize ones become the same seeded row sample every time."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    small = {"col_counts": np.arange(24, dtype=np.float64).reshape(3, 8)}
    bench.dump_outputs(str(tmp_path / "s"), dict(small))
    assert np.array_equal(np.load(tmp_path / "s" / "col_counts.npy"), small["col_counts"])
    big = {"cooccurrence": np.arange(3000 * 3000, dtype=np.float64).reshape(3000, 3000), "keys": np.ones((5, 2))}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), dict(big))
        assert sum(f.stat().st_size for f in (tmp_path / d).iterdir()) <= bench.DUMP_LIMIT
    a, rows = np.load(tmp_path / "a" / "cooccurrence.npy"), np.load(tmp_path / "a" / "cooccurrence_rows.npy")
    assert np.array_equal(a, big["cooccurrence"][rows.astype(np.int64)])
    assert np.array_equal(a, np.load(tmp_path / "b" / "cooccurrence.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "keys.npy"), big["keys"])


def test_product_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    out = _run("--config", "C1", "--steps", "1", "--warmup", "0")
    assert out.returncode != 0 and "no CPU fallback" in out.stderr and not out.stdout.strip()
