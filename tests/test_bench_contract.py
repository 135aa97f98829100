"""bench.py contract pieces, most of them checked without a GPU: the reference arm (`--impl reference`, the oracle port on the host
cores) prints one JSON line with the agreed keys, non-zero ranks print nothing, the GPU arm refuses to run without CUDA
instead of falling back to the CPU, and --dump-outputs writes the timed path's result in a form two builds can be compared by."""
import importlib
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _bench(monkeypatch):
    b = importlib.import_module("bench")
    monkeypatch.setenv("DFGPU_Q3_SF", "0.2")          # a small instance of the same Q3 workload keeps the CPU arm to seconds here
    return b


def test_reference_arm_prints_the_contract_line(monkeypatch, capsys):
    b = _bench(monkeypatch)
    args = types.SimpleNamespace(gpus=1, steps=2, warmup=1, impl="reference")
    b.run_reference(args, 0, 1)
    out = [l for l in capsys.readouterr().out.splitlines() if l.startswith("{")]
    assert len(out) == 1
    d = json.loads(out[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "rows/s" and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["metric"] == b.METRIC
    assert d["config"]["workload"].startswith("C4 TPC-H Q3-shaped pipeline, SF0.2") and d["config"]["fingerprint"][0] > 1000
    assert d["cpu_baseline"]["runs"] == 2 and d["cpu_baseline"]["best_rows_per_s"] >= d["cpu_baseline"]["median_rows_per_s"] * 0.999


def test_usable_threads_respects_affinity_and_quota(monkeypatch):
    b = importlib.import_module("bench")
    n = b.usable_threads()
    assert 1 <= n <= len(os.sched_getaffinity(0))
    assert b.cpu_sample_sf(100.0) in (100.0, 50.0, 25.0, 12.5, 6.25, 3.125, 1.5625, 0.78125)


def test_reference_arm_is_rank0_only(monkeypatch, capsys):
    b = _bench(monkeypatch)
    args = types.SimpleNamespace(gpus=2, steps=1, warmup=0, impl="reference")
    b.run_reference(args, 1, 2)
    assert capsys.readouterr().out.strip() == ""


@pytest.mark.skipif(os.path.exists("/dev/nvidiactl"), reason="needs a machine WITHOUT a GPU")
def test_gpu_arm_fails_loudly_without_cuda():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0
    assert "no CPU fallback" in (r.stderr + r.stdout) or "CUDA" in (r.stderr + r.stdout)
    assert not any(l.startswith("{") and '"value"' in l for l in r.stdout.splitlines())


class _HostBatch:
    """what dump_outputs reads from a result batch: column_numpy(i) -> (values, valid or None)"""

    def __init__(self, cols):
        self.cols = cols

    def column_numpy(self, i):
        return self.cols[i], None


def _q3_like_batches(n, seed=3):
    rng = np.random.default_rng(seed)
    key = rng.permutation(4 * n)[:n].astype(np.int64) + 1
    cols = [key, (key % 2500 + 8000).astype(np.int32), np.zeros(n, np.int32), rng.integers(0, 7_000_000_000, n).astype(np.int64)]
    cut = n // 3
    return [_HostBatch([c[:cut] for c in cols]), _HostBatch([c[cut:] for c in cols])], cols


def test_dump_outputs_is_sorted_exact_and_independent_of_batch_order(tmp_path):
    b = importlib.import_module("bench")
    batches, cols = _q3_like_batches(5000)
    assert b.dump_outputs(batches, str(tmp_path / "a")) == (5000, 1)
    assert b.dump_outputs(batches[::-1], str(tmp_path / "b")) == (5000, 1)
    order = np.argsort(cols[0])
    for name, c in zip(b.RESULT_COLUMNS, cols):
        a, r = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype == np.float64 and np.array_equal(a, r)
        assert np.array_equal(a.astype(np.int64), c[order])


def test_dump_outputs_samples_the_same_groups_under_the_size_cap(tmp_path):
    b = importlib.import_module("bench")
    batches, cols = _q3_like_batches(20000)
    cap = 200_000                                   # 20000 rows x 4 columns x 8 B = 640 kB: needs a sample
    kept, m = b.dump_outputs(batches, str(tmp_path / "a"), max_bytes=cap)
    assert m > 1 and 0 < kept < 20000
    assert sum(os.path.getsize(tmp_path / "a" / f"{name}.npy") for name in b.RESULT_COLUMNS) <= cap
    assert b.dump_outputs(batches[::-1], str(tmp_path / "b"), max_bytes=cap) == (kept, m)
    key = np.load(tmp_path / "a" / "l_orderkey.npy").astype(np.int64)
    with np.errstate(over="ignore"):
        expect = np.sort(cols[0][b.splitmix64_np(b.DUMP_SEED, cols[0].astype(np.uint64)) % np.uint64(m) == 0])
    assert np.array_equal(key, expect)
    for name in b.RESULT_COLUMNS:
        assert np.array_equal(np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy"))


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_steps_result(tmp_path):
    """a small instance of the timed Q3 path: the dumped rows are the result the fingerprint (checked against the CPU restatement of the
    same tables) describes, and --steps sets the number of timed steps"""
    out = tmp_path / "dump"
    env = dict(os.environ, DFGPU_Q3_SF="0.05")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1", "--no-secondary", "--e2e-steps", "1",
                        "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["cpu_baseline"]["same_tables_as_gpu"]
    fp = d["config"]["fingerprint"]
    arrs = [np.load(out / f"{name}.npy") for name in ("l_orderkey", "o_orderdate", "o_shippriority", "revenue")]
    assert all(a.dtype == np.float64 and len(a) == fp[0] for a in arrs) and fp[0] == d["config"]["stages"]["groups"] > 1000
    assert [int(a.astype(np.int64).sum()) % (1 << 64) for a in arrs] == fp[1:]
    assert np.all(np.diff(arrs[0]) > 0)
