"""bench.py's contract on the CPU: the reference arm (`--impl reference`) runs without a GPU, prints ONE JSON line with the keys
the driver reads, names the same config as the B200 arm, and says that each step is a bounded sample; the argument defaults
the round-end runs rely on (N = 1, K / W that finish in minutes, overlap decided by the world size)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, p.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line_on_cpu():
    j = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--records", "4000")
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in j, key
    assert j["impl"] == "reference" and j["gpu_launches"] == 0 and j["vs_baseline"] is None
    assert j["metric"] == "canonicalize+uniq records/sec" and j["unit"] == "records/s" and j["higher_is_better"] is True
    assert j["dtype"] == "u8" and j["data"] == "synthetic" and j["n_gpus"] == 1
    assert "config 2" in j["config"]["workload"] and "REDUCED" in j["config"]["workload"]      # --records: not the named config
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1 and j["cpu_baseline"]["value"] == j["value"]
    assert j["e2e"] == {"value": j["value"], "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert j["value"] > 0 and j["ms_per_step"] > 0


def test_dump_outputs_format(tmp_path, monkeypatch):
    """--dump-outputs on host tensors: a seeded sample of the records, exact hash halves, the canonical bytes of the first
    sampled records cut out of the aligned arena (record i at 32 * ((offsets[i] >> 5) + i)), at most DUMP_BASES of them."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_RECORDS", 700)
    monkeypatch.setattr(bench, "DUMP_BASES", 30000)
    rng = np.random.default_rng(5)
    n = 5000
    lens = rng.integers(1, 300, n)
    off = np.zeros(n + 1, np.int64); np.cumsum(lens, out=off[1:])
    seqs = [rng.integers(0, 256, L).astype(np.uint8) for L in lens]
    out = np.zeros(32 * ((int(off[-1]) >> 5) + n) + 32, np.uint8)
    for i, s in enumerate(seqs):
        a = 32 * ((off[i] >> 5) + i)
        out[a:a + len(s)] = s
    h = rng.integers(-2**63, 2**63 - 1, n, dtype=np.int64)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), "x_", n, {"length": torch.from_numpy(np.diff(off)), "hash": torch.from_numpy(h)},
                           canon=(torch.from_numpy(out), torch.from_numpy(off)))
    r = {f.name[2:-4]: np.load(f) for f in (tmp_path / "a").iterdir()}
    assert sorted(r) == ["canonical_bytes", "hash_hi", "hash_lo", "index", "length"]
    assert all(np.array_equal(v, np.load(tmp_path / "b" / ("x_" + k + ".npy"))) for k, v in r.items())   # the same sample
    idx = r["index"].astype(np.int64)
    assert len(idx) == 700 and np.all(np.diff(idx) > 0) and r["hash_hi"].dtype == np.float64
    u = (r["hash_hi"].astype(np.uint64) << np.uint64(32)) | r["hash_lo"].astype(np.uint64)
    assert np.array_equal(u.view(np.int64), h[idx]) and np.array_equal(r["length"], lens[idx])
    cb, ln = r["canonical_bytes"], r["length"].astype(np.int64)
    k = int((np.cumsum(ln) <= 30000).sum())
    assert cb.dtype == np.float32 and len(cb) == ln[:k].sum()
    assert np.array_equal(cb, np.concatenate([seqs[i] for i in idx[:k]]))


def test_argument_defaults():
    sys.path.insert(0, ROOT)
    import importlib
    bench = importlib.import_module("bench")
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert 'default="c2"' in src                                   # the default workload is the config BASELINE.json's metric is quoted on
    assert bench.WORKLOADS["c2"]["records"] == 10_000_000 and bench.WORKLOADS["c5"]["records"] == 12_500_000
    assert bench.WORKLOADS["c1"]["records"] == 1_000_000 and bench.WORKLOADS["c3"]["records"] == 5_000_000
    assert bench.WORKLOADS["c4"]["records"] == 200_000
