"""bench.py without a GPU: the reference arm (the CPU oracle port) prints one JSON line with the expected keys,
invalid arguments are refused, and dump_outputs (--dump-outputs) writes a result exactly, or a fixed sample of it."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "candidate sites/sec (tensor+inference)" and d["unit"] == "sites/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["vs_baseline"] is None
    assert d["config"]["workload"].startswith("cfg2_ont_r10_cdna_chr20")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_bad_arguments_refused():
    for extra in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, extra


def _chunk_result(n=400, seed=1):
    """a ChunkResult as Engine.wait returns it: the allele table has unwritten slots between candidates"""
    import numpy as np
    from clair3_rna_b200.engine import ChunkResult, ALT_DTYPE
    rng = np.random.default_rng(seed)
    alt_n = rng.integers(1, 6, n).astype(np.int32)
    alt_off = np.concatenate([[0], np.cumsum(alt_n.astype(np.int64) + 3)[:-1]])
    alt = np.zeros(int((alt_off + alt_n).max()), ALT_DTYPE)
    alt["count"] = -1
    for i in range(n):
        s = slice(alt_off[i], alt_off[i] + alt_n[i])
        alt["count"][s] = 10 * i + np.arange(alt_n[i])
        alt["order"][s] = 2 ** 32 - 1 - np.arange(alt_n[i])
    return ChunkResult(n_rows=4 * n, pos=(7 * np.arange(n) + 1).astype(np.int32),
                       depth=rng.integers(0, 99, n).astype(np.int32), probs=rng.random((n, 24), dtype=np.float32),
                       alt_off=alt_off, alt_n=alt_n, alt=alt, tensor=None, row_pos=None, row_counts=None, row_depth=None)


def _load(d):
    import numpy as np
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_writes_the_result_exactly(tmp_path):
    import numpy as np
    import bench
    r = _chunk_result()
    assert bench.dump_outputs(str(tmp_path), r) == (r.n_cand, r.n_cand)
    z = _load(str(tmp_path))
    assert sorted(z) == ["alt_base", "alt_count", "alt_kind", "alt_len", "alt_n", "alt_off", "alt_order", "alt_seq_off",
                         "depth", "pos", "probs"]
    assert all(a.dtype in (np.float32, np.float64) for a in z.values())
    assert z["probs"].dtype == np.float32 and np.array_equal(z["probs"], r.probs)
    for k in ("pos", "depth", "alt_off", "alt_n"):
        assert np.array_equal(z[k], getattr(r, k))
    want = np.concatenate([r.alt[o:o + k] for o, k in zip(r.alt_off, r.alt_n)])     # the unwritten slots left out
    for f in want.dtype.names:
        assert np.array_equal(z["alt_" + f], want[f])


def test_dump_outputs_samples_above_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import bench
    r = _chunk_result()
    monkeypatch.setattr(bench, "DUMP_LIMIT", 20000)
    k, n = bench.dump_outputs(str(tmp_path / "a"), r)
    bench.dump_outputs(str(tmp_path / "b"), r)
    a, b = _load(str(tmp_path / "a")), _load(str(tmp_path / "b"))
    assert 0 < k < n and sum(v.nbytes for v in a.values()) <= 20000
    assert all(np.array_equal(a[x], b[x]) for x in a)                                  # a fixed sample
    i = ((a["pos"] - 1) // 7).astype(np.int64)
    assert a["pos"].size == k and (np.diff(i) > 0).all() and np.array_equal(a["probs"], r.probs[i])
    assert np.array_equal(a["alt_count"], np.concatenate([10 * j + np.arange(r.alt_n[j]) for j in i]))
