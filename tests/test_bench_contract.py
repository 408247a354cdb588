"""bench.py contract checks: the reference arm (`--impl reference`, the oracle's Block-WAND port on host threads) prints
one JSON line with the keys a caller of the benchmark reads, the product arm refuses to run without CUDA (no CPU
fallback), and `--dump-outputs` writes the rows of the last timed step (checked against the oracle on a GPU)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TINY = ["--docs-per-segment", "20000", "--nq", "8", "--steps", "1", "--warmup", "3"]


def _bench(args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_reference_arm_prints_the_contract_line():
    r = _bench(["--impl", "reference"] + TINY)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "queries/sec" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["warmup"] >= 3 and d["value"] > 0
    assert d["config"]["workload"] == "or5_top100_100M_8seg"
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_product_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = _bench(TINY)
    assert r.returncode != 0 or not any(ln.startswith("{") for ln in r.stdout.splitlines())
    assert "NVIDIA" in r.stderr or "CUDA" in r.stderr or "no CPU fallback" in r.stderr


def test_steps_and_dump_outputs_arguments_are_checked():
    r = _bench(["--steps", "0"] + TINY[:-4])
    assert r.returncode != 0 and "--steps" in r.stderr
    r = _bench(["--impl", "reference", "--dump-outputs", "unused"] + TINY)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr


def test_dump_outputs_zeroes_padding_and_samples_past_the_limit(tmp_path, monkeypatch):
    import numpy as np

    import bench
    rng = np.random.default_rng(5)
    nq, k = 50, 7
    rows = (rng.random((nq, k), dtype=np.float32) + 1, rng.integers(1, 9, (nq, k)).astype(np.uint32),
            rng.integers(1, 2**32, (nq, k), dtype=np.uint64).astype(np.uint32), rng.integers(0, 9, nq).astype(np.uint32))
    bench.dump_outputs(str(tmp_path / "all"), rows, 1)
    d = {n: np.load(tmp_path / "all" / (n + ".npy")) for n in ("scores", "segment_ords", "docs", "counts", "queries")}
    assert d["scores"].dtype == np.float32 and all(d[n].dtype == np.float64 for n in ("segment_ords", "docs", "counts", "queries"))
    assert (d["queries"] == np.arange(nq)).all() and (d["counts"] == rows[3]).all()
    for q in range(nq):
        n = min(int(rows[3][q]), k)
        assert (d["scores"][q, :n] == rows[0][q, :n]).all() and (d["docs"][q, :n] == rows[2][q, :n]).all()
        assert (d["segment_ords"][q, :n] == rows[1][q, :n]).all()
        assert not d["scores"][q, n:].any() and not d["docs"][q, n:].any() and not d["segment_ords"][q, n:].any()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 10 * (k * 20 + 16))
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), rows, 1)
    qa, qb = (np.load(tmp_path / name / "queries.npy") for name in ("a", "b"))
    assert len(qa) == 10 and (qa == qb).all() and (np.diff(qa) > 0).all()
    sa = np.load(tmp_path / "a" / "scores.npy")
    assert sa.shape == (10, k) and (sa[:, 0] == np.where(rows[3] > 0, rows[0][:, 0], 0)[qa.astype(int)]).all()
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 10 * (k * 20 + 16) + 5 * 128


@pytest.mark.gpu
def test_dump_outputs_are_the_last_timed_steps_rows(tmp_path):
    """Two runs with the same arguments write the same arrays, and they are the oracle's rows for the batch of the last timed
    step (steps 3 + 3 cycle through batches 0..3, 0, 1: batch 1)."""
    import numpy as np

    import bench
    from oracle import tq_oracle as O
    args = ["--docs-per-segment", "20000", "--nq", "8", "--steps", "3", "--warmup", "3", "--no-cpu-baseline", "--parity-queries", "0"]
    for name in ("a", "b"):
        r = _bench(args + ["--dump-outputs", str(tmp_path / name)])
        assert r.returncode == 0, r.stderr[-2000:]
    names = ("scores", "segment_ords", "docs", "counts", "queries")
    a = {n: np.load(tmp_path / "a" / (n + ".npy")) for n in names}
    b = {n: np.load(tmp_path / "b" / (n + ".npy")) for n in names}
    for n in names:
        assert a[n].tobytes() == b[n].tobytes(), n
    wl = dict(bench.WORKLOADS["or5_top100_100M_8seg"], docs_per_segment=20000)
    seed = 0x7A6E7469
    dens, batches = bench.build_query_plan(wl, 8, 4, seed)
    shard = bench.make_shard(wl, dens, 0, 1, seed)
    oi = O.OracleIndex()
    shard.register(oi)
    ref = oi.search_batch(bench.marshal(shard, batches[1]), mode=0)
    assert (a["queries"] == np.arange(8)).all() and (a["counts"] == ref[3]).all() and a["counts"].sum() > 0
    for q in range(8):
        n = int(ref[3][q])
        assert (a["docs"][q, :n] == ref[2][q, :n]).all() and (a["segment_ords"][q, :n] == ref[1][q, :n]).all()
        assert a["scores"][q, :n].view(np.uint32).tolist() == ref[0][q, :n].view(np.uint32).tolist()
