"""bench.py's own arm at a reduced size on the GPU box: one JSON line, the contract keys, parity
with the oracle reported by the bench itself."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def test_bench_line_contract_small(tmp_path):
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--points", "50000", "--queries", "2000", "--steps", "3",
                        "--warmup", "3", "--recall-queries", "500", "--extra", "c5a,c3,c5b",
                        "--extra-n", "c5a=40000,c3=30000,c5b=60000", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [l for l in p.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["value"] > 0 and d["gpu_launches"] >= 3
    assert d["roofline"]["bound"] == "hbm" and 0 < d["roofline"]["frac"] < 1.5 and d["roofline"]["unit"] == "GB/s"
    assert d["e2e"]["h2d_bytes_per_step"] == 2000 * 128 * 4 and d["e2e"]["d2h_bytes_per_step"] == 2000 * 10 * 12 + 2000 * 4
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0
    par = d["config"]["parity"]
    assert par["id_rows_identical_to_oracle"] == 1.0 and par["dists_bit_identical"] is True and par["queries"] == 2000
    assert d["config"]["recall_at_10"] >= 0.95
    assert d["roofline"]["kernel_ms"] > 0 and d["roofline"]["kernel_ms"] <= d["ms_per_step"] * 1.05
    # --dump-outputs: the lists of the last timed step, what a caller of the search receives
    ids, dists, counts = (np.load(tmp_path / f"{k}.npy") for k in ("ids", "dists", "counts"))
    assert ids.dtype == np.float64 and dists.dtype == np.float32 and counts.dtype == np.float32
    assert ids.shape == dists.shape == (2000, 10) and counts.shape == (2000,) and (counts == 10).all()
    assert ((ids >= 2) & (ids < 50002)).all() and (np.diff(dists, axis=1) >= 0).all()
    # the other BASELINE configs measured in the same run (reduced sizes here), each with its own
    # oracle parity probe on the GPU-built graph
    ex = d["extra_configs"]
    fl = ex["flat"]  # K5 on the headline shard: tensor-core path, lists equal to the exact scan's
    assert "error" not in fl, fl
    assert fl["path"] == "tcgen05 candidate pass" and fl["lists_identical_to_exact_scan"]["identical"] is True
    assert fl["ms_per_batch"] > 0 and fl["roofline"]["bound"] == "tensor" and fl["candidates_per_query"] >= 10
    assert ex["c5a"]["points_per_s"] > 0 and ex["c5a"]["recall_at_10_of_built_graph"] >= 0.95
    assert ex["c5a"]["insert_stats"]["points"] == 40000 and 0 < ex["c5a"]["roofline"]["frac"] < 1.5
    for name in ("c3", "c5b"):
        e = ex[name]
        assert "error" not in e and "skipped" not in e, e
        assert e["parity"]["id_rows_identical_to_oracle"] == 1.0 and e["parity"]["dists_bit_identical"] is True, e["parity"]
        assert e["recall_at_10_merged_tie_aware"] >= 0.95 and e["shard_searches_per_s"] > 0
        assert 0 < e["roofline"]["frac"] < 1.5


def test_bench_dumps_are_reproducible_and_equal_the_oracle_search(tmp_path):
    """--dump-outputs: two runs with the same arguments write byte-identical files, and they hold the
    lists the oracle's search returns for the same queries on the same reference-built graph
    (built again here, on another thread count: the round schedule makes it the same graph)."""
    sys.path.insert(0, str(ROOT))
    import bench
    from oracle import oraclelib as O
    from semadb_b200 import synth
    n, B = 30000, 1000
    for run in ("a", "b"):
        p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--points", str(n), "--queries", str(B), "--steps", "2",
                            "--warmup", "1", "--extra", "none", "--no-cpu-baseline", "--no-probe", "--recall-queries", "200",
                            "--dump-outputs", str(tmp_path / run)], capture_output=True, text=True, timeout=900)
        assert p.returncode == 0, p.stderr[-2000:]
    names = sorted(f.name for f in (tmp_path / "a").glob("*.npy"))
    assert names == ["counts.npy", "dists.npy", "ids.npy"]
    for f in names:
        assert (tmp_path / "a" / f).read_bytes() == (tmp_path / "b" / f).read_bytes(), f
    X, Q = bench.c2_data(n, 0, B)
    oix, _, _ = bench.build_oracle_index(X, synth.start_vector(128, 99), 3)
    ref = oix.search(Q, k=10, search_size=75, threads=O.hw_threads())
    ids, dists, counts = (np.load(tmp_path / "a" / f"{k}.npy") for k in ("ids", "dists", "counts"))
    assert (ids == ref["ids"].astype(np.float64)).all() and dists.tobytes() == ref["dists"].tobytes()
    assert (counts == ref["counts"]).all()
