"""bench.py's reference arm runs on the host cores only (the oracle), so its JSON contract can be
checked without a GPU: one line on stdout, the keys the driver reads, rank != 0 silent under
torchrun. The GPU arm's line is checked on the B200 box (tests/test_bench_gpu.py)."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _run(extra_env=None):
    env = dict(os.environ)
    env.update(extra_env or {})
    p = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--points", "20000", "--queries", "300",
                        "--steps", "2", "--warmup", "1", "--gpus", "1"], capture_output=True, text=True, env=env, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return p.stdout


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = [l for l in _run().splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "vamana_search_qps" and d["unit"] == "queries/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["value"] > 0 and abs(d["ms_per_step"] * 1e-3 * d["value"] - 300) < 1e-6 * 300 + 1e-3
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"


def test_reference_arm_is_silent_on_other_ranks():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}).strip() == ""


def test_dump_outputs_keeps_the_same_seeded_rows_under_the_limit(tmp_path, monkeypatch):
    """--dump-outputs: above the size limit every array keeps the same fixed sample of rows, listed
    in rows.npy, and two runs write the same files."""
    import numpy as np
    sys.path.insert(0, str(ROOT))
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4000)
    ids = np.arange(1000 * 10, dtype=np.float64).reshape(1000, 10)
    dists = (ids * 0.5).astype(np.float32)
    for run in ("a", "b"):
        bench.dump_outputs(tmp_path / run, {"ids": ids, "dists": dists})
    got = [{p.name: np.load(p) for p in (tmp_path / run).glob("*.npy")} for run in ("a", "b")]
    assert sorted(got[0]) == ["dists.npy", "ids.npy", "rows.npy"]
    assert sum(a.nbytes for a in got[0].values()) <= 4000
    rows = got[0]["rows.npy"].astype(np.int64)
    assert len(rows) > 0 and (np.diff(rows) > 0).all()
    assert (got[0]["ids.npy"] == ids[rows]).all() and (got[0]["dists.npy"] == dists[rows]).all()
    assert all(got[0][k].tobytes() == got[1][k].tobytes() for k in got[0])
    small = {"counts": np.full(7, 10, np.float32)}
    bench.dump_outputs(tmp_path / "c", small)
    assert sorted(p.name for p in (tmp_path / "c").glob("*.npy")) == ["counts.npy"]
    assert (np.load(tmp_path / "c" / "counts.npy") == small["counts"]).all()
