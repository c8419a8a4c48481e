"""bench.py contract checks: the reference arm runs on host cores only and must print ONE JSON line with the keys a caller
reads; under a multi-rank launch only rank 0 works and prints.  The `gpu`-marked test runs the B200 arm with --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(extra_env, *args):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", **extra_env)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args], cwd=ROOT, env=env,
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.startswith("{")]


def test_reference_arm_prints_one_contract_line():
    lines = _run({}, "--steps", "1", "--warmup", "1", "--workload", "fa")
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "candidate-sites/sec" and d["unit"] == "sites/s"
    assert d["higher_is_better"] is True and d["steps"] == 1 and d["value"] > 0
    assert d["e2e"] == {"value": d["value"], "unit": "sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and "sample" in cb
    assert cb["single_process"]["value"] > 0 and cb["deployment_shape"]["processes"] >= 1
    assert "Full-alignment" in d["config"]["workload"]


def test_reference_arm_other_ranks_exit_quietly():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--steps", "1", "--warmup", "1", "--gpus", "2") == []


def test_workload_selection():
    """Default line: everything on one GPU; under a multi-rank launch the feature counter (replicas only, no exchange) is left out
    unless asked for by name."""
    sys.path.insert(0, ROOT)
    import bench
    default = "pileup,fa,fa_dwell,cascade,pileup_counts"
    assert bench.select_workloads(default, False, 1) == default.split(",")
    assert bench.select_workloads(default, False, 8) == ["pileup", "fa", "fa_dwell", "cascade"]
    assert bench.select_workloads("pileup_counts", True, 2) == ["pileup_counts"]


def test_counter_cpu_baseline_in_the_reference_deployment_shape():
    """bench.cpu_counts_all_cores: one single-threaded oracle process per chunk of the region, rates summed; together the workers
    count exactly the bases the one-process oracle counts."""
    sys.path.insert(0, ROOT)
    import bench
    from clair3_b200 import synth_reads as sr
    from oracle import pileup_oracle as po
    rec, ref, rs = sr.random_alignment(6000, depth=20, read_len=700, seed=2)
    r = bench.cpu_counts_all_cores(rec, ref, rs, 1000, 7000, 3, min_seconds=0.0)
    assert r["processes"] == 3 and r["value"] > 0 and r["unit"] == "bases/s"
    sub = po._reads_overlapping(rec, 3000, 5000)
    whole = po.clair3_pileup(rec, 3000, 5000, ref, rs)
    part = po.clair3_pileup(sub, 3000, 5000, ref, rs)
    assert len(sub["pos"]) < len(rec["pos"])
    for k in ("matrix", "major", "stats", "cand_cols"):
        assert np.array_equal(whole[k], part[k]), k


def test_summary_tool_renders_the_committed_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "bench_summary.py"), os.path.join(ROOT, "profiles", "r2_bench_line.json")],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-1000:]
    for needle in ("| pileup |", "| fa |", "| cascade |", "## pileup_counts", "bases/s"):
        assert needle in r.stdout, needle


def test_dump_outputs_writes_floats_under_the_limit(tmp_path):
    """Integer outputs are stored as float64 (exact), floating ones as float32; a dump over the limit is refused; the row sample
    is fixed, sorted and without repeats."""
    sys.path.insert(0, ROOT)
    import bench
    counts = np.arange(-5, 7, dtype=np.int64).reshape(4, 3) * (1 << 40)
    probs = np.linspace(0, 1, 24, dtype=np.float32).reshape(1, 24)
    bench.dump_outputs(str(tmp_path / "d"), {"counts": counts, "probs": probs, "ok": np.array([0, 1], np.uint8)})
    got = {k: np.load(str(tmp_path / "d" / (k + ".npy"))) for k in ("counts", "probs", "ok")}
    assert got["counts"].dtype == np.float64 and np.array_equal(got["counts"].astype(np.int64), counts)
    assert got["probs"].dtype == np.float32 and np.array_equal(got["probs"], probs)
    assert got["ok"].dtype == np.float64 and got["ok"].tolist() == [0.0, 1.0]
    with pytest.raises(SystemExit):
        bench.dump_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_MAX_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()
    rows = bench.sample_rows(10 * bench.DUMP_SAMPLE_ROWS)
    assert len(rows) == bench.DUMP_SAMPLE_ROWS and np.all(np.diff(rows) > 0)
    assert np.array_equal(rows, bench.sample_rows(10 * bench.DUMP_SAMPLE_ROWS))
    assert np.array_equal(bench.sample_rows(100), np.arange(100))


@pytest.mark.gpu
def test_b200_arm_dumps_the_last_timed_step(tmp_path):
    """Every timed region is exactly --steps steps; the dump is float arrays under 64 MB; every dumped network row is a set of
    probability distributions (written by the last step, not left over); the feature counter's dump is the C oracle's answer on
    the bench region, bit for bit."""
    sys.path.insert(0, ROOT)
    import bench
    from clair3_b200 import synth_reads as sr
    from oracle import pileup_oracle as po
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3", "--warmup", "1", "--no-cpu-baseline",
                        "--dump-outputs", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["steps"] == 3
    for name, w in d["workloads"].items():
        assert "error" not in w, (name, w)
        assert w["steps"] == 3 and w["e2e"].get("steps", 3) == 3, name
    paths = list(out.glob("*.npy"))
    assert sum(p.stat().st_size for p in paths) <= bench.DUMP_MAX_BYTES
    got = {p.stem: np.load(str(p)) for p in paths}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    heads = {24: (21, 3), 90: (21, 3, 33, 33)}
    for name in ("pileup", "fa", "fa_dwell", "cascade_pileup", "cascade_full_alignment"):
        y = got[name]
        assert y.dtype == np.float32 and y.shape[1] in heads, name
        for part in np.split(y, np.cumsum(heads[y.shape[1]])[:-1], axis=1):
            assert np.allclose(part.sum(axis=1), 1.0, atol=1e-3), name
    assert len(got["pileup"]) == 1024 and len(got["cascade_pileup"]) == len(got["cascade_pileup_rows"]) == bench.DUMP_SAMPLE_ROWS
    cfg = bench.PLP_CFG
    rec, ref, rs = sr.random_alignment(cfg["region"], depth=cfg["depth"], read_len=cfg["read_len"], seed=cfg["seed"],
                                       indel_rate=cfg["indel_rate"], origin=cfg["origin"])
    want = po.clair3_pileup(rec, cfg["origin"], cfg["origin"] + cfg["region"], ref, rs)
    rows = got["pileup_counts_rows"].astype(np.int64)
    for k in ("matrix", "major", "stats"):
        assert np.array_equal(got["pileup_counts_" + k], want[k][rows]), k
    for k in ("cand_cols", "cand_ok"):
        assert np.array_equal(got["pileup_counts_" + k], want[k]), k
