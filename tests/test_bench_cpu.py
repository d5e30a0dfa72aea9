"""CPU: the reference arm of bench.py (the oracle timed on host cores) keeps the JSON contract."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--rows", "40000", "--dim", "64",
                          "--cpu-sample-rows", "20000", "--steps", "2", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "exact_knn_queries_per_sec" and line["unit"] == "queries/s"
    assert line["value"] > 0 and line["higher_is_better"] is True and line["vs_baseline"] is None
    assert line["e2e"] == {"value": line["value"], "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = line["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and "scaled by 0.5" in cb["sample"] and cb["value"] == line["value"]
    assert line["config"]["rows"] == 40000 and "workload" in line["config"]
    assert line["config"]["queries_per_step"] == 32          # the GPU arm's step, not a shortened one


def test_reference_arm_uses_every_core_under_torchrun_env():
    """torchrun exports OMP_NUM_THREADS=1 to its workers; the reference arm must not inherit a 1-core baseline."""
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--rows", "20000", "--dim", "32",
                          "--cpu-sample-rows", "20000", "--steps", "1", "--warmup", "1", "--queries-per-step", "4"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["cpu_baseline"]["cores"] == len(os.sched_getaffinity(0))
    assert line["cpu_baseline"]["row_prefix_used"] is False and line["config"]["queries_per_step"] == 4


def test_steps_below_one_and_dump_of_reference_arm_are_refused(tmp_path):
    for args, flag in ((["--steps", "0"], "--steps"), (["--dump-outputs", str(tmp_path / "d")], "--dump-outputs")):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args],
                             capture_output=True, text=True, timeout=60, cwd=ROOT)
        assert out.returncode == 2 and flag in out.stderr
    assert not (tmp_path / "d").exists()


def test_dump_outputs_files_and_size_cap(tmp_path, monkeypatch):
    import numpy as np
    import bench
    rng = np.random.default_rng(0)
    nq, k = 40, 10
    d = rng.random((nq, k), dtype=np.float32)
    r = rng.integers(0, 1 << 45, (nq, k))
    c = np.full(nq, k, np.int32)
    bench.dump_outputs(str(tmp_path / "all"), d, r, c)
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in ("distances", "rows", "counts", "query_index")}
    assert got["distances"].dtype == np.float32 and np.array_equal(got["distances"], d)
    assert got["rows"].dtype == np.float64 and np.array_equal(got["rows"].astype(np.int64), r)
    assert np.array_equal(got["counts"], c) and np.array_equal(got["query_index"], np.arange(nq))
    # past the cap: the same fixed sample of queries every time, and the files stay under it
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 10 * (k * 12 + 16))
    for sub in ("a", "b"):
        bench.dump_outputs(str(tmp_path / sub), d, r, c)
    idx = np.load(tmp_path / "a" / "query_index.npy")
    assert len(idx) == 10 and np.array_equal(idx, np.load(tmp_path / "b" / "query_index.npy"))
    assert np.array_equal(np.load(tmp_path / "a" / "distances.npy"), d[idx.astype(np.int64)])
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 10 * (k * 12 + 16) + 4 * 128   # + .npy headers


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=60, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""
