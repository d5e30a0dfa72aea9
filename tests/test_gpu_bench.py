"""GPU: ``bench.py --dump-outputs`` writes what the timed device path returned in its last step -- every query's top-k,
equal to the streamed oracle, and the same bits from a run with another step count."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--rows", "200000", "--dim", "128", "--steps", str(steps),
           "--warmup", "1", "--configs", "none", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["parity"]["ok"] is True
    return {n: np.load(os.path.join(out_dir, f"{n}.npy")) for n in ("distances", "rows", "counts", "query_index")}


def test_dumped_outputs_are_the_last_step_and_match_the_oracle(tmp_path):
    import bench
    from oracle import cscan
    a = _bench(tmp_path / "a", 3)
    nq, k, dim = 32, 10, 128
    assert a["distances"].shape == (nq, k) and a["distances"].dtype == np.float32
    assert a["rows"].dtype == np.float64 and a["counts"].tolist() == [k] * nq
    assert np.array_equal(a["query_index"], np.arange(nq))
    Q = bench.make_queries(nq, dim)
    msg = cscan.check_knn_synthetic(a["rows"].astype(np.int64), a["distances"], a["counts"].astype(np.int32), bench.SEED, 0,
                                    200_000, dim, True, Q, k, "cosine")
    assert msg is None, msg
    b = _bench(tmp_path / "b", 1)
    for name in a:
        assert np.array_equal(a[name], b[name]), name
