"""GPU parity of the int8 shadow scan (csrc/scan_kernel.cuh, scan_kernel_q8): a single query reads the int8 shadow of the
rows, keeps 64 candidates, and the last CTA re-scores them from the fp32 matrix and certifies the answer against q8_delta;
an fp32 launch queued behind it runs only when the certificate failed.  Either way the call returns the BITS of the fp32
scan (set_tuning("scan_half", 0)).  "scan_q8" = 1 takes the tier whatever the matrix size."""
import numpy as np
import pytest

from oracle import exact, synthetic

pytestmark = pytest.mark.gpu


def _shard(dim, space, **kw):
    from mlvectordb_b200 import DeviceShard
    return DeviceShard(dim, space, **kw)


def _same(a, b):
    return all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


def _q8_vs_plain(s, Q, k, filt=None):
    """Every query alone, int8 shadow forced vs no shadow; returns (results, int8 queries, int8 uncertified)."""
    s.set_tuning("scan_half", 0)
    ref = [s.search(Q[i:i + 1], k, filt) for i in range(len(Q))]
    s.set_tuning("scan_half", -1)
    s.set_tuning("scan_q8", 1)          # (also resets the int8 tier's sit-out state)
    before = s.gemm_stats()
    got = [s.search(Q[i:i + 1], k, filt) for i in range(len(Q))]
    after = s.gemm_stats()
    for i, (g, r) in enumerate(zip(got, ref)):
        assert _same(g, r), f"query {i}: int8 shadow scan differs from the fp32 scan"
    used = after["q8_scan_queries"] - before["q8_scan_queries"]
    assert after["half_scan_queries"] - before["half_scan_queries"] >= used
    return got, used, after["q8_scan_uncertified"] - before["q8_scan_uncertified"]


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("k,dim", [(1, 96), (10, 96), (16, 128), (10, 192), (10, 768)])
def test_q8_scan_equals_the_fp32_scan_and_the_oracle(space, k, dim):
    n, nq = (60_000 if dim < 768 else 20_011), 10
    X = synthetic.rows(171, 0, n, dim, scaled=True)
    Q = synthetic.queries(172, nq, dim)
    Q[3] = X[777]                       # a stored row: distance ~0 for l2 / cosine
    s = _shard(dim, space)
    s.add(X)
    got, used, uncert = _q8_vs_plain(s, Q, k)
    assert used == nq and uncert <= 3, (used, uncert)
    L, D = exact.knn(X, Q, k, space)
    for i in range(nq):
        d, r, c = got[i]
        assert c[0] == len(L[i])
        assert exact.check_topk_parity(r[0, :c[0]], d[0, :c[0]], L[i], D[i]) is None
    s.close()


def test_tombstones_streamed_filter_appends_compaction_and_rebuild():
    n, dim, nq, k = 50_001, 100, 8, 10       # ld 100 floats, 128-byte int8 rows; a ragged last tile
    X = synthetic.rows(173, 0, n, dim, scaled=True)
    Q = synthetic.queries(174, nq, dim)
    s = _shard(dim, "l2", capacity=n + 5000)
    s.add(X)
    s.mark_deleted(np.arange(0, n, 7, dtype=np.uint64))
    _, used, _ = _q8_vs_plain(s, Q, k)
    assert used == nq
    mask = np.random.default_rng(5).random(n) < 0.6      # dense: stream + mask keeps the int8 shadow
    pf = s.prepare_filter(mask)
    s.set_tuning("gather", 0)
    got, used, _ = _q8_vs_plain(s, Q, k, pf)
    assert used == nq
    allow = np.ones(n, bool)
    allow[::7] = False
    L, D = exact.knn(X, Q, k, "l2", allow=allow & mask)
    for i in range(nq):
        assert exact.check_topk_parity(got[i][1][0], got[i][0][0], L[i], D[i]) is None
    s.set_tuning("gather", 1)                              # a gathered scan never reads the int8 shadow
    _, used, _ = _q8_vs_plain(s, Q, k, pf)
    assert used == 0
    s.set_tuning("gather", -1)
    pf.close()
    # rows appended after the shadow was built (some of them the queries' nearest), then compaction renumbers the rows
    extra = Q[:4] + np.float32(1e-3) * synthetic.queries(175, 4, dim)
    s.add(np.concatenate([extra, synthetic.rows(176, 0, 2000, dim, scaled=True) * np.float32(3.0)]))
    got, used, _ = _q8_vs_plain(s, Q, k)
    assert used == nq
    assert all(got[i][1][0, 0] == n + i for i in range(4))
    s.compact()
    _, used, _ = _q8_vs_plain(s, Q, k)
    assert used == nq
    s.close()


def test_fewer_rows_than_candidates():
    dim = 64
    X = synthetic.rows(177, 0, 40, dim)
    Q = synthetic.queries(178, 3, dim)
    s = _shard(dim, "cosine")
    s.add(X)
    got, used, uncert = _q8_vs_plain(s, Q, 10)           # 40 rows < 64 candidates: every row is re-scored, certified
    assert used == 3 and uncert == 0
    assert all(g[2][0] == 10 for g in got)
    s.close()


def test_crowded_neighbours_fail_the_certificate_then_the_fp16_tier_answers():
    """600 rows at nearly the same distance from the query: 64 int8 candidates cannot be told apart, the certificate
    fails, the queued fp32 launch answers -- same bits -- and after 16 such searches the int8 tier sits out while the fp16
    shadow answers."""
    n, dim, k = 40_000, 64, 10
    rng = np.random.default_rng(8)
    X = synthetic.rows(177, 0, n, dim)
    q0 = synthetic.queries(177, 1, dim)[0]
    off = rng.standard_normal((600, dim)).astype(np.float32)
    off /= np.linalg.norm(off, axis=1, keepdims=True)
    X[5000:5600] = q0 + 0.5 * off * (1 + 1e-4 * rng.standard_normal((600, 1)).astype(np.float32))
    Q = np.tile(q0, (40, 1)) + 1e-3 * rng.standard_normal((40, dim)).astype(np.float32)
    s = _shard(dim, "l2")
    s.add(X)
    st0 = s.gemm_stats()
    got, used, uncert = _q8_vs_plain(s, Q, k)
    st1 = s.gemm_stats()
    assert uncert >= 16 and used < 40, (used, uncert)     # failed every time it ran, then sat out
    # some of the searches it sat out read the fp16 shadow instead
    assert st1["half_scan_queries"] - st0["half_scan_queries"] > used
    L, D = exact.knn(X, Q[:3], k, "l2")
    for i in range(3):
        assert exact.check_topk_parity(got[i][1][0], got[i][0][0], L[i], D[i]) is None
    s.close()


def test_scan_half_one_still_means_the_fp16_shadow():
    n, dim, k = 30_000, 128, 10
    s = _shard(dim, "cosine")
    s.add(synthetic.rows(179, 0, n, dim))
    Q = synthetic.queries(180, 3, dim)
    s.set_tuning("scan_q8", 1)
    s.set_tuning("scan_half", 1)
    st0 = s.gemm_stats()
    for i in range(3):
        s.search(Q[i:i + 1], k)
    st1 = s.gemm_stats()
    assert st1["half_scan_queries"] - st0["half_scan_queries"] == 3
    assert st1["q8_scan_queries"] == st0["q8_scan_queries"]
    s.close()


def test_device_api_two_streams_in_flight():
    torch = pytest.importorskip("torch")
    n, dim, k, nq = 80_000, 128, 10, 16
    s = _shard(dim, "cosine", capacity=n)
    s.add_synthetic(181, 0, n, True)
    Q = synthetic.queries(182, nq, dim)
    s.set_tuning("scan_half", 0)
    ref = [s.search(Q[i:i + 1], k) for i in range(nq)]
    s.set_tuning("scan_half", -1)
    s.set_tuning("scan_q8", 1)
    before = s.gemm_stats()["q8_scan_queries"]
    dev = torch.device("cuda", 0)
    Qd = torch.from_numpy(Q).to(dev)
    streams = [torch.cuda.Stream(dev) for _ in range(2)]
    outs = []
    for i in range(nq):
        d = torch.empty((1, k), dtype=torch.float32, device=dev)
        r = torch.empty((1, k), dtype=torch.int64, device=dev)
        c = torch.empty((1,), dtype=torch.int32, device=dev)
        with torch.cuda.stream(streams[i & 1]):
            s.search_device(Qd[i:i + 1].data_ptr(), 1, k, d.data_ptr(), r.data_ptr(), c.data_ptr(), stream=streams[i & 1].cuda_stream)
        outs.append((d, r, c))
    torch.cuda.synchronize(dev)
    for i in range(nq):
        d, r, c = (t.cpu().numpy() for t in outs[i])
        assert _same((d, r, c), ref[i]), i
    assert s.gemm_stats()["q8_scan_queries"] - before == nq
    s.close()


def _half_step_rows(rng, n, d, spread):
    j = rng.integers(0, 126, size=(n, d)).astype(np.float64) + 0.5
    X = j * rng.choice([-1.0, 1.0], size=(n, d))
    X[:, 0] = 127.0
    s = 10.0 ** rng.uniform(-np.log10(spread) / 2, np.log10(spread) / 2, size=(n, 1)) / 127.0
    return (X * s).astype(np.float32)


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("dim", [96, 768])
def test_consumers_stay_within_the_bound(space, dim):
    """The int8 consumers' approximate distances (mlv_index_debug_q8_scan) against fp64, on rows half a step from their
    digits with norms spread 100x and queries along a row's residual: |a - exact| <= delta; prints the largest ratio."""
    rng = np.random.default_rng(dim)
    X = _half_step_rows(rng, 4000, dim, 1.0 if space == "cosine" else 100.0)
    s = _shard(dim, space)
    s.add(X)
    Xs = X.astype(np.float64)
    if space == "cosine":
        Xs /= np.linalg.norm(Xs, axis=1, keepdims=True)
    worst = 0.0
    for i in range(6):
        m = np.abs(X[i]).max() / 127.0
        res = X[i] - m * np.rint(X[i] / m)
        q = (np.sign(res) * (1.0 + 0.1 * rng.random(dim))).astype(np.float32)
        if i % 2:
            q = q + X[i] / np.abs(X[i]).max()
        a, info = s.debug_q8_scan(q)
        q64 = q.astype(np.float64)
        if space == "cosine":
            q64 /= np.linalg.norm(q64)
        exact_d = ((Xs - q64) ** 2).sum(axis=1) if space == "l2" else 1.0 - Xs @ q64
        assert np.isfinite(a).all() and info["delta"] > 0
        worst = max(worst, float(np.abs(a.astype(np.float64) - exact_d).max() / info["delta"]))
    print(f"q8 bound {space} d={dim}: max |a - exact| / delta = {worst:.3f}")
    assert worst <= 1.0, worst
    s.close()
