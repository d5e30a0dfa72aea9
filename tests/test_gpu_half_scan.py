"""GPU parity of the shadow scan (csrc/scan_kernel.cuh, scan_kernel_half): a single query reads the fp16 shadow of the
rows, keeps 32 candidates, and the last CTA re-scores them from the fp32 matrix and certifies the answer; an fp32 launch
queued behind it runs only when the certificate failed.  Either way the call must return the BITS of the fp32 scan
(set_tuning("scan_half", 0)) -- and those match the CPU oracle within the north_star tolerance."""
import numpy as np
import pytest

from oracle import exact, synthetic

pytestmark = pytest.mark.gpu


def _shard(dim, space, **kw):
    from mlvectordb_b200 import DeviceShard
    return DeviceShard(dim, space, **kw)


def _same(a, b):
    return all(np.array_equal(x, y, equal_nan=True) for x, y in zip(a, b))


def _half_vs_plain(s, Q, k, filt=None):
    """Every query alone, shadow scan forced on vs off; returns (results, shadow-scan queries, uncertified)."""
    s.set_tuning("scan_half", 0)
    ref = [s.search(Q[i:i + 1], k, filt) for i in range(len(Q))]
    s.set_tuning("scan_half", 1)
    if s.dim % 64 == 0:       # rows of whole 128-byte chunks take the tensor-core consumers: the FMA consumers must agree
        s.set_tuning("scan_half_mma", 0)
        for i in range(len(Q)):
            assert _same(s.search(Q[i:i + 1], k, filt), ref[i]), f"query {i}: shadow scan (FMA consumers) differs from the fp32 scan"
        s.set_tuning("scan_half_mma", 1)
        s.set_tuning("scan_half", 1)      # (resets the sit-out state for the counted run)
    before = s.gemm_stats()
    got = [s.search(Q[i:i + 1], k, filt) for i in range(len(Q))]
    after = s.gemm_stats()
    for i, (g, r) in enumerate(zip(got, ref)):
        assert _same(g, r), f"query {i}: shadow scan differs from the fp32 scan"
    return got, after["half_scan_queries"] - before["half_scan_queries"], after["half_scan_uncertified"] - before["half_scan_uncertified"]


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("k,dim", [(1, 96), (10, 96), (16, 96), (10, 128), (16, 192), (10, 768)])
def test_shadow_scan_equals_the_fp32_scan_and_the_oracle(space, k, dim):
    n, nq = (60_000 if dim < 768 else 20_011), 12      # dim 96: FMA consumers; 128 / 192 / 768: tensor-core consumers
    X = synthetic.rows(71, 0, n, dim, scaled=True)
    Q = synthetic.queries(72, nq, dim)
    Q[3] = X[777]                       # a stored row: distance ~0 for l2 / cosine
    s = _shard(dim, space)
    s.add(X)
    got, used, uncert = _half_vs_plain(s, Q, k)
    assert used == nq and uncert <= 2, (used, uncert)
    L, D = exact.knn(X, Q, k, space)
    for i in range(nq):
        d, r, c = got[i]
        assert c[0] == len(L[i])
        assert exact.check_topk_parity(r[0, :c[0]], d[0, :c[0]], L[i], D[i]) is None
    s.close()


def test_ragged_dimension_tombstones_and_a_streamed_filter():
    n, dim, nq, k = 50_001, 100, 8, 10       # ld 100 floats, 104 halves; a ragged last tile
    X = synthetic.rows(73, 0, n, dim, scaled=False)
    Q = synthetic.queries(74, nq, dim)
    s = _shard(dim, "l2")
    s.add(X)
    s.mark_deleted(np.arange(0, n, 7, dtype=np.uint64))
    got, used, _ = _half_vs_plain(s, Q, k)
    assert used == nq
    allow = np.ones(n, bool)
    allow[::7] = False
    L, D = exact.knn(X, Q, k, "l2", allow=allow)
    for i in range(nq):
        assert exact.check_topk_parity(got[i][1][0], got[i][0][0], L[i], D[i]) is None
    mask = np.random.default_rng(5).random(n) < 0.6      # dense: stream + mask keeps the shadow scan
    pf = s.prepare_filter(mask)
    s.set_tuning("gather", 0)
    got, used, _ = _half_vs_plain(s, Q, k, pf)
    assert used == nq
    L, D = exact.knn(X, Q, k, "l2", allow=allow & mask)
    for i in range(nq):
        assert exact.check_topk_parity(got[i][1][0], got[i][0][0], L[i], D[i]) is None
    s.set_tuning("gather", 1)                              # a gathered scan copies row by row: 208-byte half rows stay fp32
    _, used, _ = _half_vs_plain(s, Q, k, pf)
    assert used == 0
    pf.close()
    s.close()


@pytest.mark.parametrize("space,dim", [("l2", 128), ("cosine", 200), ("ip", 384)])
def test_gathered_scan_over_the_shadow(space, dim):
    """A selective prepared filter makes the scan copy only the passing rows; with half rows of 256 bytes and more those
    copies read the shadow (FMA or tensor-core consumers), re-rank and certificate as ever: the fp32 gathered scan's bits."""
    n, nq, k = 40_000, 8, 10
    X = synthetic.rows(95, 0, n, dim, scaled=(space != "l2"))
    Q = synthetic.queries(96, nq, dim)
    s = _shard(dim, space)
    s.add(X)
    s.mark_deleted(np.arange(5, n, 13, dtype=np.uint64))
    mask = np.random.default_rng(9).random(n) < 0.07
    pf = s.prepare_filter(mask)
    s.set_tuning("gather", 1)
    got, used, uncert = _half_vs_plain(s, Q, k, pf)
    assert used == nq and uncert <= 2, (used, uncert)
    allow = mask.copy()
    allow[5::13] = False
    L, D = exact.knn(X, Q, k, space, allow=allow)
    for i in range(nq):
        c = int(got[i][2][0])
        assert c == len(L[i])
        assert exact.check_topk_parity(got[i][1][0, :c], got[i][0][0, :c], L[i], D[i]) is None
    s.set_tuning("scan_half_gather", 0)
    _, used, _ = _half_vs_plain(s, Q, k, pf)
    assert used == 0
    pf.close()
    s.close()


def test_fewer_rows_than_candidates_and_k_beyond_the_tier():
    dim = 64
    X = synthetic.rows(75, 0, 20, dim)
    Q = synthetic.queries(76, 3, dim)
    s = _shard(dim, "cosine")
    s.add(X)
    got, used, uncert = _half_vs_plain(s, Q, 10)          # 20 rows < 32 candidates: every row is re-scored, certified
    assert used == 3 and uncert == 0
    assert all(g[2][0] == 10 for g in got)
    _, used, _ = _half_vs_plain(s, Q, 17)                  # k > 16: not this tier's
    assert used == 0
    s.close()


def test_crowded_neighbours_fail_the_certificate_and_fall_back_on_the_device():
    """600 rows within 1e-4 (relative) of the same distance from the query: 32 candidates cannot be told apart in fp16, the
    certificate fails, the queued fp32 launch answers -- same bits -- and after 16 such searches the tier sits out."""
    n, dim, k = 40_000, 64, 10
    rng = np.random.default_rng(8)
    X = synthetic.rows(77, 0, n, dim)
    q0 = synthetic.queries(77, 1, dim)[0]
    off = rng.standard_normal((600, dim)).astype(np.float32)
    off /= np.linalg.norm(off, axis=1, keepdims=True)
    X[5000:5600] = q0 + 0.5 * off * (1 + 1e-4 * rng.standard_normal((600, 1)).astype(np.float32))
    Q = np.tile(q0, (40, 1)) + 1e-3 * rng.standard_normal((40, dim)).astype(np.float32)
    s = _shard(dim, "l2")
    s.add(X)
    got, used, uncert = _half_vs_plain(s, Q, k)
    assert uncert >= 16 and used < 40, (used, uncert)     # failed every time it ran, then sat out
    L, D = exact.knn(X, Q[:3], k, "l2")
    for i in range(3):
        assert exact.check_topk_parity(got[i][1][0], got[i][0][0], L[i], D[i]) is None
    s.close()


def test_shadow_overflow_is_caught_on_the_device_and_the_shadow_rebuilt():
    n, dim, k = 30_000, 64, 10
    X = synthetic.rows(78, 0, n, dim, scaled=True)
    Q = synthetic.queries(79, 6, dim)
    s = _shard(dim, "ip", capacity=n + 64)                 # room for the late rows: norms and shadow grow in place
    s.add(X)
    _half_vs_plain(s, Q, k)                                # freezes the shadow's scale
    s.add(X[:40] * np.float32(3.0e4))                      # far beyond it: fp16 overflow when these rows are converted
    before = s.gemm_stats()["half_scan_uncertified"]
    _half_vs_plain(s, Q, k)
    assert s.gemm_stats()["half_scan_uncertified"] > before   # flagged by the kernel, answered by the fp32 launch
    _half_vs_plain(s, Q, k)                                # the shadow is rebuilt with a new scale; still the fp32 bits
    # (with rows 3e4 times larger than the rest the certificate's margin -- relative to the largest norm -- is too wide
    # for ordinary neighbours; take the outliers away and the tier certifies again)
    s.mark_deleted(np.arange(n, n + 40, dtype=np.uint64))
    s.compact()
    got, used, uncert = _half_vs_plain(s, Q, k)
    assert used == 6 and uncert == 0, (used, uncert)
    s.close()


def test_device_api_two_streams_in_flight():
    torch = pytest.importorskip("torch")
    n, dim, k, nq = 80_000, 128, 10, 16
    s = _shard(dim, "cosine", capacity=n)
    s.add_synthetic(81, 0, n, True)
    Q = synthetic.queries(82, nq, dim)
    s.set_tuning("scan_half", 0)
    ref = s.search(Q[:1], k), [s.search(Q[i:i + 1], k) for i in range(nq)]
    s.set_tuning("scan_half", 1)
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
        assert _same((d, r, c), ref[1][i]), i
    s.close()


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("dim", [96, 128])
def test_shadow_range_scan_returns_the_fp32_hit_lists(space, dim):
    """Range mode over the shadow: rows whose approximate distance is within the fp16 bound of the radius are re-scored
    from the fp32 matrix inside the kernel and tested exactly -- the hit lists are the fp32 scan's, bit for bit, with
    tombstones and a streamed filter, at radii that cut through crowded distances, and with an overflowed shadow."""
    n, nq = 50_000, 6
    X = synthetic.rows(91, 0, n, dim, scaled=(space != "l2"))
    Q = synthetic.queries(92, nq, dim)
    s = _shard(dim, space, capacity=n + 64)
    s.add(X)
    s.mark_deleted(np.arange(3, n, 11, dtype=np.uint64))
    s.set_tuning("scan_half", 0)
    d10, _, _ = s.search(Q, 40)

    def both(radius, filt=None):
        s.set_tuning("scan_half", 0)
        ref = s.range_search(Q, radius, filt)
        s.set_tuning("scan_half", 1)
        got = s.range_search(Q, radius, filt)
        assert len(got) == len(ref)
        for (gd, gr), (rd, rr) in zip(got, ref):
            assert np.array_equal(gr, rr) and np.array_equal(gd, rd)
        return got

    for j in (0, 9, 39):                                   # radius = an actual distance: the boundary row must be in
        got = both(float(d10[0, j]))
        assert len(got[0][1]) >= j + 1
    mask = np.random.default_rng(3).random(n) < 0.5
    pf = s.prepare_filter(mask)
    s.set_tuning("gather", 0)
    both(float(d10[1, 20]), pf)
    s.set_tuning("gather", -1)
    pf.close()
    if space != "cosine":
        s.add(X[:8] * np.float32(3.0e4))                   # overflows the frozen scale: every row becomes a candidate
        both(float(d10[2, 15]))
        both(float(d10[2, 15]))                            # ... and the shadow has been rebuilt
    s.close()


def test_timing_records_one_event_pair_per_search_and_per_range_query():
    """scan_time_ms averages searches, not launches: a shadow-pair search (the shadow scan and the conditional fp32 launch
    behind it) records one event pair, as does an fp32 single query; a range search records one per query, over the
    shadow or over the fp32 rows."""
    n, dim, k = 40_000, 128, 10
    X = synthetic.rows(97, 0, n, dim, scaled=True)
    Q = synthetic.queries(98, 3, dim)
    s = _shard(dim, "l2")
    s.add(X)
    s.set_tuning("scan_half", 0)
    radius = float(s.search(Q, 5)[0][:, 4].min())      # at most ~5 hits per query
    s.set_timing(True)
    s.scan_time_ms()
    for half in (1, 0):
        s.set_tuning("scan_half", half)
        before = s.gemm_stats()["half_scan_queries"]
        s.search(Q[:1], k)
        assert s.gemm_stats()["half_scan_queries"] - before == half
        ms, pairs = s.scan_time_ms()
        assert pairs == 1 and ms > 0, (half, pairs, ms)
    for half in (1, 0):
        s.set_tuning("scan_half", half)
        s.range_search(Q, radius)
        ms, pairs = s.scan_time_ms()
        assert pairs == 3 and ms > 0, (half, pairs, ms)
    s.set_timing(False)
    s.close()
