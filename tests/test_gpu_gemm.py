"""GPU parity of the tensor-core batch path (csrc/gemm_kernel.cuh) -- BASELINE.json configs[2].

The tcgen05 3xTF32 GEMM only selects candidates; scores come from the exact re-rank in the scan
kernel's arithmetic and uncertified queries fall back to the scan.  So the bar is stronger than
the oracle tolerance: the batch path must return BIT-IDENTICAL (rows, scores, counts) to the scan
path on the same handle, and both must match the CPU oracle within the north_star tolerance
(|a-b| <= 1e-5*max(|a|,|b|) + 1e-6, ties with the k-th score may swap).
"""
import numpy as np
import pytest

from oracle import exact, synthetic

pytestmark = pytest.mark.gpu


def _shard(dim, space, **kw):
    from mlvectordb_b200 import DeviceShard
    return DeviceShard(dim, space, **kw)


def _both_paths(s, Q, k, filt=None, stats=None):
    """Scan path vs tensor-core path in every tier configuration: 3xTF32 only, one-pass TF32 tier + scan, fp16-shadow
    tier + scan, and the default (fp16-shadow tier, 3xTF32 for what it cannot certify, scan for the rest).  Returns the
    default's results and its scan fallbacks; ``stats`` (dict) receives the default's counter deltas."""
    s.set_tuning("gemm", 0)
    ref = s.search(Q, k, filt)
    s.set_tuning("gemm", 1)
    for passes in (3, 1, 2, 0):
        s.set_tuning("gemm_passes", passes)
        before = s.gemm_stats()
        got = s.search(Q, k, filt)
        after = s.gemm_stats()
        assert after["searches"] == before["searches"] + 1, "the batch did not take the tensor-core path"
        fallbacks = after["fallback_queries"] - before["fallback_queries"]
        fast = after["fast_queries"] - before["fast_queries"]
        half = after["half_queries"] - before["half_queries"]
        assert fast == 0 if passes == 3 else fast <= len(Q)
        assert half == (fast if passes in (0, 2) else 0), f"gemm_passes={passes}: {half} of {fast} first-tier queries on the fp16 shadow"
        for a, b, name in zip(got, ref, ("dists", "rows", "counts")):
            assert a.dtype == b.dtype and a.shape == b.shape
            assert np.array_equal(a, b, equal_nan=True), f"{name}: tensor-core path (gemm_passes={passes}) differs from the scan path"
    if stats is not None:
        stats.update(fast=fast, fallbacks=fallbacks)
    return got, fallbacks


def _assert_oracle(got, X, Q, k, space, allow=None):
    d, r, c = got
    L, D = exact.knn(X, Q, k, space, allow=allow)
    Xn = exact.normalize_rows(X) if space == "cosine" else X
    Qn = exact.normalize_rows(Q) if space == "cosine" else np.asarray(Q, np.float32)
    for i in range(len(L)):
        assert c[i] == len(L[i])
        msg = exact.check_topk_parity(
            r[i, :c[i]], d[i, :c[i]], L[i], D[i],
            all_ref_scores=lambda l, i=i: exact.distances(Xn[l:l + 1], Qn[i], space)[0])
        assert msg is None, f"{space} q{i}: {msg}"


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
def test_approximate_distances_are_3xtf32_accurate(space):
    """The GEMM-form distances straight out of TMEM: error far below single-pass TF32 (2^-11)."""
    n, dim, nq = 1000, 96, 300           # ragged: 8 row tiles (last short), 3 K chunks, 2 query tiles
    X = synthetic.rows(3, 0, n, dim, scaled=True)
    Q = synthetic.queries(3, nq, dim)
    s = _shard(dim, space)
    s.add(X)
    A = s.debug_gemm(Q)
    Xn = exact.normalize_rows(X) if space == "cosine" else X
    Qn = exact.normalize_rows(Q) if space == "cosine" else Q
    X64, Q64 = Xn.astype(np.float64), Qn.astype(np.float64)
    dots = Q64 @ X64.T
    if space == "l2":
        true = (Q64 ** 2).sum(1)[:, None] + (X64 ** 2).sum(1)[None, :] - 2 * dots
        scale = (np.sqrt((Q64 ** 2).sum(1))[:, None] + np.sqrt((X64 ** 2).sum(1))[None, :]) ** 2
    else:
        true = 1 - dots
        scale = np.sqrt((Q64 ** 2).sum(1))[:, None] * np.sqrt((X64 ** 2).sum(1))[None, :] + 1e-30
    assert not np.isnan(A).any(), "rows missing from the candidate dump"
    rel = np.abs(A - true) / scale
    assert rel.max() < 2e-6, f"max |a - true| / scale = {rel.max():.3e} (single-pass TF32 would be ~5e-4)"
    s.close()


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("k", [10, 100])
def test_batch_path_equals_scan_and_oracle(space, k):
    n, dim, nq = 20_000, 96, 300
    X = synthetic.rows(17, 0, n, dim, scaled=(space != "l2"))
    Q = synthetic.queries(17, nq, dim)
    Q[1] = X[n // 2]                      # planted exact match
    X[7000] = X[123]                      # duplicated row: tie, ordered by row
    Q[2] = X[123]
    s = _shard(dim, space)
    s.add(X)
    st = {}
    got, fallbacks = _both_paths(s, Q, k, stats=st)
    assert fallbacks <= max(3, nq // 50), f"{fallbacks} of {nq} queries failed the certificate on benign data"
    assert st["fast"] >= nq * 3 // 4, f"only {st['fast']} of {nq} queries were certified by the one-pass tier"
    _assert_oracle(got, X, Q, k, space)
    s.close()


@pytest.mark.parametrize("n,dim,nq", [(16_385, 100, 257), (30_001, 33, 64), (50_000, 768, 40)])
def test_ragged_shapes(n, dim, nq):
    X = synthetic.rows(23, 0, n, dim, scaled=True)
    Q = synthetic.queries(23, nq, dim)
    s = _shard(dim, "cosine")
    s.add(X)
    got, _ = _both_paths(s, Q, 10)
    _assert_oracle(got, X, Q, 10, "cosine")
    s.close()


def test_tombstones_and_filter_in_the_epilogue():
    n, dim, nq = 25_000, 64, 280
    X = synthetic.rows(29, 0, n, dim)
    Q = synthetic.queries(29, nq, dim)
    s = _shard(dim, "l2")
    s.add(X)
    rng = np.random.default_rng(1)
    dead = rng.choice(n, size=5000, replace=False)
    s.mark_deleted(dead)
    live = np.ones(n, bool)
    live[dead] = False
    got, _ = _both_paths(s, Q, 10)
    _assert_oracle(got, X, Q, 10, "l2", allow=live)
    filt = rng.random(n) < 0.1
    got, _ = _both_paths(s, Q, 10, filt)
    _assert_oracle(got, X, Q, 10, "l2", allow=live & filt)
    sparse = np.zeros(n, bool)
    sparse[rng.choice(np.flatnonzero(live), size=7, replace=False)] = True   # fewer passing rows than k
    got, _ = _both_paths(s, Q, 10, sparse)
    assert (got[2] == 7).all()
    _assert_oracle(got, X, Q, 10, "l2", allow=sparse)
    s.close()


def test_adversarial_row_order_falls_back_to_the_scan():
    """Rows sorted far-to-near for one query: every round's rows beat the threshold, the candidate
    buffer overflows, the query is re-run by the scan -- results stay exact."""
    n, dim, nq = 40_000, 32, 64
    X = synthetic.rows(41, 0, n, dim)
    Q = synthetic.queries(41, nq, dim)
    order = np.argsort(-((X - Q[0]) ** 2).sum(1), kind="stable")
    X = np.ascontiguousarray(X[order])
    s = _shard(dim, "l2")
    s.add(X)
    got, fallbacks = _both_paths(s, Q, 10)
    assert fallbacks >= 1
    _assert_oracle(got, X, Q, 10, "l2")
    s.close()


def _counted(s, Q, k):
    before = s.gemm_stats()
    got = s.search(Q, k)
    after = s.gemm_stats()
    return got, {f: after[f] - before[f] for f in after if f != "gemm_ms"}


def test_predicted_thresholds_equal_the_plain_rule_in_fewer_rounds():
    """set_tuning("gemm_predict"): thresholds predicted from the rows seen so far append fewer candidates in fewer
    rounds; the answers are those of the plain k'-th-best rule and of the scan, bit for bit, and on rows in random
    order no prediction fails."""
    n, dim, nq, k = 400_000, 128, 512, 10
    s = _shard(dim, "l2", capacity=n)
    s.add_synthetic(77, 0, n, scaled=True)
    Q = synthetic.queries(78, nq, dim)
    s.mark_deleted(np.arange(0, n, 9, dtype=np.uint64))
    s.set_tuning("gemm", 0)
    ref = s.search(Q, k)
    s.set_tuning("gemm", 1)
    seen = {}
    for predict in (0, 1):
        s.set_tuning("gemm_predict", predict)
        got, d = _counted(s, Q, k)
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, ref)), f"gemm_predict={predict}"
        assert d["mispredicted_queries"] == 0 and d["half_queries"] >= nq * 9 // 10, d
        seen[predict] = d
    assert seen[1]["rounds"] < seen[0]["rounds"], seen
    assert seen[1]["fallback_queries"] == seen[0]["fallback_queries"]
    s.close()


def test_mispredicted_thresholds_are_caught_and_back_off():
    """Rows stored nearest-first around the queries' centre: the first tiles promise far more close rows than the matrix
    holds, the predicted thresholds starve the candidate buffers, the last round's check catches it (the next tier
    answers those queries) and predictions sit out 8, then 16 batches.  Answers stay the scan's bit for bit."""
    n, dim, nq, k = 150_000, 64, 256, 10
    rng = np.random.default_rng(12)
    X = synthetic.rows(61, 0, n, dim)
    c = synthetic.queries(61, 1, dim)[0]
    X = np.ascontiguousarray(X[np.argsort(((X - c) ** 2).sum(1), kind="stable")])
    Q = (c + 0.02 * rng.standard_normal((nq, dim))).astype(np.float32)
    s = _shard(dim, "l2")
    s.add(X)
    s.set_tuning("gemm", 0)
    ref = s.search(Q, k)
    s.set_tuning("gemm", 1)
    missed = []
    for _ in range(11):
        got, d = _counted(s, Q, k)
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, ref))
        missed.append(d["mispredicted_queries"])
        if d["mispredicted_queries"] == 0:
            assert d["half_queries"] >= nq * 9 // 10, d       # the plain rule certifies them on the fp16 tier
    assert missed[0] > nq // 8 and missed[9] > nq // 8, missed
    assert sum(1 for m in missed if m) == 2, missed           # batches 1-8 sat out, batch 10 sits out again (16)
    _assert_oracle((got[0][:3], got[1][:3], got[2][:3]), X, Q[:3], k, "l2")
    s.close()


def test_large_batch_on_device_generated_rows():
    """200k x 768 generated on the device, 512 queries: the batch path equals the scan path bit for bit."""
    n, dim, nq = 200_000, 768, 512
    s = _shard(dim, "cosine", capacity=n)
    s.add_synthetic(42, 0, n, scaled=True)
    Q = synthetic.queries(43, nq, dim)
    Q[5] = synthetic.rows(42, 1234, 1, dim, scaled=True)[0]
    st = {}
    got, fallbacks = _both_paths(s, Q, 10, stats=st)
    assert got[1][5, 0] == 1234
    assert fallbacks <= 10 and st["fast"] >= nq * 9 // 10
    s.close()


def test_one_pass_tier_hands_near_ties_to_the_3xtf32_tier():
    """Many near-duplicates of the query's neighbours: the exact k-th best sits within the one-pass tier's error
    of the (k'+1)-th, so that tier cannot certify; the 3xTF32 tier (or the scan) answers and results stay exact."""
    n, dim, nq, k = 30_000, 64, 32, 10
    rng = np.random.default_rng(5)
    X = synthetic.rows(81, 0, n, dim)
    Q = synthetic.queries(81, nq, dim)
    # 400 rows at almost the same distance from Q[0]: Q[0] + a fixed-length offset, directions random
    off = rng.standard_normal((400, dim)).astype(np.float32)
    off /= np.linalg.norm(off, axis=1, keepdims=True)
    X[1000:1400] = Q[0] + 0.5 * off * (1 + 1e-4 * rng.standard_normal((400, 1)).astype(np.float32))
    s = _shard(dim, "l2")
    s.add(X)
    st = {}
    got, _ = _both_paths(s, Q, k, stats=st)
    assert st["fast"] < nq, "the crowded query should not have been certified by the one-pass tier"
    assert set(got[1][0].tolist()) <= set(range(1000, 1400))
    _assert_oracle(got, X, Q, k, "l2")
    s.close()


def test_largest_k_on_the_batch_path():
    """k = 1000 (the REST bound): k' = 1280 candidates per query, 8192-slot buffers, short growth factor."""
    n, dim, nq, k = 40_000, 48, 24, 1000
    X = synthetic.rows(71, 0, n, dim)
    Q = synthetic.queries(71, nq, dim)
    s = _shard(dim, "l2")
    s.add(X)
    got, fallbacks = _both_paths(s, Q, k)
    assert (got[2] == k).all()
    _assert_oracle((got[0][:3], got[1][:3], got[2][:3]), X, Q[:3], k, "l2")
    s.close()


def test_one_pass_tier_sits_out_when_it_certifies_too_little():
    """Every query crowded: the one-pass tier fails for all of them once, then is skipped for the next batches
    (fewer GEMM rounds per batch), and the answers stay bit-identical to the scan."""
    n, dim, nq, k = 30_000, 64, 16, 10
    rng = np.random.default_rng(6)
    X = synthetic.rows(91, 0, n, dim)
    q0 = synthetic.queries(91, 1, dim)[0]
    off = rng.standard_normal((600, dim)).astype(np.float32)
    off /= np.linalg.norm(off, axis=1, keepdims=True)
    X[2000:2600] = q0 + 0.5 * off * (1 + 1e-4 * rng.standard_normal((600, 1)).astype(np.float32))
    Q = np.tile(q0, (nq, 1)) + 1e-3 * rng.standard_normal((nq, dim)).astype(np.float32)
    s = _shard(dim, "l2")
    s.add(X)
    s.set_tuning("gemm", 0)
    ref = s.search(Q, k)
    s.set_tuning("gemm", 1)
    rounds = []
    for _ in range(3):
        before = s.gemm_stats()
        got = s.search(Q, k)
        after = s.gemm_stats()
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, ref))
        rounds.append(after["rounds"] - before["rounds"])
        assert after["fast_queries"] - before["fast_queries"] <= nq // 2
    assert rounds[1] < rounds[0] and rounds[2] == rounds[1], rounds   # batches 2 and 3 ran one tier only
    s.close()


@pytest.mark.parametrize("space", ["l2", "cosine"])
def test_filtered_batch_multiplies_a_compacted_copy_of_the_passing_rows(space):
    """Selective filter on the tensor-core path: the passing-and-live rows are gathered into a dense matrix, the tiers
    run on it and candidate positions are mapped back -- bit-identical to the scan (which gathers row by row) for a
    prepared filter, a per-call mask and a device-evaluated predicate; a dense filter keeps the masked epilogue."""
    n, dim, nq, k = 200_000, 64, 300, 10
    X = synthetic.rows(57, 0, n, dim, scaled=True)
    Q = synthetic.queries(57, nq, dim)
    rng = np.random.default_rng(9)
    s = _shard(dim, space)
    s.add(X)
    dead = rng.choice(n, size=20_000, replace=False)
    s.mark_deleted(dead)
    live = np.ones(n, bool)
    live[dead] = False
    buckets = rng.integers(0, 100, n).astype(np.int32)
    s.set_column(0, buckets)
    for cut, gathered in ((20, True), (80, False)):
        mask = buckets < cut
        Q[0] = X[np.flatnonzero(mask & live)[77]]
        pf = s.prepare_filter(mask)
        wf = s.where([(0, "<", cut)])
        for filt in (pf, mask, wf):
            before = s.gemm_stats()["gathered_searches"]
            got, _ = _both_paths(s, Q, k, filt)
            after = s.gemm_stats()["gathered_searches"]
            assert (after - before == 4) == gathered, (cut, after - before)     # one per tier configuration
            assert got[1][0, 0] == np.flatnonzero(mask & live)[77] and mask[got[1]].all() and live[got[1]].all()
        _assert_oracle((got[0][:4], got[1][:4], got[2][:4]), X, Q[:4], k, space, allow=mask & live)
        pf.close()
        wf.close()
    # fewer passing rows than a GEMM round is worth: the gathered scan answers (same results, no compaction)
    tiny = buckets < 1
    before = s.gemm_stats()["gathered_searches"]
    got, _ = _both_paths(s, Q, k, tiny)
    assert s.gemm_stats()["gathered_searches"] == before
    _assert_oracle((got[0][:3], got[1][:3], got[2][:3]), X, Q[:3], k, space, allow=tiny & live)
    s.close()


@pytest.mark.parametrize("space", ["l2", "ip"])
def test_one_pass_distances_stay_inside_the_certificate_bound(space):
    """The certificate of the one-pass tier assumes |a - exact| <= delta_rel * scale with delta_rel = 2^-9 (1 + 2^-11) +
    d 2^-22 (ip; half of it on the l2 scale).  Worst case for the truncation: every value just below a TF32 step and all
    products of one sign -- the measured error must approach the bound from below, random data stays far inside."""
    n, dim, nq = 2048, 768, 64
    rng = np.random.default_rng(3)
    step = 2.0 ** -10                                       # TF32 keeps 10 explicit mantissa bits
    worst = lambda shape: ((1.0 + rng.integers(0, 1024, shape) * step + step * (1 - 2.0 ** -13))
                           * 2.0 ** rng.integers(-2, 3, shape)).astype(np.float32)
    for X, Q, expect_close in ((worst((n, dim)), worst((nq, dim)), True),
                               (synthetic.rows(4, 0, n, dim, scaled=True), synthetic.queries(4, nq, dim), False)):
        s = _shard(dim, space)
        s.add(X)
        s.set_tuning("gemm_passes", 1)
        A = s.debug_gemm(Q)
        X64, Q64 = X.astype(np.float64), Q.astype(np.float64)
        dots = Q64 @ X64.T
        xn, qn = np.sqrt((X64 ** 2).sum(1)), np.sqrt((Q64 ** 2).sum(1))
        if space == "l2":
            true = (qn ** 2)[:, None] + (xn ** 2)[None, :] - 2 * dots
            scale = (xn.max() + qn[:, None]) ** 2 * np.ones_like(dots)
            bound = 0.5 * (2.0 ** -9 * (1 + 2.0 ** -11) + dim * 2.0 ** -22)
        else:
            true = 1 - dots
            scale = xn.max() * qn[:, None] * np.ones_like(dots)
            bound = 2.0 ** -9 * (1 + 2.0 ** -11) + dim * 2.0 ** -22
        rel = np.abs(A - true) / scale
        assert not np.isnan(A).any()
        assert rel.max() < bound, f"{space}: {rel.max():.3e} exceeds the certificate's delta {bound:.3e}"
        if expect_close:
            assert rel.max() > 0.25 * bound, f"worst-case input only reached {rel.max():.3e} of {bound:.3e}"
        else:
            assert rel.max() < 0.1 * bound
        s.close()


@pytest.mark.parametrize("space", ["l2", "ip"])
def test_fp16_tier_distances_stay_inside_the_certificate_bound(space):
    """The fp16-shadow tier rounds both operands to 11 significant bits (scaled by exact powers of two):
    |a - exact| <= delta_rel * scale with delta_rel = 2^-10 (1 + 2^-12) + d 2^-22 (ip; half on the l2 scale).  Worst case
    for round-to-nearest: every value just below a half step and all products of one sign; data spread over many
    binades and data with huge / tiny magnitudes (the scales keep the halves in range) stay inside as well."""
    n, dim, nq = 2048, 768, 64
    rng = np.random.default_rng(3)
    step = 2.0 ** -10
    worst = lambda shape: ((1.0 + rng.integers(0, 1024, shape) * step + 0.5 * step * (1 - 2.0 ** -12))
                           * 2.0 ** rng.integers(-2, 3, shape)).astype(np.float32)
    benign = (synthetic.rows(4, 0, n, dim, scaled=True), synthetic.queries(4, nq, dim))
    cases = [(worst((n, dim)), worst((nq, dim)), True),
             (benign[0], benign[1], False),
             (benign[0] * np.float32(3.0e6), benign[1] * np.float32(2.0e-7), False),       # far outside fp16's own range
             (benign[0] * (2.0 ** rng.integers(-12, 1, (n, 1))).astype(np.float32), benign[1], False)]   # rows over 12 binades
    for X, Q, expect_close in cases:
        s = _shard(dim, space)
        s.add(X)
        s.set_tuning("gemm_passes", 2)
        A = s.debug_gemm(Q)
        X64, Q64 = X.astype(np.float64), Q.astype(np.float64)
        dots = Q64 @ X64.T
        xn, qn = np.sqrt((X64 ** 2).sum(1)), np.sqrt((Q64 ** 2).sum(1))
        e = 2.0 ** -10 * (1 + 2.0 ** -12) + dim * 2.0 ** -22
        if space == "l2":
            true = (qn ** 2)[:, None] + (xn ** 2)[None, :] - 2 * dots
            scale = (xn.max() + qn[:, None]) ** 2 * np.ones_like(dots)
            bound = 0.5 * e
        else:
            true = 1 - dots
            scale = xn.max() * qn[:, None] * np.ones_like(dots)
            bound = e
        rel = np.abs(A - true) / scale
        assert not np.isnan(A).any() and np.isfinite(A).all()
        assert rel.max() < bound, f"{space}: {rel.max():.3e} exceeds the certificate's delta {bound:.3e}"
        if expect_close:
            assert rel.max() > 0.2 * bound, f"worst-case input only reached {rel.max():.3e} of {bound:.3e}"
        s.close()


def test_fp16_shadow_follows_adds_deletes_compaction_and_rescales():
    """The shadow is built lazily and must follow the matrix: appended rows are converted with the frozen scale, rows far
    larger than anything seen when it was frozen overflow -> the batch is answered by the next tiers and the shadow is
    rebuilt; compaction invalidates it.  Results stay bit-identical to the scan throughout."""
    n, dim, nq, k = 20_000, 96, 40, 10
    X = synthetic.rows(33, 0, n, dim, scaled=True)
    Q = synthetic.queries(33, nq, dim)
    s = _shard(dim, "l2")
    s.add(X[: n // 2])

    def check(expect_half=None):
        s.set_tuning("gemm", 0)
        ref = s.search(Q, k)
        s.set_tuning("gemm", 1)
        before = s.gemm_stats()
        got = s.search(Q, k)
        after = s.gemm_stats()
        assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(got, ref))
        half = after["half_queries"] - before["half_queries"]
        if expect_half is not None:
            assert (half > nq // 2) == expect_half, half
        return got

    check(True)
    s.add(X[n // 2:])                                   # appended rows: converted incrementally
    got = check(True)
    _assert_oracle((got[0][:4], got[1][:4], got[2][:4]), X, Q[:4], k, "l2")
    s.mark_deleted(got[1][:, 0])                        # the nearest row of every query goes away
    check(True)
    s.compact()
    check(True)
    first_big = s.rows
    big = X[:50] * np.float32(1.0e4)                    # 2^13 x the frozen scale's headroom: fp16 overflow
    s.add(big)
    check(False)                                        # this batch: overflow flag -> 3xTF32 tier / scan
    # (with those outliers in the matrix no one-pass tier can certify: its error bound is relative to the largest row)
    s.mark_deleted(np.arange(first_big, first_big + 50))
    s.compact()                                         # norms, largest norm and shadow are rebuilt: fresh scale
    check(True)
    s.close()


@pytest.mark.parametrize("space", ["l2", "cosine"])
def test_cta_pair_kernel_equals_the_single_tile_kernel(space):
    """Wide batches (>= 129 queries) run the one-pass tiers on gemm_topk_pair_kernel (tcgen05 cta_group::2: a CTA pair
    computes 256 x 256 per instruction, each SM staging its own rows and half of the query tile); gemm_wide 0 keeps the
    single-tile kernel.  Odd row-tile counts, a ragged K (dim % 64 != 0), two query tiles, tombstones: both return the
    scan's bits."""
    n, dim, nq, k = 60_050, 200, 300, 10
    X = synthetic.rows(51, 0, n, dim, scaled=True)
    Q = synthetic.queries(51, nq, dim)
    Q[7] = X[n - 1]
    s = _shard(dim, space)
    s.add(X)
    s.mark_deleted(np.arange(3, n, 11))
    s.set_tuning("gemm", 0)
    ref = s.search(Q, k)
    s.set_tuning("gemm", 1)
    for wide in (0, 3):
        s.set_tuning("gemm_wide", wide)
        for passes in (2, 1, 0):
            s.set_tuning("gemm_passes", passes)
            before = s.gemm_stats()
            got = s.search(Q, k)
            after = s.gemm_stats()
            assert after["searches"] == before["searches"] + 1
            assert after["fast_queries"] - before["fast_queries"] >= nq * 9 // 10, (wide, passes)
            for a, b, name in zip(got, ref, ("dists", "rows", "counts")):
                assert np.array_equal(a, b, equal_nan=True), f"{name}: gemm_wide={wide} gemm_passes={passes} differs from the scan"
    live = np.ones(n, bool)
    live[3::11] = False
    _assert_oracle((ref[0][:4], ref[1][:4], ref[2][:4]), X, Q[:4], k, space, allow=live)
    if space != "cosine":
        assert ref[1][7, 0] == n - 1 or not live[n - 1]
    s.close()


@pytest.mark.parametrize("wide", [0, None])
@pytest.mark.parametrize("passes", [0, 1, 2, 3])
def test_each_round_is_one_timed_region_and_two_launches(passes, wide):
    """With timing on, a batch adds one timed region per GEMM round.  Once the row norms and the fp16 shadow exist, it
    launches the query preparation, then per tier the query split, a GEMM and a refine per round and the re-rank, and the
    gather / scatter around a 3xTF32 tier that re-runs failing queries.  wide None = the default (CTA pairs)."""
    n, dim, nq, k = 20_000, 128, 300, 10       # 300 queries: 256-wide tiles, the CTA-pair kernel on one-pass tiers
    rng = np.random.default_rng(31)
    s = _shard(dim, "l2")
    s.add(rng.standard_normal((n, dim), dtype=np.float32))
    Q = rng.standard_normal((nq, dim), dtype=np.float32)
    s.set_tuning("gemm", 1)
    s.set_tuning("gemm_passes", passes)
    if wide is not None:
        s.set_tuning("gemm_wide", wide)
    s.set_timing(True)
    s.search(Q, k)                             # builds the row norms and (passes 0, 2) the fp16 shadow
    before, launches = s.gemm_stats(), s.kernel_launches()
    s.search(Q, k)
    after, launches = s.gemm_stats(), s.kernel_launches() - launches
    d = {f: after[f] - before[f] for f in ("searches", "rounds", "fast_queries", "half_queries", "fallback_queries")}
    assert d["searches"] == 1 and d["rounds"] > 0 and d["fallback_queries"] == 0, d
    assert d["half_queries"] == (d["fast_queries"] if passes in (0, 2) else 0), d
    assert passes != 3 or d["fast_queries"] == 0, d
    assert after["gemm_launches_timed"] == d["rounds"], (after["gemm_launches_timed"], d)   # gemm_stats drains the regions it reports
    second = passes == 0 and d["fast_queries"] < nq
    tiers = 2 if second else 1
    assert launches == 1 + 2 * tiers + 2 * d["rounds"] + (2 if second else 0), (launches, d)
    s.close()


def test_debug_rounds_are_neither_counted_nor_timed():
    """debug_gemm_rounds launches the query preparation, the split and a GEMM and a refine per round, and leaves the
    search counters and the timed regions alone."""
    n, dim, nq = 20_000, 128, 64
    rng = np.random.default_rng(32)
    s = _shard(dim, "l2")
    s.add(rng.standard_normal((n, dim), dtype=np.float32))
    Q = rng.standard_normal((nq, dim), dtype=np.float32)
    s.set_timing(True)
    s.set_tuning("gemm", 1)
    s.search(Q, 10)                            # builds the row norms
    before, launches = s.gemm_stats(), s.kernel_launches()
    rounds = [(8, 96), (40, 96), (-(-n // 128), 96)]
    for bn, passes in ((64, 1), (64, 3), (0, 2)):
        s.debug_gemm_rounds(Q, passes=passes, bn=bn, cap=1024, rounds=rounds, kprime=96)
    after, launches = s.gemm_stats(), s.kernel_launches() - launches
    assert after["rounds"] == before["rounds"] and after["searches"] == before["searches"]
    assert after["gemm_launches_timed"] == 0
    assert launches == 3 * (2 + 2 * len(rounds)), launches
    s.close()
