"""What a batch-path GEMM round emits (csrc/gemm_kernel.cuh), checked row by row.

rerank_kernel certifies an answer on the premise that every row outside a query's candidate set has an approximate
distance a >= a_k'.  That holds only if the GEMM epilogue (epilogue_constants, epilogue_drain, hitq_flush) emits EVERY
row with a <= the query's threshold exactly once, with the right key, and refine_kernel keeps the k' smallest.  End-to-end
equality with the scan sees a lost or doubled candidate only when it is one of the k best; these tests see all of them.

mlv_index_debug_gemm_rounds runs the production kernels -- gemm_topk_kernel (BN 64 / 128 / 256) or gemm_topk_pair_kernel,
refine_kernel after each round -- and returns the raw candidate buffers.  The reference is a_r, the kernel's own
approximate distance of row r from a run at threshold +inf (test 1 shows that run is complete, unique and reproducible);
the fp64 reference bounds a_r itself."""
import numpy as np
import pytest

from oracle import exact, synthetic

pytestmark = pytest.mark.gpu

BM = 128                                             # rows per tile
KERNELS = [(p, bn) for p in (1, 2, 3) for bn in (64, 128, 256)] + [(1, 0), (2, 0)]   # (passes, bn); bn 0 = CTA pair


def _kid(kern):
    return f"p{kern[0]}-" + ("pair" if kern[1] == 0 else f"bn{kern[1]}")


def _shard(dim, space, X, dead=None):
    from mlvectordb_b200 import DeviceShard
    s = DeviceShard(dim, space)
    s.add(X)
    if dead is not None and len(dead):
        s.mark_deleted(np.asarray(dead, np.uint64))
    return s


def _pow2(n):
    return 1 << (int(n) - 1).bit_length()


def _hits(out, n):
    """-> (times each (query, row) was emitted [nq, n], emitted distance [nq, n] (NaN where none)); nothing beyond cap."""
    from mlvectordb_b200.shard import key_parts
    keys, counts = out["keys"], out["counts"]
    nq, cap = keys.shape
    assert (counts <= cap).all(), "more hits than slots"
    valid = np.arange(cap)[None, :] < counts[:, None]
    d, r = key_parts(keys[valid])
    qi = np.nonzero(valid)[0]
    assert (r < n).all(), "a row beyond the matrix was emitted"
    mult = np.zeros((nq, n), np.int64)
    np.add.at(mult, (qi, r.astype(np.int64)), 1)
    A = np.full((nq, n), np.nan, np.float32)
    A[qi, r.astype(np.int64)] = d
    return mult, A


def _sorted_keys(out):
    keys, counts = out["keys"], out["counts"]
    stored = np.arange(keys.shape[1])[None, :] < np.minimum(counts, keys.shape[1])[:, None]
    return np.sort(np.where(stored, keys, np.uint64(2 ** 64 - 1)), axis=1)


def _approx(s, Q, kern, n, allow):
    """a_r [nq, n] of one kernel (NaN for rows that take no part), asserting the +inf run emitted each allowed row once."""
    out = s.debug_gemm_rounds(Q, *kern, cap=_pow2(n))
    mult, A = _hits(out, n)
    assert out["pad_count"] == 0 and (mult == allow[None, :]).all(), f"{_kid(kern)}: incomplete emission at +inf"
    return A


# ---- 1. emission at +inf -----------------------------------------------------------------------------------------------
N1, D1 = 1111, 100        # 9 row tiles (odd: the pair kernel's unpaired tile; the last holds 87 rows); dim 100: ragged K chunks


@pytest.mark.parametrize("kern", KERNELS, ids=_kid)
@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
def test_emission_at_inf_is_complete_unique_and_reproducible(space, kern):
    X = synthetic.rows(11, 0, N1, D1, scaled=space != "l2")
    dead = np.arange(4, N1, 13)
    s = _shard(D1, space, X, dead)
    mask = np.random.default_rng(2).random(N1) < 0.8
    allow = mask.copy()
    allow[dead] = False
    tiles = -(-N1 // BM)
    for nq in (1, 64, 65, 129, 300):
        Q = synthetic.queries(12 + nq, nq, D1)
        out = s.debug_gemm_rounds(Q, *kern, cap=2048, mask=mask)
        mult, A = _hits(out, N1)
        assert out["pad_count"] == 0, f"nq {nq}: padding queries emitted {out['pad_count']} hits"
        assert (mult[:, ~allow] == 0).all(), f"nq {nq}: a tombstoned or filtered row was emitted"
        assert (mult[:, allow] == 1).all(), f"nq {nq}: rows lost {(mult[:, allow] == 0).sum()}, doubled {(mult > 1).sum()}"
        assert (out["counts"] == allow.sum()).all() and np.isfinite(A[:, allow]).all()
        ref = _sorted_keys(out)
        variants = [{}]
        if nq in (65, 300):
            variants += [{"max_ctas": 1}, {"max_ctas": 7}]   # one CTA (pair) walks every item: stage ring and accumulator phases
        for v in variants:
            again = s.debug_gemm_rounds(Q, *kern, cap=2048, mask=mask, **v)
            assert np.array_equal(_sorted_keys(again), ref), f"nq {nq} {v}: keys differ between runs"
        if nq == 129:
            part = s.debug_gemm_rounds(Q, *kern, cap=2048, mask=mask, rounds=[(5, 0)])
            inside = allow & (np.arange(N1) < 5 * BM)
            assert (_hits(part, N1)[0] == inside[None, :]).all(), "a round emitted rows outside its tiles"
            split = s.debug_gemm_rounds(Q, *kern, cap=2048, mask=mask, rounds=[(2, 0), (5, 0), (tiles, 0)])
            assert np.array_equal(_sorted_keys(split), ref), "three rounds emit other keys than one"
    s.close()


# ---- 2. the pair kernel against fp64 and against the single-tile kernel --------------------------------------------------
def _delta_rel(passes, l2, ld):
    """gemm_kernel.cuh: the certificate's bound on |a - exact| / scale, evaluated like the device (float32)."""
    f = np.float32
    if passes == 3:
        return f(1.220703125e-4)
    base = f(1.953125e-3) * (f(1) + f(4.8828125e-4)) if passes == 1 else f(9.765625e-4) * (f(1) + f(2.44140625e-4))
    e = f(base + f(ld) * f(2.384185791015625e-7)) + f(9.5367431640625e-7)
    return f(0.5) * e if l2 else e


def _exact_and_scale(s, Q):
    """fp64 GEMM-form distances [nq, rows] of the stored rows to the prepared queries, and the certificate's scale."""
    X = s.export_rows().astype(np.float64)
    Q = np.asarray(Q, np.float64)
    if s.space == "cosine":
        Q = Q / np.linalg.norm(Q, axis=1, keepdims=True)
    dots = Q @ X.T
    xn, qn = np.sqrt((X ** 2).sum(1)), np.sqrt((Q ** 2).sum(1))
    if s.space == "l2":
        return (qn ** 2)[:, None] + (xn ** 2)[None, :] - 2 * dots, ((xn.max() + qn) ** 2)[:, None]
    scale = np.ones((len(Q), 1)) if s.space == "cosine" else (xn.max() * qn)[:, None]
    return 1 - dots, scale


@pytest.mark.parametrize("passes", [1, 2])
@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
def test_pair_kernel_distances_against_fp64_and_the_single_tile_kernel(space, passes):
    n, dim, nq = 2048, 768, 256
    rng = np.random.default_rng(3 + passes)
    step = 2.0 ** -10
    # truncation (TF32) / round-to-nearest (fp16) worst case: every value just below a step / a half step, one sign
    off = step * (1 - 2.0 ** -13) if passes == 1 else 0.5 * step * (1 - 2.0 ** -12)
    worst = lambda shape: ((1.0 + rng.integers(0, 1024, shape) * step + off) * 2.0 ** rng.integers(-2, 3, shape)).astype(np.float32)
    benign = (synthetic.rows(4, 0, n, dim, scaled=True), synthetic.queries(4, nq, dim))
    cases = [("worst", worst((n, dim)), worst((nq, dim))), ("benign",) + benign,
             ("huge rows, tiny queries", benign[0] * np.float32(3.0e6), benign[1] * np.float32(2.0e-7)),
             ("rows over 12 binades", benign[0] * (2.0 ** rng.integers(-12, 1, (n, 1))).astype(np.float32), benign[1])]
    allow = np.ones(n, bool)
    for name, X, Q in cases:
        s = _shard(dim, space, X)
        A = _approx(s, Q, (passes, 0), n, allow)
        single = _approx(s, Q, (passes, 256), n, allow)
        true, scale = _exact_and_scale(s, Q)
        ratio = float((np.abs(A - true) / scale).max() / _delta_rel(passes, space == "l2", s.info().ld))
        same = np.array_equal(A.view(np.uint32), single.view(np.uint32))
        print(f"pair kernel, passes {passes}, {space}, {name}: {ratio:.3f} of delta; bit-identical to BN 256: {same}")
        assert ratio < 1.0, f"{name}: |a - exact| reached {ratio:.3f} of delta * scale"
        if name == "worst" and space != "cosine":   # cosine rows are normalised by the index: off the worst-case grid
            assert ratio > (0.25 if passes == 1 else 0.2), f"worst-case input only reached {ratio:.3f} of delta"
        assert same, f"{name}: the pair kernel's distances differ from the single-tile kernel's " \
                     f"(max {np.abs(A.astype(np.float64) - single).max():.3e})"
        s.close()


# ---- 3. the threshold test is exact ------------------------------------------------------------------------------------
KP = 96
RANKS = (1, 31, 32, 33, KP)


def _threshold_data(name):
    """(space, X, Q): data on which the relaxed pre-test and the exact test could disagree if the relaxation were wrong."""
    rng = np.random.default_rng(len(name))
    n, dim, nq = 1500, 100, 68
    if name == "l2 cancellation":           # rows = c + noise, |c| >> spread: |x|^2 + |q|^2 - 2 x.q cancels 12 bits
        c = 1000.0 * rng.standard_normal(dim) / np.sqrt(dim)
        return "l2", (c + 0.01 * rng.standard_normal((n, dim))).astype(np.float32), (c + 0.01 * rng.standard_normal((nq, dim))).astype(np.float32)
    if name == "ip, |dot| >> 1":             # negative distances down to about -300
        return "ip", (30.0 * rng.standard_normal((n, dim))).astype(np.float32), rng.standard_normal((nq, dim)).astype(np.float32)
    if name == "ip above 3e38":              # distances 3.06e38 .. 3.2e38: finite thresholds beyond the relaxation's guard
        X = 1.75e18 * (1 + 0.01 * rng.random((n, dim)))
        Q = -1.75e18 * (1 + 0.01 * rng.random((nq, dim)))
        return "ip", X.astype(np.float32), Q.astype(np.float32)
    if name == "huge rows, tiny queries":    # far outside fp16's own range: the shadow's scales carry it
        return "l2", synthetic.rows(9, 0, n, dim, scaled=True) * np.float32(3.0e6), synthetic.queries(9, nq, dim) * np.float32(2.0e-7)
    # many identical rows nearest to every query: ties exactly at the thresholds
    X = synthetic.rows(8, 0, n, dim, scaled=True)
    twin = synthetic.queries(8, 1, dim)[0]
    X[rng.choice(n, 300, replace=False)] = twin
    return "cosine", X, (twin + 0.05 * rng.standard_normal((nq, dim))).astype(np.float32)


def _threshold_grid(A):
    """Per query: a_r at ranks 1, 31, 32, 33, k', ~n/2, the next float below each, -inf, +inf, NaN, +0, -0 (query i takes
    entry i % 17)."""
    out = np.empty(len(A), np.float32)
    for i, a in enumerate(A):
        srt = np.sort(a[np.isfinite(a)])
        grid = []
        for rk in RANKS + (len(srt) // 2,):
            grid += [srt[rk - 1], np.nextafter(srt[rk - 1], np.float32(-np.inf))]
        grid += [-np.inf, np.inf, np.nan, 0.0, -0.0]
        out[i] = np.float32(grid[i % len(grid)])
    return out


@pytest.mark.parametrize("kern", KERNELS, ids=_kid)
@pytest.mark.parametrize("data", ["l2 cancellation", "ip, |dot| >> 1", "ip above 3e38", "huge rows, tiny queries", "cosine ties"])
def test_threshold_selection_is_exact(data, kern):
    space, X, Q = _threshold_data(data)
    n = len(X)
    s = _shard(X.shape[1], space, X)
    allow = np.ones(n, bool)
    A = _approx(s, Q, kern, n, allow)
    if data == "ip above 3e38":
        assert (A > 3.0e38).all() and np.isfinite(A).all()
    thr = _threshold_grid(A)
    out = s.debug_gemm_rounds(Q, *kern, cap=_pow2(n), thresholds=thr)
    mult, got = _hits(out, n)
    want = A <= thr[:, None]
    for i in np.nonzero((mult != want).any(1))[0][:3]:
        lost, extra = np.nonzero(want[i] & (mult[i] == 0))[0], np.nonzero((mult[i] != want[i]) & (mult[i] != 0))[0]
        pytest.fail(f"{data} {_kid(kern)} q{i} thr {thr[i]!r}: {len(lost)} rows at or below it lost (a {A[i, lost[:3]]}), "
                    f"{len(extra)} wrong emissions (counts {mult[i, extra[:3]]}, a {A[i, extra[:3]]})")
    assert np.array_equal(got[want].view(np.uint32), A[want].view(np.uint32)), "a key's distance differs from a_r"
    assert (out["counts"] == want.sum(1)).all() and out["pad_count"] == 0
    s.close()


# ---- 4. hit-queue flushes and candidate-buffer overflow -----------------------------------------------------------------
KINDS = (0, 1, 31, 32, 33, None, None, None, None, None, None, None)   # hits per query column; None = +inf (every row)


def _queue_data():
    """Query j of a special kind owns a block of 32 rows (64 for 33 hits: two warps) whose distances to it are far below
    everything else; +inf columns fill every warp's queue with 32 hits each, so queues of 256 and 176 entries flush
    inside a 32-column chunk at fill levels that are not multiples of 32."""
    rng = np.random.default_rng(21)
    dim, nq = 64, 256
    Q = (3.0 * rng.standard_normal((nq, dim))).astype(np.float32)
    kinds = [KINDS[j % len(KINDS)] for j in range(nq)]
    blocks, owner = [], {}
    for j, h in enumerate(kinds):
        if h:
            m = 64 if h == 33 else 32
            U = rng.standard_normal((m, dim))
            U /= np.linalg.norm(U, axis=1, keepdims=True)
            radius = rng.permutation(0.5 + 0.25 * np.arange(m))[:, None]
            owner[j] = sum(len(b) for b in blocks) + np.arange(m)
            blocks.append(Q[j] + radius * U)
    X = np.vstack(blocks + [3.0 * rng.standard_normal((203, dim))]).astype(np.float32)
    return X, Q, kinds, owner


@pytest.mark.parametrize("kern", KERNELS, ids=_kid)
def test_queue_flushes_and_overflowing_buffers_keep_every_hit(kern):
    X, Q, kinds, owner = _queue_data()
    n = len(X)
    s = _shard(X.shape[1], "l2", X)
    allow = np.ones(n, bool)
    A = _approx(s, Q, kern, n, allow)
    thr = np.full(len(Q), np.inf, np.float32)
    for j, h in enumerate(kinds):
        if h is not None:
            srt = np.sort(A[j])
            thr[j] = np.nextafter(srt[0], np.float32(-np.inf)) if h == 0 else srt[h - 1]
            if h:
                assert set(np.nonzero(A[j] <= thr[j])[0]) <= set(owner[j].tolist()), "the data misses its design"
    want = A <= thr[:, None]
    out = s.debug_gemm_rounds(Q, *kern, cap=_pow2(n), thresholds=thr)
    mult, _ = _hits(out, n)
    assert (mult == want).all(), f"{_kid(kern)}: lost {(want & (mult == 0)).sum()}, doubled {(mult > 1).sum()}, wrong {(~want & (mult > 0)).sum()}"
    # a buffer smaller than the hits: the count is the true total, the stored keys distinct true hits
    from mlvectordb_b200.shard import key_parts
    small = s.debug_gemm_rounds(Q, *kern, cap=100, thresholds=thr)
    assert np.array_equal(small["counts"], want.sum(1)), "the uncapped count is wrong"
    for j in range(len(Q)):
        m = min(int(small["counts"][j]), 100)
        d, r = key_parts(small["keys"][j, :m])
        assert len(set(r.tolist())) == m and want[j, r.astype(np.int64)].all(), f"q{j}: stored keys are not distinct true hits"
        assert np.array_equal(d.view(np.uint32), A[j, r.astype(np.int64)].view(np.uint32))
    s.close()


# ---- 5. rounds and refine_kernel against a numpy model -------------------------------------------------------------------
def _model(a, allow, thr0, rounds, kprime, cap):
    """One query through the rounds: a round appends the allowed rows of its tiles with a <= thr; refine keeps the k'
    smallest keys and sets thr = min(thr, the jrank-th key); flags bit 0 = overflow, bit 2 = the final round starved
    (fewer keys than jrank under a finite threshold) or its k'-th key lies above the threshold in force.
    -> (sorted keys, count, thr, flags), or None once a buffer overflowed (which keys survive is then a race)."""
    from mlvectordb_b200.shard import key_parts, make_keys
    keys = make_keys(a, np.arange(len(a)))
    kept, thr, flags, seen = np.empty(0, np.uint64), np.float32(thr0), 0, 0
    for i, (end, jrank) in enumerate(rounds):
        final = i + 1 == len(rounds)
        r = np.arange(seen * BM, min(end * BM, len(a)))
        r = r[allow[r] & (a[r] <= thr)]
        merged = np.sort(np.concatenate([kept, keys[r]]))
        if len(merged) > cap:
            return None
        d = key_parts(merged)[0]
        if len(merged) < jrank:
            if final and thr < np.inf:
                flags |= 4
            kept = merged
        else:
            if final and len(merged) >= kprime and not d[kprime - 1] <= thr:
                flags |= 4
            thr = np.minimum(thr, d[jrank - 1])
            kept = merged[:kprime]
        seen = end
    return kept, len(kept), thr, flags


def _schedules(tiles, A, allow):
    """name -> (rounds, kprime, cap, initial thresholds or None)."""
    srt = np.sort(np.where(allow[None, :], A, np.inf), axis=1)
    return {
        "plain rule": ([(8, KP), (20, KP), (tiles, KP)], KP, 1024, None),
        "predicted": ([(2, 32), (6, 40), (16, 64), (tiles, KP)], KP, 1024, None),
        "prediction fails the final check": ([(2, 2), (tiles, KP)], KP, 1024, None),
        "prediction starves": ([(2, 32), (tiles, KP)], KP, 1024, srt[:, 49]),
        "tight k'": ([(2, 32), (8, 32), (tiles, 32)], 32, 1024, None),
    }


@pytest.mark.parametrize("kern", [(1, 256), (2, 0), (3, 64)], ids=_kid)
@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
def test_rounds_and_refine_match_a_numpy_model(space, kern):
    from mlvectordb_b200.shard import key_parts
    n, dim, nq = 5000, 64, 40
    X = synthetic.rows(31, 0, n, dim, scaled=space != "l2")
    dead = np.arange(7, n, 17)
    s = _shard(dim, space, X, dead)
    Q = synthetic.queries(32, nq, dim)
    allow = np.ones(n, bool)
    allow[dead] = False
    A = _approx(s, Q, kern, n, allow)
    tiles = -(-n // BM)
    seen_flags = set()
    for name, (rounds, kprime, cap, thr0) in _schedules(tiles, A, allow).items():
        out = s.debug_gemm_rounds(Q, *kern, cap=cap, kprime=kprime, rounds=rounds, thresholds=thr0)
        for i in range(nq):
            m = _model(A[i], allow, np.inf if thr0 is None else thr0[i], rounds, kprime, cap)
            assert m is not None, f"{name}: the schedule overflows q{i}"
            keys, count, thr, flags = m
            assert out["counts"][i] == count and out["flags"][i] == flags, \
                f"{name} q{i}: count {out['counts'][i]} flags {out['flags'][i]}, model {count} {flags}"
            assert np.float32(out["thr"][i]).tobytes() == np.float32(thr).tobytes(), f"{name} q{i}: thr {out['thr'][i]!r}, model {thr!r}"
            assert np.array_equal(np.sort(out["keys"][i, :count]), keys), f"{name} q{i}: kept keys differ"
            seen_flags.add(int(flags))
    assert seen_flags >= {0, 4}, seen_flags
    # overflow: every row passes the first round's +inf threshold, 128 slots hold 128 of them
    out = s.debug_gemm_rounds(Q, *kern, cap=128, kprime=KP, rounds=[(tiles, KP)])
    assert (out["flags"] == 1).all() and (out["counts"] == KP).all()
    for i in range(nq):
        d, r = key_parts(out["keys"][i, :KP])
        assert len(set(r.tolist())) == KP and allow[r.astype(np.int64)].all() and (np.diff(out["keys"][i, :KP].astype(np.uint64)) > 0).all()
        assert np.array_equal(d.view(np.uint32), A[i, r.astype(np.int64)].view(np.uint32)) and out["thr"][i] == d[-1]
    s.close()
    # fewer rows than jrank: all kept; a finite initial threshold makes the final round starve (bit 2)
    Xs = X[:60]
    s = _shard(dim, space, Xs)
    As = _approx(s, Q, kern, 60, np.ones(60, bool))
    thr0 = np.where(np.arange(nq) % 2 == 0, np.inf, np.sort(As, axis=1)[:, 29]).astype(np.float32)
    out = s.debug_gemm_rounds(Q, *kern, cap=1024, kprime=KP, rounds=[(1, KP)], thresholds=thr0)
    assert np.array_equal(out["counts"], np.where(np.isinf(thr0), 60, 30)) and np.array_equal(out["flags"], np.where(np.isinf(thr0), 0, 4))
    assert np.array_equal(out["thr"].view(np.uint32), thr0.view(np.uint32))
    s.close()


# ---- 6. the certificate, end to end ------------------------------------------------------------------------------------
def _kprime(k, passes):
    if passes == 3:
        return (k + max(16, k // 4) + 31) // 32 * 32
    return (max(2 * k, k + 64) + 31) // 32 * 32


SPREADS = (0.1, 0.3, 1.0, 3.0, 10.0)
CROWD = 160                                # rows around a crowded query's k-th best: more than k' of every tier


def _crowds(space, dim, delta, nq, seed):
    """Background rows and queries; query i < 4 * len(SPREADS) also gets CROWD rows whose exact distances spread over
    SPREADS[i % 5] x delta * scale around one value.  -> (X, Q, crowded query ids)."""
    rng = np.random.default_rng(seed)
    Q = rng.standard_normal((nq, dim))
    bg = rng.standard_normal((2000, dim))
    crowds, ids = [], np.arange(4 * len(SPREADS))
    xmax_bg = np.linalg.norm(bg, axis=1).max()
    for i in ids:
        q, spread = Q[i], SPREADS[i % len(SPREADS)]
        qn = np.linalg.norm(q)
        qh = q / qn
        V = rng.standard_normal((CROWD, dim))
        V -= np.outer(V @ qh, qh)
        V /= np.linalg.norm(V, axis=1, keepdims=True)
        t = rng.uniform(-1, 1, CROWD)
        if space == "l2":
            rho0 = 0.3 * qn
            ds = delta * (max(xmax_bg, 2 * qn) + qn) ** 2
            C = q + np.sqrt(rho0 ** 2 + spread * ds * t / 2)[:, None] * V
        elif space == "ip":
            xmax = 1.5 * xmax_bg
            beta = 0.95 * xmax + spread * delta * xmax * t / 2
            C = beta[:, None] * qh + np.sqrt(xmax ** 2 - beta ** 2)[:, None] * 0.3 * V
        else:
            cos = 0.95 + spread * delta * t / 2
            C = cos[:, None] * qh + np.sqrt(1 - cos ** 2)[:, None] * V
        crowds.append(C)
    X = np.vstack([bg] + crowds)
    return X[rng.permutation(len(X))].astype(np.float32), Q.astype(np.float32), ids


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
def test_certificate_replay_per_tier_and_kernel(space):
    """Each tier forced (gemm_passes 1 / 2 / 3) on each kernel (gemm_wide 0 / 1): answers are the scan's bits, and the
    number of queries the tier certified equals a host replay of a_k' - delta * scale > e_k, with a_k' the k'-th smallest
    key of the kernel's own a_r and e_k the exact k-th distance."""
    k, dim, nq = 10, 64, 160
    for passes in (1, 2, 3):
        ld = dim
        X, Q, crowded = _crowds(space, dim, float(_delta_rel(passes, space == "l2", ld)), nq, seed=40 + passes)
        n = len(X)
        s = _shard(dim, space, X)
        s.set_tuning("gemm", 0)
        ref = s.search(Q, k)
        s.set_tuning("gemm", 1)
        s.set_tuning("gemm_passes", passes)
        _, scale = _exact_and_scale(s, Q)
        dsc = (_delta_rel(passes, space == "l2", ld) * scale[:, 0].astype(np.float32)).astype(np.float32)
        kp = _kprime(k, passes)
        outcomes = set()
        for wide in ((0, 1) if passes != 3 else (0,)):
            s.set_tuning("gemm_wide", wide)
            A = _approx(s, Q, (passes, 0 if wide else 256), n, np.ones(n, bool))
            akp = np.sort(A, axis=1)[:, kp - 1]
            ek = ref[0][:, k - 1]
            lhs = (akp - dsc).astype(np.float32)
            lhs64 = akp.astype(np.float64) - dsc.astype(np.float64)
            tol = 4 * np.spacing(np.maximum(np.abs(akp), np.abs(ek)))
            near = (np.abs(lhs - ek) <= tol) | (np.abs(lhs64 - ek) <= tol) | ((lhs > ek) != (lhs64 > ek))
            predicted = lhs > ek
            before = s.gemm_stats()
            got = s.search(Q, k)
            after = s.gemm_stats()
            d = {f: after[f] - before[f] for f in ("searches", "fallback_queries", "fast_queries", "half_queries")}
            assert d["searches"] == 1
            for a, b, what in zip(got, ref, ("dists", "rows", "counts")):
                assert np.array_equal(a, b), f"passes {passes} wide {wide}: {what} differ from the scan"
            certified = nq - d["fallback_queries"]
            assert d["fast_queries"] == (certified if passes != 3 else 0)
            assert d["half_queries"] == (certified if passes == 2 else 0)
            lo = int((predicted & ~near).sum())
            assert lo <= certified <= lo + int(near.sum()), \
                f"passes {passes} wide {wide}: {certified} certified, the replay says {lo} (+{int(near.sum())} within ulps)"
            outcomes |= set(predicted[crowded][~near[crowded]].tolist())
        assert outcomes == {True, False}, f"passes {passes}: only certified={outcomes} among the crowded queries"
        L, D = exact.knn(X, Q[crowded], k, space)
        for j, i in enumerate(crowded):
            msg = exact.check_topk_parity(got[1][i], got[0][i], L[j], D[j])
            assert msg is None, f"passes {passes} q{i}: {msg}"
        s.close()
