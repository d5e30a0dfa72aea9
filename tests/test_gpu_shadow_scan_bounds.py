"""The shadow scan's fp16 error bound and its certificate, checked against fp64 (csrc/scan_kernel.cuh, scan_kernel_half).

Two claims rest on delta_rel (gemm_kernel.cuh, gemm_delta_rel_f16): |approx - exact| <= delta_rel * scale for every row.
The kNN certificate accepts an answer when a_32 - delta * scale > exact_k, and range mode re-scores only rows with
approx <= r + delta * scale.  mlv_index_debug_half_scan exposes the approximate distances of the very consumers a search
runs (FMA or mma.sync), so the bound is measured directly, and the certificate and the range margin are replayed on data
built to sit within a few delta * scale of the decision."""
import numpy as np
import pytest

from oracle import exact, synthetic

pytestmark = pytest.mark.gpu

KP = 32                                  # candidates the shadow scan keeps (HALF_SCAN_KPRIME)
MMA_MAX_DIM = 3264                       # longest rows (a multiple of 64) with two 16-row stages in 227 KB of shared memory


def _shard(dim, space, **kw):
    from mlvectordb_b200 import DeviceShard
    return DeviceShard(dim, space, **kw)


def _worst(rng, shape):
    """Round-to-nearest worst case: every value just below a half step of 11 significant bits, positive, 2^-2..2^2."""
    step = 2.0 ** -10
    return ((1.0 + rng.integers(0, 1024, shape) * step + 0.5 * step * (1 - 2.0 ** -12))
            * 2.0 ** rng.integers(-2, 3, shape)).astype(np.float32)


def _snap(x):
    """Move every value to just below a half step of its 11-significant-bit grid (the worst case survives the shadow's
    power-of-two scale)."""
    x = np.asarray(x, np.float64)
    m, e = np.frexp(np.abs(x))                           # |x| = m 2^e, m in [0.5, 1)
    step = np.ldexp(1.0, e - 11)
    y = (np.floor(np.abs(x) / step) + 0.5 * (1 - 2.0 ** -12)) * step
    return (np.sign(x) * np.where(x == 0, 0, y)).astype(np.float32)


def _exact(s, q):
    """fp64 distances of the stored rows (cosine: as normalised by the index) to the prepared query."""
    X = s.export_rows().astype(np.float64)
    q = np.asarray(q, np.float64)
    if s.space == "l2":
        return ((X - q) ** 2).sum(1)
    if s.space == "cosine":
        nq = np.sqrt((q * q).sum())
        q = q / nq if nq > 0 else q
    return 1.0 - X @ q


def _measure(s, q):
    """max |approx - exact| / (delta * scale) over the live rows of one query (0 when scale is 0)."""
    A, info = s.debug_half_scan(q)
    live = np.isfinite(A)
    err = np.abs(A[live].astype(np.float64) - _exact(s, q)[live])
    lim = float(info["delta_rel"]) * float(info["scale"])
    assert not np.isnan(A).any()
    if lim == 0:
        assert err.max() == 0
        return 0.0, info
    return float(err.max() / lim), info


BOUND_CASES = [(96, 1), (100, 1), (128, 1), (768, 1), (MMA_MAX_DIM, 1), (768, 0)]   # (dim, scan_half_mma)


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("dim,mma", BOUND_CASES)
def test_shadow_scan_distances_stay_inside_the_certificate_bound(space, dim, mma):
    n = 2048 if dim <= 768 else 512
    rng = np.random.default_rng(dim + 7 * mma)
    kind = 2 if (dim % 64 == 0 and mma) else 1
    benign = (synthetic.rows(4, 0, n, dim, scaled=True), synthetic.queries(4, 3, dim))
    zero_row = benign[0].copy()
    zero_row[17] = 0
    cases = {"worst": (_worst(rng, (n, dim)), _worst(rng, (3, dim))),
             "benign": benign,
             "huge rows, tiny query": (benign[0] * np.float32(3.0e6), benign[1] * np.float32(2.0e-7)),
             "12 binades": (benign[0] * (2.0 ** rng.integers(-12, 1, (n, 1))).astype(np.float32), benign[1]),
             "zero query, zero row": (zero_row, np.vstack([np.zeros((1, dim), np.float32), benign[1][:1]]))}
    for name, (X, Q) in cases.items():
        s = _shard(dim, space)
        s.add(X)
        s.set_tuning("scan_half_mma", mma)
        worst = 0.0
        for q in Q:
            frac, info = _measure(s, q)
            assert info["consumers"] == kind and info["overflow"] == 0
            assert frac < 1.0, f"{space} dim {dim} {name}: |approx - exact| reached {frac:.3f} of delta * scale"
            worst = max(worst, frac)
        print(f"shadow scan bound: {space} dim {dim} consumers {'mma' if kind == 2 else 'fma'} {name}: {worst:.3f} of delta")
        if name == "worst" and space != "cosine":
            # on a B200 this input uses 0.16 - 0.21 (FMA) / 0.21 - 0.39 (mma) of delta: far less means the test is vacuous.
            # (cosine rows and queries are normalised by the index, which moves them off the half-step positions)
            floor = 0.12 if kind == 1 else 0.2
            assert worst > floor, f"worst-case input only reached {worst:.3f} of delta"
        s.close()


@pytest.mark.parametrize("space", ["l2", "ip"])
@pytest.mark.parametrize("dim", [100, 768])
def test_rows_appended_after_the_scale_froze_stay_inside_the_bound(space, dim):
    """The shadow's scale freezes when it is built; rows appended later up to 3.9x the largest norm still fit fp16 (two
    bits of headroom): no overflow, max |x|^2 grows, and the bound holds with the grown scale."""
    n = 2048
    X = synthetic.rows(5, 0, n, dim, scaled=True)
    Q = synthetic.queries(5, 3, dim)
    s = _shard(dim, space, capacity=n + 64)
    s.add(X)
    _, before = s.debug_half_scan(Q[0])                   # freezes the scale
    xmax = float(np.sqrt(before["max_norm2"]))
    spike = np.zeros((1, dim), np.float32)
    spike[0, 3] = np.float32(3.9 * xmax)                   # one component at 3.9x the frozen largest norm
    s.add(np.vstack([spike, X[:31] * np.float32(3.9)]))
    for q in Q:
        frac, info = _measure(s, q)
        assert info["overflow"] == 0 and info["x_unscale"] == before["x_unscale"]
        assert info["max_norm2"] > 10 * before["max_norm2"]
        assert frac < 1.0, f"{space} dim {dim}: {frac:.3f} of delta after the late rows"
    s.close()


# ---- adversarial neighbourhoods -------------------------------------------------------------------------------------
SPREADS = (0.1, 0.3, 1.0, 3.0, 10.0)
M = 48                                    # rows spread around the k-th, more than the 32 candidates


def _crowd(space, dim, spread, seed, n_bg=2000):
    """Rows whose exact distances to q are spread over `spread` x delta * scale around a common value (worst-case
    rounding components), behind background rows far away.  Returns (X, q)."""
    rng = np.random.default_rng(seed)
    q = _worst(rng, (dim,)).astype(np.float64)
    qn = np.linalg.norm(q)
    qh = q / qn
    bg = _worst(rng, (n_bg, dim)) * rng.choice(np.float32([-1, 1]), (n_bg, dim))
    V = rng.standard_normal((M, dim))
    V -= np.outer(V @ qh, qh)
    V /= np.linalg.norm(V, axis=1, keepdims=True)
    t = rng.uniform(-1, 1, M)
    e = 2.0 ** -10 * (1 + 2.0 ** -12) + dim * 2.0 ** -22
    if space == "l2":
        delta = 0.5 * e
        rho0 = 0.15 * qn
        xmax = max(np.linalg.norm(bg, axis=1).max(), qn + rho0)
        ds = delta * (xmax + qn) ** 2
        rho = np.sqrt(rho0 ** 2 + spread * ds * t / 2)
        C = q + rho[:, None] * V
    elif space == "ip":
        xmax = 1.5 * np.linalg.norm(bg, axis=1).max()
        ds = e * xmax * qn
        beta = (0.95 * xmax + spread * ds * t / 2 / qn)          # dot = beta |q|
        C = beta[:, None] * qh + np.sqrt(np.maximum(xmax ** 2 - beta ** 2, 0))[:, None] * 0.3 * V
    else:
        ds = e
        cos = 0.95 + spread * ds * t / 2
        C = cos[:, None] * qh + np.sqrt(1 - cos ** 2)[:, None] * V
    X = np.vstack([bg, _snap(C)]).astype(np.float32)
    perm = rng.permutation(len(X))                        # neighbours spread over the tiles
    return X[perm], q.astype(np.float32)


def _keys_order(A):
    """Row order by the kernel's key: (approximate distance, row)."""
    return np.lexsort((np.arange(len(A)), A))


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("dim,mma", [(96, 1), (128, 1), (128, 0)])
def test_certificate_replay_on_adversarial_neighbourhoods(space, dim, mma):
    """Replays the certificate from the debug view and compares it with the kernel's decision; whenever the kernel
    certified, no row outside the 32 candidates beats the returned k-th in fp64; answers are the fp32 scan's bits."""
    outcomes, crossed = set(), False
    for si, spread in enumerate(SPREADS):
        X, q = _crowd(space, dim, spread, seed=100 * si + dim + mma)
        s = _shard(dim, space)
        s.add(X)
        s.set_tuning("scan_half_mma", mma)
        A, info = s.debug_half_scan(q)
        ex = _exact(s, q)
        order = _keys_order(A)
        cand = order[:KP]
        a32 = np.float32(A[order[KP - 1]])
        dsc = np.float32(np.float32(info["delta_rel"]) * np.float32(info["scale"]))
        outside = np.ones(len(A), bool)
        outside[cand] = False
        crossed |= bool(ex[outside].min() < ex[cand].max())
        for k in (1, 10, 16):
            s.set_tuning("scan_half", 0)
            ref = s.search(q[None], k)
            s.set_tuning("scan_half", 1)                    # (also resets the sit-out state)
            st0 = s.gemm_stats()
            got = s.search(q[None], k)
            st1 = s.gemm_stats()
            assert st1["half_scan_queries"] - st0["half_scan_queries"] == 1
            uncert = st1["half_scan_uncertified"] - st0["half_scan_uncertified"]
            assert all(np.array_equal(g, r) for g, r in zip(got, ref)), f"{space} spread {spread} k {k}: differs from the fp32 scan"
            ek = np.float32(ref[0][0, k - 1])
            # the kernel's comparison, fused or not: skip only when it is within an ulp of equality
            lhs = (np.float32(a32 - dsc), np.float32(np.float64(a32) - np.float64(dsc)))
            if all(abs(float(v) - float(ek)) > float(np.spacing(ek)) for v in lhs) and (lhs[0] > ek) == (lhs[1] > ek):
                predicted = bool(lhs[0] > ek)
                assert predicted == (uncert == 0), f"{space} spread {spread} k {k}: certificate predicted {predicted}, kernel {uncert == 0}"
            outcomes.add(uncert == 0)
            if uncert == 0:
                kth = ex[int(ref[1][0, k - 1])]
                tol = 4 * np.spacing(np.float32(abs(kth) + 1e-30))
                assert ex[outside].min() >= kth - tol, f"{space} spread {spread} k {k}: a row outside the candidates beats the certified k-th"
            L, D = exact.knn(X, q[None], k, space)
            assert exact.check_topk_parity(got[1][0], got[0][0], L[0], D[0]) is None
        s.close()
    assert outcomes == {True, False}, f"only certified={outcomes} occurred: the spreads miss the decision"
    assert crossed, "approximate and exact order never disagree across the candidate boundary"


@pytest.mark.parametrize("space", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("dim,mma", [(96, 1), (128, 1)])
def test_range_margin_keeps_every_true_hit(space, dim, mma):
    """Range mode re-scores rows with approx <= r + delta * scale: every row with exact <= r must be among them, at radii on
    actual distances and half a margin either side, with tombstones and a streamed filter; the hit lists are the fp32
    scan's bits and the fp64 oracle's."""
    for si, spread in enumerate((0.3, 3.0)):
        X, q = _crowd(space, dim, spread, seed=500 + 10 * si + dim)
        n = len(X)
        s = _shard(dim, space)
        s.add(X)
        s.set_tuning("scan_half_mma", mma)
        s.set_tuning("gather", 0)
        dead = np.arange(5, n, 9, dtype=np.uint64)
        s.mark_deleted(dead)
        mask = np.random.default_rng(si).random(n) < 0.7
        pf = s.prepare_filter(mask)
        allow = mask.copy()
        allow[dead.astype(np.int64)] = False
        A, info = s.debug_half_scan(q)
        assert not np.isfinite(A[dead.astype(np.int64)]).any()
        ex = _exact(s, q)
        margin = np.float32(np.float32(info["delta_rel"]) * np.float32(info["scale"]))
        s.set_tuning("scan_half", 0)
        d_ref = s.search(q[None], 40)[0][0]
        radii = []
        for j in (0, 15, 39):
            r = np.float32(d_ref[j])
            radii += [r, np.float32(r - margin / 2), np.float32(r + margin / 2)]
        for r in radii:
            live = np.isfinite(A)
            true_hits = live & (ex <= r)
            assert (A[true_hits] <= np.float32(r + margin)).all(), f"{space} r {r}: a true hit is outside the re-score margin"
            for filt, allowed in ((None, live), (pf, allow)):
                s.set_tuning("scan_half", 0)
                ref = s.range_search(q[None], float(r), filt, max_hits=4096)
                s.set_tuning("scan_half", 1)
                got = s.range_search(q[None], float(r), filt, max_hits=4096)
                assert np.array_equal(got[0][0], ref[0][0]) and np.array_equal(got[0][1], ref[0][1])
                L, _ = exact.range_search(X, q[None], float(r), space, allow=allowed)
                tol = 1e-5 * abs(float(r)) + 1e-6
                for row in set(got[0][1].tolist()) ^ set(np.asarray(L[0]).tolist()):
                    assert abs(ex[row] - float(r)) <= 2 * tol, f"row {row} is not at the radius"
        pf.close()
        s.close()


@pytest.mark.parametrize("space", ["l2", "cosine"])
@pytest.mark.parametrize("dim", [96, 128])
def test_identical_rows_across_the_candidate_boundary(space, dim):
    """40 identical nearest rows, more than the 32 candidates: the answer is the k lowest row ids with identical scores,
    whether the kernel certifies (it cannot tell them apart) or falls back."""
    rng = np.random.default_rng(dim)
    X = synthetic.rows(6, 0, 4000, dim, scaled=True)
    q = synthetic.queries(6, 1, dim)[0]
    twin = q + np.float32(0.01) * rng.standard_normal(dim).astype(np.float32)
    ids = np.sort(rng.choice(len(X), 40, replace=False))
    X[ids] = twin
    s = _shard(dim, space)
    s.add(X)
    for k in (10, 16):
        s.set_tuning("scan_half", 0)
        ref = s.search(q[None], k)
        s.set_tuning("scan_half", 1)
        d, r, c = s.search(q[None], k)
        assert all(np.array_equal(g, h) for g, h in zip((d, r, c), ref))
        assert r[0].tolist() == ids[:k].tolist()
        assert (d[0] == d[0, 0]).all()
    s.close()
