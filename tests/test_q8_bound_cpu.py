"""The int8 shadow scan's error bound, restated in numpy (csrc/scan_kernel.cuh: q8_delta, the query's digits in scan_body;
csrc/gemm_kernel.cuh: convert_rows_q8_kernel).  A row is x = s_x x^ + e (one scale per row, |e| <= e_x <= E), the query
q = t (h + l / 254) + r, and the consumers compute a = s_x t (D_h + D_l / 254) from exact integer sums in fp32.  On random
rows and on rows built to defeat the bound -- every element half a step from its digit, the query aligned with the row's
residual so that every product has one sign, row norms spread 100x -- |a - exact| <= delta, exact in fp64."""
import numpy as np
import pytest

F = np.float32


def _f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32)


def quantize_rows(X):
    """-> digits [n, d] int8, s_x [n], e_x [n] (rounded up as the kernel does), like convert_rows_q8_kernel."""
    X = _f32(X)
    d = X.shape[1]
    m = np.abs(X).max(axis=1)
    s = _f32(m / F(127))
    inv = np.where(m > 0, _f32(F(127) / np.where(m > 0, m, F(1))), F(0)).astype(np.float32)
    dq = np.clip(np.rint(_f32(X * inv[:, None])), -127, 127).astype(np.float32)
    r = _f32(X.astype(np.float64) - s.astype(np.float64)[:, None] * dq)          # one fma: exact product, one rounding
    ss = _f32((r.astype(np.float64) ** 2).sum(axis=1))
    e = _f32(np.sqrt(ss) * (1.0 + (d + 4) * 2.0 ** -22) + 2.0 ** -60)
    return dq.astype(np.int8), s, e


def quantize_query(q):
    """-> h, l int8 digits, t, |r| and t (|h| + |l| / 254) rounded up as the kernel does."""
    q = _f32(q)
    d = q.shape[0]
    m = F(np.abs(q).max())
    t = _f32(m / F(127))
    inv = _f32(F(127) / m) if m > 0 else F(0)
    tl = _f32(t * _f32(1.0 / 254.0))
    h = np.clip(np.rint(_f32(q * inv)), -127, 127).astype(np.float32)
    r1 = _f32(q.astype(np.float64) - float(t) * h)
    l = np.clip(np.rint(_f32(_f32(r1 * inv) * F(254))), -127, 127).astype(np.float32)
    r = _f32(r1.astype(np.float64) - float(tl) * l)
    rn = float(np.sqrt(np.sum(r.astype(np.float64) ** 2))) * (1 + d * 2.0 ** -23) + float(t) * np.sqrt(d) * 2.0 ** -22
    tq = float(t) * (np.linalg.norm(h) + np.linalg.norm(l) / 254.0) * 1.0001
    return h.astype(np.int8), l.astype(np.int8), float(t), F(rn), F(tq)


def q8_delta(l2, d, xmax, E, qn, rn, tq):
    """scan_kernel.cuh q8_delta, in fp32."""
    A = F(xmax) + F(E)
    dot = F(E) * F(qn) + A * F(rn)
    eps = F(d + 64) * F(2.0 ** -22)
    if not l2:
        return float(dot + eps * A * (F(qn) + F(tq)) + F(2.0 ** -22))
    w = A + F(qn) + F(tq)
    return float(F(2) * dot + F(2) * eps * w * w)


def approx(dq, s, h, l, t, metric, xn, qn2):
    """What the consumers compute per row: exact int32 sums, then the fp32 form."""
    Dh = _f32(dq.astype(np.int64) @ h.astype(np.int64))
    Dl = _f32(dq.astype(np.int64) @ l.astype(np.int64))
    sm = _f32(s * _f32(Dh + _f32(Dl * _f32(1.0 / 254.0))))
    if metric == "l2":
        return _f32(xn.astype(np.float64) + float(qn2) - 2.0 * float(t) * sm.astype(np.float64))
    return _f32(1.0 - float(t) * sm.astype(np.float64))


def check(X, q, metric):
    """max |a - exact| / delta over the rows (exact in fp64)."""
    X = _f32(X)
    q = _f32(q)
    if metric == "cosine":
        X = _f32(X / np.linalg.norm(X.astype(np.float64), axis=1, keepdims=True))
        q = _f32(q / np.linalg.norm(q.astype(np.float64)))
    d = X.shape[1]
    dq, s, e = quantize_rows(X)
    h, l, t, rn, tq = quantize_query(q)
    xn = _f32((X.astype(np.float64) ** 2).sum(axis=1))
    qn2 = _f32((q.astype(np.float64) ** 2).sum())
    xmax = 1.0 if metric == "cosine" else float(np.sqrt(F(xn.max())))
    delta = q8_delta(metric == "l2", d, xmax, float(e.max()), float(np.sqrt(qn2)), rn, tq)
    a = approx(dq, s, h, l, t, metric, xn, qn2).astype(np.float64)
    X64, q64 = X.astype(np.float64), q.astype(np.float64)
    exact = ((X64 - q64) ** 2).sum(axis=1) if metric == "l2" else 1.0 - X64 @ q64
    return float(np.abs(a - exact).max() / delta)


def half_step_rows(rng, n, d, spread=1.0):
    """Every element (j + 1/2) s: the largest rounding residual per digit; one element at 127 s fixes the scale."""
    j = rng.integers(0, 126, size=(n, d)).astype(np.float64) + 0.5
    X = j * rng.choice([-1.0, 1.0], size=(n, d))
    X[:, 0] = 127.0
    s = 10.0 ** rng.uniform(-np.log10(spread) / 2, np.log10(spread) / 2, size=(n, 1)) / 127.0
    return X * s


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("d", [96, 128, 768])
def test_random_rows_within_the_bound(metric, d):
    rng = np.random.default_rng(d)
    X = rng.uniform(-1, 1, size=(4000, d)) * rng.uniform(0.5, 1.0, size=(4000, 1))
    for _ in range(4):
        q = rng.standard_normal(d)
        assert check(X, q, metric) <= 1.0


@pytest.mark.parametrize("metric", ["l2", "ip", "cosine"])
@pytest.mark.parametrize("d", [96, 128, 768])
def test_adversarial_rows_within_the_bound(metric, d):
    rng = np.random.default_rng(100 + d)
    spread = 1.0 if metric == "cosine" else 100.0
    X = half_step_rows(rng, 2000, d, spread)
    worst = 0.0
    for i in range(8):
        # the query along one row's residual: every product e_i q_i has the same sign (Cauchy-Schwarz is tight)
        dq, s, _ = quantize_rows(X[i:i + 1])
        res = X[i] - s[0] * dq[0].astype(np.float64)
        q = np.sign(res) * (1.0 + 0.1 * rng.random(d))
        if i % 2:
            q = q + X[i] / np.abs(X[i]).max()          # ... plus the row itself: a near neighbour
        worst = max(worst, check(X, q, metric))
    assert worst <= 1.0, worst


def test_query_residual_digit_is_small():
    """The second digit leaves a query residual about 254 times smaller than one digit would."""
    rng = np.random.default_rng(3)
    q = rng.standard_normal(768)
    h, l, t, rn, _ = quantize_query(q)
    r_one = np.linalg.norm(q - t * h.astype(np.float64))
    assert rn < r_one / 100


def test_zero_rows_and_query_are_exact():
    X = np.zeros((4, 128))
    X[1, 5] = 0.25
    dq, s, e = quantize_rows(X)
    assert s[0] == 0 and (dq[0] == 0).all() and e[0] < 1e-17
    assert check(X, np.zeros(128), "ip") <= 1.0
