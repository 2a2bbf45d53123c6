"""CPU model of the int8 64-query pass (scan_umma_kernel<SEG, true>): the per-row int8 quantiser of store_convert_kernel,
the two-part int8 query of query_prep_kernel and the epilogue's fp32 key sa8 * (s1 * acc1 + s2 * acc2) + sb, checked
against the allowance finish.cu certifies with; then the certificate model of tests/test_certificate_model.py run on
int8 keys."""
import os
import sys

import numpy as np
from hypothesis import given, settings, strategies as st

from oracle import knn

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_certificate_model import _finish, _model_search  # noqa: E402

F32 = np.float32


def _quantise(A):
    """int8 codes and scale per row: s = max|a| / 127 (float32), code = rint(a / s) in [-127, 127]; zero rows: 0, 0."""
    A = np.asarray(A, dtype=F32)
    s = (np.abs(A).max(axis=1) / F32(127)).astype(F32)
    safe = np.where(s > 0, s, F32(1))[:, None]
    c = np.where(s[:, None] > 0, np.clip(np.rint(A / safe), -127, 127), 0).astype(np.int64)
    return c, s


def _query_parts(q_hat):
    """q_hat ~ s1 q1 + s2 q2: q2 codes the float32 residual q_hat - s1 q1; rho_q of the pair in fp64."""
    q_hat = np.asarray(q_hat, dtype=F32)[None, :]
    q1, s1 = _quantise(q_hat)
    r = (q_hat - s1[:, None] * q1.astype(F32)).astype(F32)
    q2, s2 = _quantise(r)
    qh = q_hat[0].astype(np.float64)
    approx = float(s1[0]) * q1[0].astype(np.float64) + float(s2[0]) * q2[0].astype(np.float64)
    h = np.sqrt((qh * qh).sum())
    rho_q = float(np.sqrt(((qh - approx) ** 2).sum()) / h) if h > 0 else 0.0
    return q1[0], q2[0], F32(s1[0]), F32(s2[0]), rho_q


def _int8_keys(X, q_hat, sa8, sb):
    """the epilogue: exact integer dots, then fp32 s1 * acc1 + s2 * acc2 (fma), * sa8 + sb (fma)."""
    x8, _ = _quantise(X)
    q1, q2, s1, s2, rho_q = _query_parts(q_hat)
    a1 = (x8 @ q1).astype(F32)                       # |acc| < 2^24: exact in float32
    a2 = (x8 @ q2).astype(F32)
    inner = (s1.astype(np.float64) * a1 + (s2 * a2).astype(np.float64)).astype(F32)      # fma: one rounding
    key = (inner.astype(np.float64) * sa8.astype(np.float64) + sb.astype(np.float64)).astype(F32)
    return key, rho_q


def _rho_x8(X):
    x8, s = _quantise(X)
    X64 = X.astype(np.float64)
    xn = np.sqrt((X64 * X64).sum(axis=1))
    res = np.sqrt(((X64 - s[:, None].astype(np.float64) * x8) ** 2).sum(axis=1))
    return float(np.where(xn > 0, res / np.where(xn > 0, xn, 1), 0).max()), xn, s


def _rows(rng, n, d, kind, scale):
    X = (rng.standard_normal((n, d)) * scale * rng.uniform(0.2, 3.0, size=(n, 1))).astype(F32)
    if kind == "zero":
        X[rng.integers(0, n, size=max(1, n // 5))] = 0.0
    elif kind == "tiny":
        X[rng.integers(0, n, size=max(1, n // 5))] *= F32(1e-30)
    elif kind == "outlier":                          # one huge channel: every other element quantises coarsely
        X[rng.integers(0, n, size=max(1, n // 5)), int(rng.integers(0, d))] = F32(300.0 * scale)
    return X


@settings(max_examples=40, deadline=None, derandomize=True)
@given(st.integers(1, 120), st.sampled_from([768, 1024]), st.integers(0, 2**31 - 1), st.sampled_from([1e-3, 1.0, 50.0]),
       st.sampled_from(["plain", "zero", "tiny", "outlier"]))
def test_int8_allowance_bounds_the_int8_scan_error_cosine(n, d, seed, scale, kind):
    """|int8 key - exact cosine| <= eps = rho_x8 (1 + rho_q8) + rho_q8 + d 2^-23 (finish.cu, acc_allowance unchanged)
    with sa8 = s_x / ||x||, for zero rows, tiny rows and rows with one huge outlier channel."""
    rng = np.random.default_rng(seed)
    X = _rows(rng, n, d, kind, scale)
    q = rng.standard_normal(d).astype(F32)
    q64 = q.astype(np.float64)
    q_hat = (q64 / np.sqrt((q64 * q64).sum())).astype(F32)
    rho_x, xn, s = _rho_x8(X)
    sa8 = np.where(xn > 0, s.astype(np.float64) / np.where(xn > 0, xn, 1), 0).astype(F32)
    key, rho_q = _int8_keys(X, q_hat, sa8, np.zeros(n, dtype=F32))
    eps = (rho_x * (1.0 + rho_q) + rho_q + d * 2.0 ** -23) * 1.0001
    exact = knn.cos64(X, q)
    assert np.abs(key.astype(np.float64) - exact).max() <= eps
    assert rho_q <= 1e-4                              # two parts: ~(1/254)^2 relative
    if kind != "outlier":
        assert rho_x <= 0.03                          # unit-scale rows stay under the AUTO limit RASS_INT8_RHO_MAX


@settings(max_examples=40, deadline=None, derandomize=True)
@given(st.integers(1, 120), st.sampled_from([768, 1024]), st.integers(0, 2**31 - 1), st.sampled_from([1e-2, 1.0, 20.0]),
       st.sampled_from(["plain", "zero", "tiny", "outlier"]))
def test_int8_allowance_bounds_the_int8_scan_error_l2(n, d, seed, scale, kind):
    """Same for L2: sa8 = s_x, key = sa8 * dot - fl32(||x||^2 / 2) against the exact surrogate x.q - ||x||^2 / 2; the
    allowance scales with max ||x|| * ||q|| and adds the rounding of the per-row offset (finish.cu)."""
    rng = np.random.default_rng(seed)
    X = _rows(rng, n, d, kind, scale)
    q = (rng.standard_normal(d) * rng.uniform(0.1, 4.0)).astype(F32)
    q64 = q.astype(np.float64)
    qn = float(np.sqrt((q64 * q64).sum()))
    rho_x, xn, s = _rho_x8(X)
    X64 = X.astype(np.float64)
    n2 = (X64 * X64).sum(axis=1)
    sb = (-0.5 * n2).astype(F32)
    key, rho_q = _int8_keys(X, q, s, sb)
    xm = float(xn.max())
    e = rho_x * (1.0 + rho_q) + rho_q + d * 2.0 ** -23
    eps = (e * xm * qn * 1.0001 + 6.0e-8 * xm * xm) * 1.0001
    exact = X64 @ q64 - 0.5 * n2
    assert np.abs(key.astype(np.float64) - exact).max() <= eps


@settings(max_examples=60, deadline=None, derandomize=True)
@given(st.integers(0, 2**31 - 1), st.sampled_from([1, 10, 32, 100]), st.sampled_from([2, 5, 16]),
       st.sampled_from([(256, 32), (512, 128)]), st.booleans(), st.sampled_from(["iid", "cluster", "dups"]))
def test_certified_means_exact_on_int8_keys(seed, k, n_segs, seg_keep, seeded, kind):
    """The scan -> pool -> certificate model on int8 keys with the int8 allowance: whenever the certificate holds, the
    re-ranked candidates are the exact top-k (random, clustered and duplicate-laden rows)."""
    rng = np.random.default_rng(seed)
    n, d = int(rng.integers(300, 4000)), 64
    X = rng.standard_normal((n, d)).astype(F32)
    q = rng.standard_normal(d).astype(F32)
    if kind == "cluster":
        lo = int(rng.integers(0, n - 200))
        X[lo:lo + 200] = (q[None, :] + 0.05 * rng.standard_normal((200, d))).astype(F32)
    elif kind == "dups":
        X[rng.integers(0, n, size=40)] = X[int(rng.integers(0, n))]
    q64 = q.astype(np.float64)
    q_hat = (q64 / np.sqrt((q64 * q64).sum())).astype(F32)
    rho_x, xn, s = _rho_x8(X)
    sa8 = (s.astype(np.float64) / xn).astype(F32)
    key, rho_q = _int8_keys(X, q_hat, sa8, np.zeros(n, dtype=F32))
    eps = float(F32((rho_x * (1.0 + rho_q) + rho_q + d * 2.0 ** -23) * 1.0001))
    exact = knn.cos64(X, q)
    seg, keep = seg_keep
    seed_rows = rng.choice(n, size=min(n, 256), replace=False) if seeded else None
    pools, thr = _model_search(key, exact, k, n_segs, 64, seg, keep, seed_rows, keep + 8, rng)
    top, certified = _finish(pools, thr, eps, exact, k)
    want = np.lexsort((np.arange(n), -exact))[:k]
    if certified:
        assert top.tolist() == want.tolist()
