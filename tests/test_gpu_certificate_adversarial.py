"""The kNN certificate end to end on corpora built to defeat the scan shadows.

Every kNN answer rests on one inequality in finish_kernel (finish.cu): t + eps < s_k, with
eps = rho_x (1 + rho_q) + rho_q + dim_pad 2^-23 (L2: times max||x|| ||q||, plus 6e-8 max||x||^2).  On ordinary data the
shadow's ranking already puts the true top-k inside the rerank window, so eps decides nothing.  The corpora here are
built so that it does:

* Winners have the highest exact keys, and every component of theirs sits just off a rounding midpoint of the shadow,
  on the side that rounds the component's contribution to the key *down*; decoys have exact keys a fraction of eps
  lower and round *up*.  The shadow then ranks every decoy above every winner, each off by most of eps.
* The int8 shadow: one anchor channel pins max|x| = A, so s_x = A / 127 is known, and every other component is
  s_x (c +- 0.48).  The bf16 shadow: components half a bf16 step (less 2 %) above a bf16 value; the queries' own
  components sit just off bf16 midpoints too, and winners carry their larger level where the query rounds towards
  zero, decoys where it rounds away, so the query's rounding (rho_q) pushes the same way as the rows'.
* A few tuning channels set each row's exact key to a chosen target (one scalar solved per row); the anchor and the
  query's norm channel are zero in the other operand.
* Regime (a), "window": the rows are scattered, so no segment of the candidate pool holds more than a couple of them;
  the winners stay in the pool and the rerank has to reorder them.  Regime (b), "dropped": each query's rows are
  adjacent, three decoys to a winner, in whole 128-row tiles (and, for queries 0 and 1, over three periods of the
  streaming scan's row interleave), so every segment that sees them keeps only decoys, the winners leave the pool
  and the first pass must not certify.

The CPU tests prove each corpus legal (every row's model error <= the eps finish.cu computes), near the bound
(winners and decoys off by >= eps / 2) and adversarial (the model's top-k shares at most k / 2 ids with the exact
one).  The GPU tests check that the kernels' own keys rank decoys above winners, then that every path returns the
fp64 oracle's ids.
"""
import functools
import math
import os
import sys
import zlib

import numpy as np
import pytest

from oracle import knn, synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from test_certificate_model import _bf16  # noqa: E402
from test_int8_scan_cpu import _query_parts, _quantise, _rho_x8  # noqa: E402

F32 = np.float32
KS = (1, 10, 32, 100)
RHO8_MAX = 0.03          # RASS_INT8_RHO_MAX (engine.cu): AUTO scans the int8 shadow only at or below it
NT_OF_D = {100: 8}       # tuning channels 2 .. NT + 1 (32, fewer at small d); channel 0 = anchor, 1 = the query's norm
MARGIN = 0.04            # bf16: distance from the midpoint, in half steps (rint is half-to-even: stay clear of it)
FRAC8 = 0.48             # int8: |x| / s_x = c + 0.48 (rounds to c) or c + 0.52 (rounds to c + 1)
TILE = 128               # rows of a tcgen05 tile: one tile is read by one CTA into one segment
STREAM_PERIOD = 148 * 2 * 8 * 4   # rows between two visits of a streaming-scan CTA (148 SMs, 2 CTAs each, 8 warps, 4 rows)
LONG_BLOCK = 3 * STREAM_PERIOD    # queries 0 and 1 in regime (b): every streaming CTA sees >= 72 of their decoys
W_FRAC = (0.02, 0.12)    # winners' exact keys: kappa0 + eps * U(W_FRAC)
D_FRAC = (0.0, 0.10)     # decoys' exact keys:  kappa0 - eps * U(D_FRAC)
N_ADV_A = 100            # regime (a): winners and decoys per query
T_REF_COS, T_REF_L2 = 0.35, 0.6   # where the tuning channels sit for the centre key (fractions of their scale)


class Spec:
    def __init__(self, name, shadow, metric, d, regime, qnorm=1.0, level8=24, n_bg=24000):
        self.name, self.shadow, self.metric, self.d, self.regime = name, shadow, metric, d, regime
        self.qnorm, self.level8, self.n_bg = qnorm, level8, n_bg
        self.dim_pad = (d + 255) // 256 * 256

    def __repr__(self):
        return self.name


COS, L2 = knn.COSINE, knn.L2
# L2 query norms are powers of two near 1e-2, 1 and 1e2, so the queries' rounding positions survive the scaling
SPECS = [
    Spec("i8-cos-1024-a", "i8", COS, 1024, "a"),
    Spec("i8-cos-1024-b", "i8", COS, 1024, "b"),
    Spec("bf16-cos-1024-a", "bf16", COS, 1024, "a"),
    Spec("bf16-cos-1024-b", "bf16", COS, 1024, "b"),
    Spec("i8-l2-1024-a-q128", "i8", L2, 1024, "a", qnorm=128.0),
    Spec("bf16-l2-1024-b-q128", "bf16", L2, 1024, "b", qnorm=128.0),
    Spec("i8-l2-768-a-q1", "i8", L2, 768, "a", qnorm=1.0),
    Spec("bf16-l2-768-a-q1/128", "bf16", L2, 768, "a", qnorm=2.0 ** -7),
    Spec("i8-l2-100-b-q1/128", "i8", L2, 100, "b", qnorm=2.0 ** -7),
    Spec("bf16-cos-100-a", "bf16", COS, 100, "a"),
    Spec("i8-cos-768-b", "i8", COS, 768, "b"),
    Spec("i8hot-cos-1024-a", "i8", COS, 1024, "a", level8=11),    # rho_x8 > 0.03: only PATH_UMMA8 scans it
]
SPEC = {s.name: s for s in SPECS}


# ---------------------------------------------------------------------------------------------------------------------
# construction (numpy, fp64 where it matters)
# ---------------------------------------------------------------------------------------------------------------------
def _nt(d):
    return NT_OF_D.get(d, 32)


def _bf16_grid(v):
    """(largest bf16 value <= v, bf16 step there) for v > 0."""
    step = 2.0 ** (math.floor(math.log2(v)) - 7)
    return math.floor(v / step) * step, step


def _queries(d, B, rng):
    """Unit queries (exactly: fl32(q / ||q||) == q): channel 0 zero, channel 1 sets the norm, the rest +-m_j with
    m_j half a bf16 step (+-2 %) above a bf16 value.  tau_j = +1: the query's bf16 rounds away from zero there."""
    NT = _nt(d)
    v0, step = _bf16_grid(0.98 / math.sqrt(d - 2))
    sig = rng.choice([-1.0, 1.0], size=(B, d))
    tau = rng.choice([-1.0, 1.0], size=(B, d))
    n_s = d - NT - 2           # over the attacked channels exactly half each way, so winners and decoys share a norm
    tau[:, NT + 2:] = np.where(rng.permuted(np.arange(n_s)[None, :].repeat(B, axis=0), axis=1) % 2 == 0, 1.0, -1.0)
    Q = (sig * (v0 + 0.5 * step * (1.0 + MARGIN * tau))).astype(F32).astype(np.float64)
    Q[:, 0] = 0.0
    Q[:, 1] = np.sqrt(1.0 - (Q[:, 2:] ** 2).sum(axis=1))
    return Q.astype(F32), sig, tau


def _base_rows(spec, sig, tau, down, R):
    """Rows for one query without their tuning channels: down = True rounds the key down (winners)."""
    n, d = down.size, spec.d
    NT = _nt(d)
    S = slice(NT + 2, d)
    n_s = d - NT - 2
    X = np.zeros((n, d), dtype=np.float64)
    if spec.shadow == "i8":
        L = spec.level8
        s = R / math.sqrt(127.0 ** 2 + n_s * (L + 0.5) ** 2) * 0.97
        A = F32(127.0 * s)
        s_x = float(A / F32(127))
        frac = np.where(down, L + FRAC8, L + 1 - FRAC8)[:, None]       # |x| / s_x: rounds to L (down) or L + 1 (up)
        X[:, 0] = float(A)
        X[:, S] = sig[None, S] * (s_x * frac).astype(F32)
    else:
        a0, astep = _bf16_grid(R * math.sqrt(0.85 * 2.0 / (n_s * 1.0625)))
        pos = np.where(down, 0.5 * (1.0 - MARGIN), 0.5 * (1.0 + MARGIN))[:, None]   # below / above the midpoint
        mag = a0 + pos * astep
        # the larger level where the query's rounding pushes the same way as the row's: tau = -1 for winners
        big = np.where(down[:, None], tau[None, S] < 0, tau[None, S] > 0)
        X[:, S] = sig[None, S] * np.where(big, mag, mag / 4.0)
    return X.astype(F32).astype(np.float64)


def _tune(spec, X, q, sig, targets):
    """Set the tuning channels of every row to sig_j * t so that its exact key hits its target."""
    NT = _nt(spec.d)
    T = slice(2, NT + 2)
    q64 = q.astype(np.float64)
    qn = math.sqrt(float(q64 @ q64))
    D0 = X @ q64
    N0 = (X * X).sum(axis=1)
    QT = float(np.abs(q64[T]).sum())
    if spec.metric == COS:
        key = lambda t: (D0 + t * QT) / (np.sqrt(N0 + NT * t * t) * qn)
        t_peak = QT * N0 / (D0 * NT)                # the key rises on [0, t_peak]
        lo, hi = np.zeros_like(t_peak), t_peak
    else:
        key = lambda t: D0 + t * QT - 0.5 * (N0 + NT * t * t)
        t_ref = T_REF_L2 * float(np.median(N0 / (np.abs(X) @ np.abs(np.sign(q64)))))
        t_v = QT / NT                               # vertex of the parabola
        if t_v >= 3 * t_ref:
            lo, hi = np.zeros(len(X)), np.full(len(X), 3 * t_ref)
        else:
            lo, hi = np.full(len(X), t_v), np.full(len(X), t_v + 3 * t_ref)
    f_lo, f_hi = key(lo), key(hi)
    inc = f_hi > f_lo
    assert np.all(np.minimum(f_lo, f_hi) < targets) and np.all(targets < np.maximum(f_lo, f_hi)), \
        (spec, (np.minimum(f_lo, f_hi) - targets).max(), (targets - np.maximum(f_lo, f_hi)).max())
    for _ in range(80):
        mid = 0.5 * (lo + hi)
        up = (key(mid) < targets) == inc
        lo, hi = np.where(up, mid, lo), np.where(up, hi, mid)
    X[:, T] = sig[None, T] * (0.5 * (lo + hi))[:, None]
    return X.astype(F32)


def _kappa0(spec, x, q):
    """The key the targets are centred on: a base row's key with its tuning channels at a fixed point of their range."""
    NT = _nt(spec.d)
    T = slice(2, NT + 2)
    q64 = q.astype(np.float64)
    D0, N0, QT = float(x @ q64), float(x @ x), float(np.abs(q64[T]).sum())
    if spec.metric == COS:
        t = T_REF_COS * QT * N0 / (D0 * NT)
        return (D0 + t * QT) / math.sqrt((N0 + NT * t * t) * float(q64 @ q64))
    t = T_REF_L2 * N0 / float(np.abs(x) @ np.abs(np.sign(q64)))
    return D0 + t * QT - 0.5 * (N0 + NT * t * t)


def _eps_estimate(spec, qn, R):
    """The allowance the corpus will get, before it exists (targets only need its scale)."""
    if spec.shadow == "i8":
        n_s = spec.d - _nt(spec.d) - 2
        L = spec.level8
        e = FRAC8 * math.sqrt(n_s) / math.sqrt(127.0 ** 2 + n_s * (L + 0.5) ** 2) + 2e-4
    else:
        e = 2 * 2.0 ** -8
    e += spec.dim_pad * 2.0 ** -23
    return e * R * qn + 6e-8 * R * R if spec.metric == L2 else e


def _layout(spec, B, rng):
    """Roles of the adversarial rows per query and where they go.  Returns (query of each adversarial row, its role:
    True = winner) in corpus order and the position of every adversarial row among all rows."""
    owner, role = [], []
    if spec.regime == "a":
        for b in range(B):
            owner += [b] * (2 * N_ADV_A)
            role += [True] * N_ADV_A + [False] * N_ADV_A
        owner, role = np.array(owner), np.array(role)
        n = owner.size + spec.n_bg
        pos = np.sort(rng.choice(n, size=owner.size, replace=False))
        perm = rng.permutation(owner.size)
        return owner[perm], role[perm], pos, n
    # regime (b): blocks of adjacent rows, D D D W repeating, each block a whole number of tiles
    for b in range(B):
        length = LONG_BLOCK if b < 2 else 4 * TILE
        owner += [b] * length
        role += [(i % 4) == 3 for i in range(length)]
    owner, role = np.array(owner), np.array(role)
    return owner, role, np.arange(owner.size), owner.size + spec.n_bg


def _background(spec, n, R, rng):
    """Unit rows; for L2 scaled relative to R, the largest norm of the attacked rows."""
    X = synth.embeddings(n, spec.d, 7000 + spec.d).astype(np.float64)
    if spec.metric == L2:
        if spec.qnorm >= 16:
            X *= rng.uniform(0.5 / 8, 1.0, size=(n, 1)) * R     # norms spread over ~0.5 .. R
        else:
            # small queries: the key is ~ -||x||^2 / 2, so the background lies just outside the attacked rows' norms
            X *= rng.uniform(1.002, 1.02, size=(n, 1)) * R
    return X.astype(F32)


B_MAX = 130


@functools.lru_cache(maxsize=1)
def build(name, B=B_MAX):
    """(X [n, d] fp32, Q [B, d] fp32, owner [n] (-1 = background), winner [n] bool) of spec `name`."""
    spec = SPEC[name]
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    R = 8.0 if spec.metric == L2 else 1.0
    Q, sig, tau = _queries(spec.d, B, rng)
    if spec.metric == L2:
        Q = (Q * F32(spec.qnorm)).astype(F32)
    owner_adv, win_adv, pos, n = _layout(spec, B, rng)
    X = np.empty((n, spec.d), dtype=F32)
    owner = np.full(n, -1, dtype=np.int64)
    winner = np.zeros(n, dtype=bool)
    eps = _eps_estimate(spec, spec.qnorm if spec.metric == L2 else 1.0, R)
    for b in range(B):
        sel = owner_adv == b
        down = win_adv[sel]
        Xb = _base_rows(spec, sig[b], tau[b], down, R)
        k0 = _kappa0(spec, Xb[0], Q[b])
        u = rng.uniform(size=down.size)
        targets = np.where(down, k0 + eps * (W_FRAC[0] + (W_FRAC[1] - W_FRAC[0]) * u),
                           k0 - eps * (D_FRAC[0] + (D_FRAC[1] - D_FRAC[0]) * u))
        X[pos[sel]] = _tune(spec, Xb, Q[b], sig[b], targets)
        owner[pos[sel]] = b
        winner[pos[sel]] = down
    bg = np.setdiff1d(np.arange(n), pos, assume_unique=True)
    X64 = X[pos].astype(np.float64)
    X[bg] = _background(spec, bg.size, math.sqrt(float((X64 * X64).sum(axis=1).max())), rng)
    return X, Q, owner, winner


# ---------------------------------------------------------------------------------------------------------------------
# models of the scans and of finish.cu's allowance
# ---------------------------------------------------------------------------------------------------------------------
def _f32_up(v):
    """float(v) rounded up to float32, as __double2float_ru."""
    f = F32(v)
    return f if float(f) >= v else np.nextafter(f, F32(np.inf))


def _eps(rho_x, rho_q, dim_pad, metric, xm, qn):
    """finish_kernel's allowance, in float32 as it computes it."""
    e = F32(rho_x) * (F32(1) + F32(rho_q)) + F32(rho_q) + F32(dim_pad * 1.1920929e-7)
    if metric == L2:
        e = e * F32(xm) * F32(qn) * F32(1.0001) + F32(6.0e-8) * F32(xm) * F32(xm)
    return float(e * F32(1.0001))


def _q_hat(q, metric):
    q64 = q.astype(np.float64)
    n = math.sqrt(float(q64 @ q64))
    return (q64 * (1.0 / n)).astype(F32) if metric == COS else q.astype(F32), n


def _int8_key(acc1, acc2, s1, s2, sa8, sb):
    """int8_key (common.cuh): fma(fma(s1, acc1, s2 * acc2), sa8, sb) in float32."""
    inner = (float(s1) * acc1.astype(np.float64) + (F32(s2) * acc2.astype(F32)).astype(np.float64)).astype(F32)
    return (inner.astype(np.float64) * sa8.astype(np.float64) + sb.astype(np.float64)).astype(F32)


class Store:
    """What store_convert_kernel derives from the rows: norms, scan scales and offsets, residual bounds."""

    def __init__(self, X, metric):
        self.X, self.metric = X, metric
        X64 = X.astype(np.float64)
        self.n2 = (X64 * X64).sum(axis=1)
        self.xn = np.sqrt(self.n2)
        self.xm = float(_f32_up(self.xn.max()))
        self.sb = np.zeros(len(X), F32) if metric == COS else (-0.5 * self.n2).astype(F32)
        self.sa = (1.0 / self.xn).astype(F32) if metric == COS else np.ones(len(X), F32)
        self.x16 = _bf16(X)
        res = np.sqrt(((X64 - self.x16) ** 2).sum(axis=1)) / self.xn
        self.rho_x = float(_f32_up(res.max()))
        rho8, _, s_x = _rho_x8(X)
        self.rho_x8 = float(_f32_up(rho8))
        self.x8, _ = _quantise(X)
        self.sa8 = (s_x.astype(np.float64) / self.xn).astype(F32) if metric == COS else s_x.astype(F32)

    def exact(self, q):
        """Exact keys in the scan's units: cosine, or x.q - ||x||^2 / 2 for L2."""
        q64 = q.astype(np.float64)
        dot = self.X.astype(np.float64) @ q64
        if self.metric == COS:
            return dot / (self.xn * math.sqrt(float(q64 @ q64)))
        return dot - 0.5 * self.n2

    def model(self, q, shadow, dim_pad):
        """(approximate keys of the scan over `shadow`, the allowance finish.cu certifies that scan with)."""
        q_hat, qn = _q_hat(q, self.metric)
        if shadow == "i8":
            q1, q2, s1, s2, rho_q = _query_parts(q_hat)
            acc = self.x8.astype(np.float64) @ np.stack([q1, q2], axis=1).astype(np.float64)   # exact: |acc| < 2^24
            key = _int8_key(acc[:, 0], acc[:, 1], s1, s2, self.sa8, self.sb)
            return key.astype(np.float64), _eps(self.rho_x8, rho_q, dim_pad, self.metric, self.xm, qn)
        if shadow == "bf16":                       # the tcgen05 passes: bf16 rows and bf16 query
            qb = _bf16(q_hat).astype(np.float64)
            h = q_hat.astype(np.float64)
            rho_q = float(_f32_up(math.sqrt(float(((h - qb) ** 2).sum()) / float(h @ h))))
        else:                                      # "stream": bf16 rows, fp32 query, no query residual
            qb, rho_q = q_hat.astype(np.float64), 0.0
        dot = (self.x16.astype(np.float64) @ qb).astype(F32)
        key = (dot.astype(np.float64) * self.sa + self.sb).astype(F32)
        return key.astype(np.float64), _eps(self.rho_x, rho_q, dim_pad, self.metric, self.xm, qn)


def _top(key, k):
    """top-k rows of the order (key desc, row asc)."""
    return np.lexsort((np.arange(key.size), -key))[:k]


def _shadows(spec):
    """The scans whose shadow the corpus attacks: int8 -> the int8 pass; bf16 -> the tcgen05 passes and the
    streaming pass."""
    return ("i8",) if spec.shadow == "i8" else ("bf16", "stream")


CPU_QUERIES = (0, 1, 2, B_MAX - 1)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: every corpus is legal, near the bound and adversarial under the models
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", [s.name for s in SPECS])
def test_corpus_is_legal_near_the_bound_and_adversarial(name):
    spec = SPEC[name]
    X, Q, owner, winner = build(name)
    st = Store(X, spec.metric)
    if spec.shadow == "i8":
        assert (st.rho_x8 > RHO8_MAX) == (spec.level8 < 20), st.rho_x8
    for shadow in _shadows(spec):
        for b in CPU_QUERIES:
            approx, eps = st.model(Q[b], shadow, spec.dim_pad)
            exact = st.exact(Q[b])
            err = approx - exact
            # legal: the allowance bounds the model's error of every row
            assert np.abs(err).max() <= eps, (shadow, b, np.abs(err).max(), eps)
            # near the bound: winners off by >= eps / 2 downwards, decoys upwards
            mine = owner == b
            assert err[mine & winner].max() <= -eps / 2, (shadow, b, err[mine & winner].max() / eps)
            assert err[mine & ~winner].min() >= eps / 2, (shadow, b, err[mine & ~winner].min() / eps)
            # adversarial: the shadow's top-k shares at most half its ids with the exact top-k
            for k in KS:
                want = _top(exact, k)
                assert np.all(winner[want] & (owner[want] == b))
                assert np.intersect1d(_top(approx, k), want).size <= k // 2, (shadow, b, k)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def _rb():
    import rassengine_b200 as rb
    return rb


@pytest.fixture(scope="module", params=[s.name for s in SPECS])
def corpus(request):
    """(spec, X, Q, owner, winner, oracle rows [B_MAX, 100], oracle scores) of one spec."""
    spec = SPEC[request.param]
    X, Q, owner, winner = build(spec.name)
    want_rows, _, want_scores = knn.knn_exact(X, Q, max(KS), metric=spec.metric)
    return spec, X, Q, owner, winner, want_rows, want_scores


def _attacked(spec, path, rb):
    """Whether a first pass over `path` scans the shadow the corpus attacks."""
    if spec.shadow == "i8":
        return path == rb.PATH_UMMA8
    return path in (rb.PATH_STREAM, rb.PATH_UMMA, rb.PATH_GEMM)


@pytest.mark.gpu
def test_kernel_keys_rank_decoys_above_winners(corpus):
    """The kernels' own scan keys (raw accumulators from the debug entry points, sa / sa8 / sb recomputed here) are
    the model's, and rank the decoys above the winners: without this the id tests below would be vacuous."""
    rb = _rb()
    spec, X, Q, owner, winner, want_rows, _ = corpus
    st = Store(X, spec.metric)
    with rb.Engine(dim=spec.d, metric=spec.metric) as e:
        e.append(X)
        if spec.shadow == "i8":
            acc, x8, q8 = e.debug_umma8_scores(Q[:64])
            assert np.array_equal(x8[:, :spec.d].astype(np.int64), st.x8)
            kernel = []
            for b in range(64):
                q1, q2, s1, s2, _ = _query_parts(_q_hat(Q[b], spec.metric)[0])
                assert np.array_equal(q8[b, :spec.d], q1) and np.array_equal(q8[64 + b, :spec.d], q2), b
                kernel.append(_int8_key(acc[:, b], acc[:, 64 + b], s1, s2, st.sa8, st.sb))
            sets = [("umma8", np.stack(kernel, axis=1), "i8", 64)]
        else:
            dots = e.debug_umma_scores(Q[:64])
            gdots = e.debug_gemm_scores(Q)
            key = lambda dd: (dd.astype(np.float64) * st.sa[:, None] + st.sb[:, None]).astype(F32)
            sets = [("umma", key(dots[:, :64]), "bf16", 64), ("gemm", key(gdots[:, :B_MAX]), "bf16", B_MAX)]
    for what, keys, shadow, nq in sets:
        for b in range(nq):
            model, eps = st.model(Q[b], shadow, spec.dim_pad)
            kb = keys[:, b].astype(np.float64)
            # int8: exact integer dots, the same fp32 expression; bf16: another summation order
            tol = 1e-6 * np.abs(model).max() if shadow == "i8" else 2.0 ** -23 * spec.dim_pad * np.abs(model).max()
            assert np.abs(kb - model).max() <= tol, (what, b)
            mine = owner == b
            assert kb[mine & ~winner].min() > kb[want_rows[b, :max(KS)]].max(), (what, b)
            for k in KS:
                assert np.intersect1d(_top(kb, k), want_rows[b, :k]).size <= k // 2, (what, b, k)


RUNS = [("stream", 1), ("stream", 2), ("umma", 64), ("umma8", 64), ("gemm", 100), ("gemm", B_MAX), ("exact", 6)]
AUTO_B = (1, 2, 64, B_MAX)


def _check_run(spec, rb, B, k, path, rows, scores, st, want_rows, want_scores, tag):
    assert np.array_equal(rows, want_rows[:B, :k]), (tag, B, k, st)
    np.testing.assert_allclose(scores, want_scores[:B, :k], rtol=1e-5, atol=0)
    # every query is certified by the first pass, by the bf16 retry or computed by the fp64 scan
    assert st["n_certified"] + st["n_fallback"] == B and 0 <= st["n_retried"] <= B, (tag, st)
    first = B - st["n_retried"] if st["n_retried"] else st["n_certified"]
    if spec.regime == "b" and _attacked(spec, st["path"], rb):
        assert first < B, (tag, B, k, st)          # the winners left the pool: the first pass must not certify
    print(f"[{spec.name}] {tag} B={B} k={k}: path {st['path']}, first pass certified {first} of {B}, "
          f"retried {st['n_retried']}, fp64 {st['n_fallback']}, max candidates {st['max_candidates']}")


@pytest.mark.gpu
def test_ids_equal_the_oracle_on_every_path(corpus):
    """Every path at k in {1, 10, 32, 100}: the fp64 oracle's ids and scores, stats that account for every query, and in
    regime (b) a first pass over the attacked shadow that does not certify everything.  AUTO gets a fresh engine per
    case (int8_k_max is sticky per handle)."""
    rb = _rb()
    spec, X, Q, owner, winner, want_rows, want_scores = corpus
    paths = {"stream": rb.PATH_STREAM, "umma": rb.PATH_UMMA, "umma8": rb.PATH_UMMA8, "gemm": rb.PATH_GEMM,
             "exact": rb.PATH_EXACT}
    with rb.Engine(dim=spec.d, metric=spec.metric) as e:
        e.append(X)
        for tag, B in RUNS:
            e.set_path(paths[tag])
            for k in KS:
                rows, scores = e.search_knn(Q[:B], k)
                st = e.last_stats
                assert st["path"] == paths[tag] or (st["path"] == rb.PATH_UMMA and tag == "umma8"), (tag, st)
                _check_run(spec, rb, B, k, paths[tag], rows, scores, st, want_rows, want_scores, tag)
    int8_auto = _rho_x8(X)[0] <= RHO8_MAX
    for B in AUTO_B:
        for k in KS:
            with rb.Engine(dim=spec.d, metric=spec.metric) as e:
                e.append(X)
                rows, scores = e.search_knn(Q[:B], k)
                st = e.last_stats
            if 2 <= B <= 64:
                assert st["path"] == (rb.PATH_UMMA8 if int8_auto else rb.PATH_UMMA), st
            _check_run(spec, rb, B, k, rb.PATH_AUTO, rows, scores, st, want_rows, want_scores, "auto")


REGIME_B = "i8-cos-1024-b"


@pytest.mark.gpu
def test_dropped_winners_through_overlapped_async_slots():
    """Regime (b) through both async slots with RASS_OPT_ASYNC_OVERLAP on: a batch whose winners left the pool is
    reported as not final (its flag counts the uncertified queries), and the blocking repeat returns the oracle's ids;
    a final batch already has them."""
    import torch
    rb = _rb()
    spec = SPEC[REGIME_B]
    X, Q, owner, winner = build(REGIME_B)
    B, k, n_batches = 64, 10, 4
    batches = [Q[(i % 2) * 64:(i % 2) * 64 + B] for i in range(n_batches)]
    want = [knn.knn_exact(X, q, k)[0] for q in batches[:2]]
    not_final = 0
    with rb.Engine(dim=spec.d) as e:
        e.append(X)
        e.set_path(rb.PATH_UMMA8)
        e.set_async_overlap(True)
        Qd = [torch.from_numpy(np.ascontiguousarray(q)).cuda() for q in batches]
        rows = [torch.full((B, k), -7, dtype=torch.int64, device="cuda") for _ in range(2)]
        scores = [torch.empty((B, k), dtype=torch.float32, device="cuda") for _ in range(2)]
        flags = [torch.empty(1, dtype=torch.int64, device="cuda") for _ in range(2)]
        torch.cuda.synchronize()
        for i in range(0, n_batches, 2):
            for s in range(2):
                e.search_knn_dev_async(Qd[i + s].data_ptr(), B, k, rows[s].data_ptr(), scores[s].data_ptr(), 0, s,
                                       flags[s].data_ptr())
            for s in range(2):
                final, st = e.search_knn_dev_wait(s)
                got = rows[s].cpu().numpy().copy()
                if final:
                    assert int(flags[s].item()) == 0 and np.array_equal(got, want[s]), (i, s, st)
                else:
                    not_final += 1
                    assert int(flags[s].item()) == st["n_fallback"] > 0, (i, s, st)
        e.set_async_overlap(False)
        for s in range(2):
            r, _ = e.search_knn(batches[s], k)
            assert np.array_equal(r, want[s])
    assert not_final > 0


@pytest.mark.gpu
def test_tombstoned_winners_vanish_and_the_next_rows_come_up():
    """Regime (b) with every query's ten best winners tombstoned: they never come back, and the rows behind them (the
    next winners, still below the decoys in the shadow) are the oracle's over the live rows."""
    rb = _rb()
    spec = SPEC[REGIME_B]
    X, Q, owner, winner = build(REGIME_B)
    B, k = 64, 10
    top = knn.knn_exact(X, Q[:B], k)[0]
    alive = np.ones(len(X), dtype=bool)
    alive[top.ravel()] = False
    want_rows, _, want_scores = knn.knn_exact(X, Q[:B], k, alive=alive)
    assert np.all(winner[want_rows])
    with rb.Engine(dim=spec.d) as e:
        e.append(X)
        for r in top.ravel():
            e.tombstone(int(r))
        for path in (rb.PATH_UMMA8, rb.PATH_AUTO, rb.PATH_UMMA):
            e.set_path(path)
            rows, scores = e.search_knn(Q[:B], k)
            assert not np.isin(rows, top).any()
            _check_run(spec, rb, B, k, path, rows, scores, e.last_stats, want_rows, want_scores, f"tombstones/{path}")
