"""GPU checks of the int8 64-query pass (scan_umma_kernel<SEG, true>): its raw accumulators against integer dot
products, then ids identical to the oracle through RASS_PATH_UMMA8 and through AUTO, the ladder to the bf16 pass when
an int8 certificate fails, and the stores that have no int8 shadow.  Runs on the B200 box only (-m gpu)."""
import numpy as np
import pytest

from oracle import knn, synth

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-5


def _rb():
    import rassengine_b200 as rb
    return rb


def _check(rows, scores, want_rows, want_scores):
    assert np.array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=0)


def _int8_codes(X):
    """store_convert_kernel's quantiser in float32: s = max|x| / 127, code = rint(x / s) in [-127, 127]."""
    amax = np.abs(X).max(axis=1, keepdims=True).astype(np.float32)
    s = amax / np.float32(127)
    with np.errstate(divide="ignore", invalid="ignore"):
        c = np.where(s > 0, np.rint(X / np.where(s > 0, s, 1)), 0)
    return np.clip(c, -127, 127).astype(np.int8)


@pytest.mark.parametrize("d", [768, 1024])
def test_umma8_raw_accumulators_equal_integer_dots(d):
    """The kind::i8 accumulators equal numpy's int64 dot products of the int8 operands the pass read (instruction and
    smem descriptors, the UINT8 tensor maps, the 128-row query block); the rows are the quantiser's codes, and the
    query block's pad rows are zero.  1000 rows leave the last tile partly out of range."""
    rb = _rb()
    n, B = 1000, 50
    X = synth.embeddings(n, d, 7)
    X[3] = 0.0                                     # a zero row: scale 0, codes 0
    Q = synth.embeddings(B, d, 8)
    with rb.Engine(dim=d) as e:
        e.append(X)
        acc, x8, q8 = e.debug_umma8_scores(Q)
    dim_pad = x8.shape[1]
    assert np.array_equal(x8[:, :d], _int8_codes(X)) and not x8[:, d:].any()
    assert not q8[B:64].any() and not q8[64 + B:].any()
    assert q8[:B].any() and q8[64:64 + B].any()
    want = x8.astype(np.int64) @ q8.astype(np.int64).T
    assert np.array_equal(acc.astype(np.int64), want)
    assert dim_pad == (d + 255) // 256 * 256


@pytest.mark.parametrize("metric", ["cos", "l2"])
@pytest.mark.parametrize("d", [768, 1024])
def test_umma8_ids_equal_oracle(metric, d):
    """RASS_PATH_UMMA8 for B in {2, 17, 64} and k in {1, 10, 32, 100}: ids identical to the oracle (k = 100 goes through
    the bf16 pass for the queries whose int8 certificate fails); AUTO takes the int8 pass for 2..64 queries and counts
    one byte per element, and returns the same ids whichever pass it takes at k = 100."""
    rb = _rb()
    m = knn.COSINE if metric == "cos" else knn.L2
    n = 20000
    X = synth.embeddings(n, d, 11)
    Q = synth.embeddings(64, d, 13)
    with rb.Engine(dim=d, metric=m) as e:
        e.append(X)
        for k in (1, 10, 32, 100):
            want_rows, _, want_scores = knn.knn_exact(X, Q, k, metric=m)
            for B in (2, 17, 64):
                e.set_path(rb.PATH_UMMA8)
                rows, scores = e.search_knn(Q[:B], k)
                st = e.last_stats
                _check(rows, scores, want_rows[:B], want_scores[:B])
                assert st["path"] == rb.PATH_UMMA8, (k, B, st)
                e.set_path(rb.PATH_AUTO)
                rows, scores = e.search_knn(Q[:B], k)
                st = e.last_stats
                _check(rows, scores, want_rows[:B], want_scores[:B])
                if k <= 32:
                    assert st["path"] == rb.PATH_UMMA8, st
                    assert st["n_certified"] == B and st["n_retried"] == 0, (k, B, st)
                    assert st["bytes_streamed"] == n * ((d + 255) // 256 * 256), st


def test_umma8_tombstones_prefilter_and_growth():
    """Appends that grow the store across several chunks of its growable arrays (the int8 planes grow in place with the
    others), tombstones and the exact pre-filter: ids identical to the oracle over the alive rows."""
    rb = _rb()
    d = 1024
    parts = [synth.embeddings(n, d, 21 + i) for i, n in enumerate((30000, 45000, 50000))]
    Q = synth.embeddings(24, d, 25)
    rng = np.random.default_rng(26)
    with rb.Engine(dim=d) as e:
        e.set_path(rb.PATH_UMMA8)
        X = np.zeros((0, d), dtype=np.float32)
        for p in parts:
            e.append(p)
            X = np.concatenate([X, p])
            want_rows, _, want_scores = knn.knn_exact(X, Q, 10)
            rows, scores = e.search_knn(Q, 10)
            _check(rows, scores, want_rows, want_scores)
        dead = want_rows[:, 0]                      # every query's best row goes
        for r in dead:
            e.tombstone(int(r))
        alive = np.ones(X.shape[0], dtype=bool)
        alive[dead] = False
        want_rows, _, want_scores = knn.knn_exact(X, Q, 10, alive=alive)
        rows, scores = e.search_knn(Q, 10)
        _check(rows, scores, want_rows, want_scores)
        e.set_knn_prefilter(True)
        mask = rng.integers(0, 5, size=X.shape[0]) == 0
        e.set_row_filter(mask)
        want_rows, _, want_scores = knn.knn_exact(X, Q, 10, alive=alive & mask)
        rows, scores = e.search_knn(Q, 10)
        _check(rows, scores, want_rows, want_scores)
        assert e.last_stats["path"] == rb.PATH_UMMA8


def test_umma8_overlapped_async_slots_equal_the_oracle():
    """Both async slots in flight through the int8 pass (each slot's workspace holds its own int8 query block and
    tensor map), a blocking search in between."""
    import torch
    rb = _rb()
    B, k, n_batches = 64, 10, 8
    X = synth.embeddings(150000, 1024, 31)
    Qs = [synth.embeddings(B, 1024, 32 + i) for i in range(n_batches)]
    want = [knn.knn_exact(X, Q, k)[0] for Q in Qs]
    with rb.Engine(dim=1024) as e:
        e.append(X)
        e.set_path(rb.PATH_UMMA8)
        e.set_async_overlap(True)
        Qd = [torch.from_numpy(Q).cuda() for Q in Qs]
        rows = [torch.full((B, k), -7, dtype=torch.int64, device="cuda") for _ in range(2)]
        scores = [torch.empty((B, k), dtype=torch.float32, device="cuda") for _ in range(2)]
        flags = [torch.empty(1, dtype=torch.int64, device="cuda") for _ in range(2)]
        torch.cuda.synchronize()
        got = [None] * n_batches

        def collect(i):
            final, st = e.search_knn_dev_wait(i & 1)
            assert final and int(flags[i & 1].item()) == 0 and st["path"] == rb.PATH_UMMA8, (i, st)
            got[i] = rows[i & 1].cpu().numpy().copy()

        for i in range(n_batches):
            if i >= 2:
                collect(i - 2)
            e.search_knn_dev_async(Qd[i].data_ptr(), B, k, rows[i & 1].data_ptr(), scores[i & 1].data_ptr(), 0, i & 1,
                                   flags[i & 1].data_ptr())
            if i == 3:
                r, _ = e.search_knn(Qs[0], k)
                assert np.array_equal(r, want[0])
        collect(n_batches - 2)
        collect(n_batches - 1)
        e.set_async_overlap(False)
    for i in range(n_batches):
        assert np.array_equal(got[i], want[i]), i


@pytest.mark.parametrize("flags", ["bf16_only", "no_int8"])
def test_stores_without_the_int8_shadow_take_the_bf16_pass(flags):
    """A BF16_ONLY store and a RASS_NO_INT8_SHADOW store have no int8 planes: AUTO resolves 2..64 queries to the bf16
    pass and forcing the int8 one is refused.  RASS_NO_INT8_SHADOW alone still keeps the fp32 rows."""
    rb = _rb()
    X = synth.embeddings(20000, 1024, 41)
    Q = synth.embeddings(17, 1024, 42)
    f = rb.BF16_ONLY if flags == "bf16_only" else rb.NO_INT8_SHADOW
    with rb.Engine(dim=1024, flags=f) as e:
        e.append(X)
        rows, scores = e.search_knn(Q, 10)
        assert e.last_stats["path"] == rb.PATH_UMMA
        with pytest.raises(rb.RassError):
            e.set_path(rb.PATH_UMMA8)
        if flags == "no_int8":
            want_rows, _, want_scores = knn.knn_exact(X, Q, 10)
            _check(rows, scores, want_rows, want_scores)
            assert np.array_equal(e.read_rows(0, 100), X[:100])


def test_failed_int8_certificates_get_the_bf16_pass():
    """40000 rows whose cosines to the queries spread evenly over [0.4, 0.8]: within twice the int8 allowance of the
    k-th best key the candidate segments hold more rows than the rerank takes in total (RASS_CAND_MAX), so no int8
    certificate holds; the bf16 pass, with a third of the allowance, certifies them all, and the ids are the oracle's.
    AUTO then takes the bf16 pass directly at that k and above, and keeps the int8 pass below it."""
    rb = _rb()
    rng = np.random.default_rng(51)
    d, n_c, B = 1024, 40000, 4
    q = rng.standard_normal(d)
    q /= np.linalg.norm(q)
    U = rng.standard_normal((n_c, d))
    U -= (U @ q)[:, None] * q[None, :]
    U /= np.linalg.norm(U, axis=1, keepdims=True)
    c = rng.uniform(0.4, 0.8, size=n_c)
    cluster = (c[:, None] * q[None, :] + np.sqrt(1 - c * c)[:, None] * U).astype(np.float32)
    X = np.concatenate([synth.embeddings(20000, d, 52), cluster])
    Q = (q[None, :] + 1e-3 * rng.standard_normal((B, d))).astype(np.float32)
    want_rows, _, want_scores = knn.knn_exact(X, Q, 10)
    want1 = knn.knn_exact(X, Q, 1)[0]
    with rb.Engine(dim=d) as e:
        e.append(X)
        rows, scores = e.search_knn(Q, 10)
        st = e.last_stats
        rows2, scores2 = e.search_knn(Q, 10)
        st2 = e.last_stats
        rows1, _ = e.search_knn(Q, 1)
        st1 = e.last_stats
    _check(rows, scores, want_rows, want_scores)
    assert st["path"] == rb.PATH_UMMA8 and st["n_retried"] == B and st["n_fallback"] == 0, st
    _check(rows2, scores2, want_rows, want_scores)
    assert st2["path"] == rb.PATH_UMMA and st2["n_retried"] == 0 and st2["n_fallback"] == 0, st2
    assert np.array_equal(rows1, want1) and st1["path"] == rb.PATH_UMMA8, st1


def test_one_query_searches_stream_the_bf16_shadow():
    """A one-query search (a hybrid call per request, as `/ask` issues them) still takes the streaming pass over the bf16
    shadow on a store that has the int8 one: 2 bytes per element, which is what scripts that subtract the kNN pass from
    a hybrid call's byte count rely on."""
    rb = _rb()
    n, d = 20000, 1024
    X = synth.embeddings(n, d, 61)
    Q = synth.embeddings(1, d, 62)
    with rb.Engine(dim=d) as e:
        e.append(X)
        rows, scores = e.search_knn(Q, 10)
        st = e.last_stats
    want_rows, _, want_scores = knn.knn_exact(X, Q, 10)
    _check(rows, scores, want_rows, want_scores)
    assert st["path"] == rb.PATH_STREAM and st["bytes_streamed"] == n * d * 2, st
