"""GPU parity: the CUDA kNN paths (through the C ABI) against the numpy oracle and the golden fixtures.

Bar: ids bit-identical to the oracle (fp64-accumulated key, (key desc, row asc)); scores within 1e-5 relative
(BASELINE.json north_star).  Runs on the B200 box only (-m gpu)."""
import json
import math
import os

import numpy as np
import pytest

from oracle import knn, synth

pytestmark = pytest.mark.gpu

SCORE_RTOL = 1e-5


def _engine(**kw):
    import rassengine_b200 as rb
    return rb.Engine(**kw)


def _paths():
    import rassengine_b200 as rb
    return {"stream": rb.PATH_STREAM, "umma": rb.PATH_UMMA, "exact": rb.PATH_EXACT, "auto": rb.PATH_AUTO,
            "gemm": rb.PATH_GEMM}


def _load_case(golden_dir, name):
    g = np.load(os.path.join(golden_dir, name + ".npz"))
    meta = json.loads(str(g["meta"]))
    X = synth.embeddings(meta["n"], meta["d"], synth.SEED_CORPUS)
    if meta["dup_pairs"]:
        synth.plant_duplicates(X, len(meta["dup_pairs"]))
    Q = (synth.clustered_queries(X, meta["nq"]) if meta["clustered"]
         else synth.embeddings(meta["nq"], meta["d"], synth.SEED_QUERIES))
    return X, Q, meta, g


def _check(rows, scores, want_rows, want_scores):
    assert np.array_equal(rows, want_rows)
    np.testing.assert_allclose(scores, want_scores, rtol=SCORE_RTOL, atol=0)


TINY_X = np.array([[1, 0, 0, 0], [0, 1, 0, 0], [1, 1, 0, 0], [1, 0, 0, 0],
                   [0, 0, 0, 0], [-1, 0, 0, 0], [3, 4, 0, 0], [0, 0, 1, 0]], dtype=np.float32)
TINY_Q = np.array([[2, 0, 0, 0]], dtype=np.float32)
TINY_ORDER = [0, 3, 2, 6, 1, 4, 7, 5]
TINY_SCORE = [1.0, 1.0, 1 / (2 - math.sqrt(0.5)), 1 / 1.4, 0.5, 0.5, 0.5, 1 / 3]


@pytest.mark.parametrize("path", ["stream", "umma", "gemm", "exact"])
def test_tiny_hand_set(path):
    """Duplicates, a zero row, unnormalised rows, k > rows (same literals as tests/test_oracle.py)."""
    with _engine(dim=4) as e:
        e.set_path(_paths()[path])
        r0, s0 = e.search_knn(TINY_Q, 3)          # empty index -> no hits
        assert (r0 == -1).all()
        assert e.append(TINY_X) == 0
        assert e.count() == 8
        rows, scores = e.search_knn(TINY_Q, 8)
        assert rows[0].tolist() == TINY_ORDER
        np.testing.assert_allclose(scores[0], np.array(TINY_SCORE, dtype=np.float32), rtol=1e-6)
        rows, _ = e.search_knn(TINY_Q, 3)
        assert rows[0].tolist() == TINY_ORDER[:3]
        rows, scores = e.search_knn(TINY_Q, 20)    # fewer rows than k: return what exists, pad with -1
        assert rows[0, :8].tolist() == TINY_ORDER and (rows[0, 8:] == -1).all()
        # tombstone + overwrite (bulk "index" = insert-or-overwrite by _id)
        e.tombstone(0)
        assert e.count() == 7
        rows, _ = e.search_knn(TINY_Q, 3)
        assert rows[0].tolist() == [3, 2, 6]
        e.overwrite(0, np.array([5, 0, 0, 0], dtype=np.float32))
        assert e.count() == 8
        rows, _ = e.search_knn(TINY_Q, 2)
        assert rows[0].tolist() == [0, 3]
        np.testing.assert_array_equal(e.read_rows(6, 1)[0], TINY_X[6])


@pytest.mark.parametrize("path", ["stream", "umma", "gemm", "exact"])
def test_tiny_l2(path):
    import rassengine_b200 as rb
    with _engine(dim=4, metric=rb.METRIC_L2) as e:
        e.set_path(_paths()[path])
        e.append(TINY_X)
        rows, scores, keys = e.search_knn(TINY_Q, 3, want_keys=True)
        assert rows[0].tolist() == [0, 3, 2]
        np.testing.assert_allclose(keys[0], [1, 1, 2])
        np.testing.assert_allclose(scores[0], [0.5, 0.5, 1 / 3], rtol=1e-6)


@pytest.mark.parametrize("path", ["stream", "umma", "gemm", "exact", "auto"])
@pytest.mark.parametrize("name", ["knn_small", "knn_clustered_dups", "knn_small_k100"])
def test_seeded_golden(golden_dir, name, path):
    X, Q, meta, g = _load_case(golden_dir, name)
    if path == "exact":
        Q = Q[:8]
    with _engine(dim=meta["d"]) as e:
        e.set_path(_paths()[path])
        # ragged appends exercise the staging path
        e.append(X[:7])
        e.append(X[7:12345])
        e.append(X[12345:])
        assert e.rows() == meta["n"]
        rows, scores, keys = e.search_knn(Q, meta["k"], want_keys=True)
        st = e.last_stats
    nq = Q.shape[0]
    _check(rows, scores, g["rows"][:nq].astype(np.int64), g["score"][:nq])
    np.testing.assert_allclose(keys, g["cos"][:nq], rtol=0, atol=1e-12)
    assert st["n_queries"] == nq
    assert st["n_certified"] + st["n_fallback"] == nq


def test_umma_raw_scores_match_bf16_math():
    """The tcgen05 accumulators equal the fp32 dot products of the bf16-rounded operands (descriptor check)."""
    import torch
    n, d = 1000, 1024
    X = synth.embeddings(n, d, 7)
    Q = synth.embeddings(64, d, 8)
    with _engine(dim=d) as e:
        e.append(X)
        got = e.debug_umma_scores(Q)
    xb = torch.from_numpy(X).to(torch.bfloat16).to(torch.float64)
    qn = Q / np.linalg.norm(Q.astype(np.float64), axis=1, keepdims=True)
    qb = torch.from_numpy(qn.astype(np.float32)).to(torch.bfloat16).to(torch.float64)
    want = (xb @ qb.T).numpy()
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)


def test_gemm_raw_scores_match_bf16_math():
    """Same check for the CTA-pair kernel (cta_group::2 descriptors, both CTAs' halves of the query block); 300 rows
    leave the second CTA of the last tile partly out of range."""
    import torch
    n, d = 300 + 256 * 3, 1024
    X = synth.embeddings(n, d, 9)
    Q = synth.embeddings(200, d, 10)
    with _engine(dim=d) as e:
        e.append(X)
        got = e.debug_gemm_scores(Q)
    xb = torch.from_numpy(X).to(torch.bfloat16).to(torch.float64)
    qn = Q / np.linalg.norm(Q.astype(np.float64), axis=1, keepdims=True)
    qb = torch.from_numpy(qn.astype(np.float32)).to(torch.bfloat16).to(torch.float64)
    want = (xb @ qb.T).numpy()
    np.testing.assert_allclose(got[:, :200], want, rtol=0, atol=2e-5)
    assert not got[:, 200:].any()


@pytest.mark.parametrize("path", ["stream", "umma", "gemm"])
def test_cfg1_100k_golden(golden_dir, path):
    """BASELINE.json configs[0]: 100k x 1024, 1k queries, exact cosine top-10 -- ids identical to the golden file."""
    X, Q, meta, g = _load_case(golden_dir, "knn_cfg1")
    nq = 64 if path == "stream" else 1000
    with _engine(dim=meta["d"], capacity_rows=meta["n"]) as e:
        e.set_path(_paths()[path])
        e.append(X)
        rows, scores = e.search_knn(Q[:nq], meta["k"])
        st = e.last_stats
    _check(rows, scores, g["rows"][:nq].astype(np.int64), g["score"][:nq])
    assert st["n_fallback"] == 0, st


@pytest.mark.parametrize("dim", [384, 768, 100])
def test_other_dims(dim):
    X = synth.embeddings(5000, dim, 3)
    Q = synth.embeddings(9, dim, 4)
    want_rows, _, want_scores = knn.knn_exact(X, Q, 10)
    for path in ("stream", "umma", "gemm"):
        with _engine(dim=dim) as e:
            e.set_path(_paths()[path])
            e.append(X)
            rows, scores = e.search_knn(Q, 10)
        _check(rows, scores, want_rows, want_scores)


def test_bf16_corpus_mode():
    """BASELINE config 5 stores a bf16 corpus: the bf16 values are the data, the oracle sees them widened."""
    import rassengine_b200 as rb
    import torch
    X = synth.embeddings(20000, 1024, 11)
    Q = synth.embeddings(16, 1024, 12)
    Xb = torch.from_numpy(X).to(torch.bfloat16).to(torch.float32).numpy()
    want_rows, _, want_scores = knn.knn_exact(Xb, Q, 10)
    for path in ("stream", "umma", "gemm"):
        with _engine(dim=1024, flags=rb.BF16_ONLY) as e:
            e.set_path(_paths()[path])
            e.append(X)
            np.testing.assert_array_equal(e.read_rows(5, 3), Xb[5:8])
            rows, scores = e.search_knn(Q, 10)
        _check(rows, scores, want_rows, want_scores)


def test_unnormalised_rows_and_l2_seeded():
    import rassengine_b200 as rb
    rng = np.random.default_rng(5)
    X = (rng.standard_normal((8000, 256)) * rng.uniform(0.1, 5.0, size=(8000, 1))).astype(np.float32)
    Q = rng.standard_normal((5, 256)).astype(np.float32)
    for metric, om in ((rb.METRIC_COSINE, knn.COSINE), (rb.METRIC_L2, knn.L2)):
        want_rows, _, want_scores = knn.knn_exact_full(X, Q, 10, metric=om)
        for path in ("stream", "umma", "gemm"):
            with _engine(dim=256, metric=metric) as e:
                e.set_path(_paths()[path])
                e.append(X)
                rows, scores = e.search_knn(Q, 10)
            _check(rows, scores, want_rows, want_scores)


@pytest.mark.parametrize("dim", [1024, 768])
@pytest.mark.parametrize("metric_name", ["cosine", "l2"])
def test_seeded_threshold_paths_l2_and_dim768(dim, metric_name):
    """The threshold seed (store.cu) only runs from 8192 rows up, and takes a generic path when dim_pad != 1024; the L2
    metric scales its bound by the row / query norms.  20k unnormalised rows, both tcgen05 scans, k = 10 and 100."""
    import rassengine_b200 as rb
    rng = np.random.default_rng(71 + dim)
    n = 20000
    X = (rng.standard_normal((n, dim)) * rng.uniform(0.5, 2.0, size=(n, 1))).astype(np.float32)
    Q = rng.standard_normal((70, dim)).astype(np.float32)
    metric, om = (rb.METRIC_COSINE, knn.COSINE) if metric_name == "cosine" else (rb.METRIC_L2, knn.L2)
    for k in (10, 100):
        want_rows, _, want_scores = knn.knn_exact(X, Q, k, metric=om)
        for path in ("umma", "gemm"):
            with _engine(dim=dim, metric=metric) as e:
                e.set_path(_paths()[path])
                e.append(X)
                rows, scores = e.search_knn(Q, k)
                st = e.last_stats
            _check(rows, scores, want_rows, want_scores)
            assert st["n_certified"] + st["n_fallback"] == Q.shape[0], st


def test_merge_topk_matches_single_shard():
    """Row-sharded corpus: per-shard top-k merged on the device equals the single-engine answer."""
    import torch
    X = synth.embeddings(30000, 1024, 21)
    Q = synth.embeddings(12, 1024, 22)
    k, G = 10, 3
    want_rows, want_key, want_scores = knn.knn_exact(X, Q, k)
    bounds = [0, 9000, 21000, 30000]
    keys, rows = [], []
    engines = []
    for g in range(G):
        e = _engine(dim=1024)
        e.set_row_base(bounds[g])
        e.append(X[bounds[g]:bounds[g + 1]])
        r, s, kk = e.search_knn(Q, k, want_keys=True)
        keys.append(kk)
        rows.append(r)
        engines.append(e)
    dk = torch.from_numpy(np.stack(keys)).cuda()
    dr = torch.from_numpy(np.stack(rows)).cuda()
    out_r = torch.empty((Q.shape[0], k), dtype=torch.int64, device="cuda")
    out_s = torch.empty((Q.shape[0], k), dtype=torch.float32, device="cuda")
    engines[0].merge_topk_dev(dk.data_ptr(), dr.data_ptr(), G, Q.shape[0], k, out_r.data_ptr(), out_s.data_ptr())
    engines[0].sync()
    _check(out_r.cpu().numpy(), out_s.cpu().numpy(), want_rows, want_scores)
    for e in engines:
        e.close()


@pytest.mark.parametrize("path", ["stream", "umma", "gemm", "exact"])
def test_prefiltered_knn_matches_oracle_alive_mask(path):
    """SURVEY.md 8f N1: bool.must[knn] + filter[term patientId] as an exact PRE-filter -- top-k of the rows that pass,
    ids identical to the oracle restricted to those rows; includes a filter that leaves fewer than k rows."""
    X = synth.embeddings(30000, 1024, 31)
    Q = synth.embeddings(5, 1024, 32)
    rng = np.random.default_rng(33)
    patient = rng.integers(0, 40, size=X.shape[0])
    with _engine(dim=1024) as e:
        e.set_path(_paths()[path])
        e.append(X)
        e.tombstone(17)
        e.set_knn_prefilter(True)
        for mask in (patient == 3, patient < 20, np.arange(X.shape[0]) < 4):
            alive = mask.copy()
            alive[17] = False
            want_rows, _, want_scores = knn.knn_exact(X, Q, 10, alive=alive)
            e.set_row_filter(mask)
            rows, scores = e.search_knn(Q, 10)
            kk = want_rows.shape[1]
            _check(rows[:, :kk], scores[:, :kk], want_rows, want_scores)
            assert (rows[:, kk:] == -1).all()
        e.set_row_filter(None)              # no filter: back to the whole corpus
        alive = np.ones(X.shape[0], dtype=bool)
        alive[17] = False
        want_rows, _, want_scores = knn.knn_exact(X, Q, 10, alive=alive)
        rows, scores = e.search_knn(Q, 10)
        _check(rows, scores, want_rows, want_scores)


@pytest.mark.parametrize("path", ["stream", "umma", "gemm"])
def test_top100_inside_one_cluster_of_adjacent_rows_is_certified(path):
    """Chunks of one document are adjacent rows and close to each other.  400 such rows hold the whole top-100 of a
    query, so the fast pass (segments that keep 32..64 entries) cannot certify k = 100; the failed queries get a second
    pass with 512-entry segments (>= 128 entries above every pivot) on the tensor cores, not the fp64 scan."""
    rng = np.random.default_rng(61)
    X = synth.embeddings(60000, 1024, 62)
    centre = X[123].copy()
    lo = 20000
    X[lo:lo + 400] = centre[None, :] + 0.02 * rng.standard_normal((400, 1024)).astype(np.float32)
    X[lo:lo + 400] /= np.linalg.norm(X[lo:lo + 400], axis=1, keepdims=True)
    Q = (centre[None, :] + 0.01 * rng.standard_normal((70, 1024))).astype(np.float32)
    Q[1::2] = synth.embeddings(35, 1024, 63)            # every other query is unrelated to the cluster
    if path == "stream":
        Q = Q[:2]
    want_rows, _, want_scores = knn.knn_exact(X, Q, 100)
    assert ((want_rows[0::2] >= lo) & (want_rows[0::2] < lo + 400)).mean() > 0.95
    with _engine(dim=1024) as e:
        e.set_path(_paths()[path])
        e.append(X)
        rows, scores = e.search_knn(Q, 100)
        st = e.last_stats
        rows10, scores10 = e.search_knn(Q, 10)          # k <= 32 never needs the second pass
        st10 = e.last_stats
    _check(rows, scores, want_rows, want_scores)
    _check(rows10, scores10, want_rows[:, :10], want_scores[:, :10])
    assert st["n_fallback"] == 0 and st["n_certified"] == Q.shape[0], st
    if path == "stream":       # row groups are dealt round-robin to 2368 warps: no list ever sees more than a few of them
        assert st["n_retried"] == 0, st
    else:
        assert 0 < st["n_retried"] <= (Q.shape[0] + 1) // 2, st
    assert st10["n_retried"] == 0 and st10["n_fallback"] == 0, st10


def test_async_search_publishes_the_certificate_outcome():
    """rass_search_knn_dev_async leaves the number of uncertified queries in *flag_out_dev -- the word a row-sharded
    caller all-gathers with its candidates (sharded.py) -- written by the last CTA of the last finish launch: 0 on
    ordinary queries, the number of failed queries when a top-100 sits inside one cluster of adjacent rows (the async
    form does not retry; the caller repeats with the blocking call).  The word is overwritten, not accumulated."""
    import torch
    rng = np.random.default_rng(61)
    X = synth.embeddings(60000, 1024, 62)
    centre = X[123].copy()
    lo = 20000
    X[lo:lo + 400] = centre[None, :] + 0.02 * rng.standard_normal((400, 1024)).astype(np.float32)
    X[lo:lo + 400] /= np.linalg.norm(X[lo:lo + 400], axis=1, keepdims=True)
    Q = (centre[None, :] + 0.01 * rng.standard_normal((70, 1024))).astype(np.float32)
    Q[1::2] = synth.embeddings(35, 1024, 63)
    want_rows, _, _ = knn.knn_exact(X, Q, 10)
    B = Q.shape[0]
    with _engine(dim=1024) as e:
        e.append(X)
        Qd = torch.from_numpy(Q).cuda()
        rows = torch.empty((B, 100), dtype=torch.int64, device="cuda")
        scores = torch.empty((B, 100), dtype=torch.float32, device="cuda")
        flag = torch.empty(1, dtype=torch.int64, device="cuda")
        for path in ("umma", "gemm"):           # 70 queries: two finish launches on the 64-per-pass path, one on the other
            e.set_path(_paths()[path])
            flag.fill_(-5)
            torch.cuda.synchronize()
            e.search_knn_dev_async(Qd.data_ptr(), B, 10, rows.data_ptr(), scores.data_ptr(), 0, 0, flag.data_ptr())
            final, st = e.search_knn_dev_wait(0)
            assert final and int(flag.item()) == 0 and st["n_certified"] == B, (path, st, int(flag.item()))
            assert np.array_equal(rows.cpu().numpy().reshape(-1)[:B * 10].reshape(B, 10), want_rows), path
            flag.fill_(-5)
            torch.cuda.synchronize()
            e.search_knn_dev_async(Qd.data_ptr(), B, 100, rows.data_ptr(), scores.data_ptr(), 0, 1, flag.data_ptr())
            final, st = e.search_knn_dev_wait(1)
            assert not final and 0 < st["n_fallback"] <= 35 and int(flag.item()) == st["n_fallback"], (path, st)
            assert st["n_certified"] == B - st["n_fallback"], (path, st)


@pytest.mark.parametrize("path,B,k", [("umma", 64, 10), ("umma", 70, 10), ("gemm", 300, 10), ("stream", 1, 10),
                                      ("umma", 33, 100)])
def test_overlapped_async_slots_equal_the_oracle(path, B, k):
    """RASS_OPT_ASYNC_OVERLAP: both slots in flight on their own streams and workspaces, a different batch in each, many
    rounds back to back, a blocking search in between -- every batch's ids are the oracle's.  A workspace shared by
    mistake, a missing stream dependency or a tile-counter left dirty by the scan's scheduler shows up here as a wrong
    or torn list."""
    import torch
    n_batches = 12
    X = synth.embeddings(150000, 1024, 71)
    Qs = [synth.embeddings(B, 1024, 72 + i) for i in range(n_batches)]
    want = [knn.knn_exact(X, Q, k)[0] for Q in Qs]
    with _engine(dim=1024) as e:
        e.append(X)
        e.set_path(_paths()[path])
        e.set_async_overlap(True)
        side = torch.cuda.Stream()
        Qd = [torch.from_numpy(Q).cuda() for Q in Qs]
        rows = [torch.full((B, k), -7, dtype=torch.int64, device="cuda") for _ in range(2)]
        scores = [torch.empty((B, k), dtype=torch.float32, device="cuda") for _ in range(2)]
        flags = [torch.empty(1, dtype=torch.int64, device="cuda") for _ in range(2)]
        joined = [torch.empty((B, k), dtype=torch.int64, device="cuda") for _ in range(2)]
        torch.cuda.synchronize()
        got = [None] * n_batches

        def collect(i):
            slot = i & 1
            final, st = e.search_knn_dev_wait(slot)
            assert final and int(flags[slot].item()) == 0, (i, st)
            side.synchronize()
            # the copy made on the side stream behind rass_async_join sees the finished list as well
            assert torch.equal(joined[slot], rows[slot]), i
            got[i] = rows[slot].cpu().numpy().copy()

        for i in range(n_batches):
            slot = i & 1
            if i >= 2:
                collect(i - 2)
            e.search_knn_dev_async(Qd[i].data_ptr(), B, k, rows[slot].data_ptr(), scores[slot].data_ptr(), 0, slot,
                                   flags[slot].data_ptr())
            e.async_join(slot, side.cuda_stream)
            with torch.cuda.stream(side):
                joined[slot].copy_(rows[slot])
            if i == 5:          # a blocking search while both slots are busy: ordered behind them, same answer
                r, _ = e.search_knn(Qs[0], k)
                assert np.array_equal(r, want[0])
        collect(n_batches - 2)
        collect(n_batches - 1)
        for i in range(n_batches):
            assert np.array_equal(got[i], want[i]), (path, i)
        e.set_async_overlap(False)
        r, _ = e.search_knn(Qs[1], k)
        assert np.array_equal(r, want[1])


def _bf16_residual(X, chunk=16384):
    """||x - bf16(x)|| / ||x|| per row: what store_convert_kernel raises the store's rho_x to."""
    import torch
    out = []
    for i in range(0, X.shape[0], chunk):
        t = torch.from_numpy(X[i:i + chunk])
        d = (t - t.to(torch.bfloat16).to(torch.float32)).double()
        out.append((d.norm(dim=1) / t.double().norm(dim=1)).numpy())
    return np.concatenate(out)


def test_overlapped_async_slots_after_an_append_equal_the_oracle():
    """RASS_OPT_ASYNC_OVERLAP with an append between overlapped rounds.  Every element of the appended rows sits just
    below a bf16 rounding midpoint, so their rounding residual is larger than any row's stored before and the store's
    rho_x (the certificate's allowance for the fp32 rows) rises; they are near copies of the later queries, so they
    enter those queries' top-k.  Both slots go on after the append, and every batch returns the oracle's ids over the
    grown corpus."""
    import torch
    B, k, n_before, n_batches = 64, 10, 4, 10
    X = synth.embeddings(150000, 1024, 81)
    Qs = [synth.embeddings(B, 1024, 82 + i) for i in range(n_batches)]
    rng = np.random.default_rng(83)
    later = np.concatenate(Qs[n_before:])
    block = np.concatenate([later + s / 32 * rng.standard_normal(later.shape, dtype=np.float32) for s in (0.3, 0.5, 0.7)])
    block = ((block.view(np.uint32) & 0xFFFF0000) | 0x7FFF).view(np.float32)
    assert _bf16_residual(block).min() > _bf16_residual(X).max()
    X_all = np.concatenate([X, block])
    want = [knn.knn_exact(X if i < n_before else X_all, Q, k)[0] for i, Q in enumerate(Qs)]
    assert all(((w >= X.shape[0]).sum(axis=1) >= 3).all() for w in want[n_before:])
    with _engine(dim=1024) as e:
        e.append(X)
        e.set_async_overlap(True)
        Qd = [torch.from_numpy(Q).cuda() for Q in Qs]
        rows = [torch.full((B, k), -7, dtype=torch.int64, device="cuda") for _ in range(2)]
        scores = [torch.empty((B, k), dtype=torch.float32, device="cuda") for _ in range(2)]
        flags = [torch.empty(1, dtype=torch.int64, device="cuda") for _ in range(2)]
        torch.cuda.synchronize()
        got = [None] * n_batches

        def collect(i):
            final, st = e.search_knn_dev_wait(i & 1)
            assert final and int(flags[i & 1].item()) == 0, (i, st)
            got[i] = rows[i & 1].cpu().numpy().copy()

        for i in range(n_batches):
            if i == n_before:           # both slots collected, then the append
                collect(i - 2)
                collect(i - 1)
                e.append(block)
            elif i >= 2 and got[i - 2] is None:
                collect(i - 2)
            e.search_knn_dev_async(Qd[i].data_ptr(), B, k, rows[i & 1].data_ptr(), scores[i & 1].data_ptr(), 0, i & 1,
                                   flags[i & 1].data_ptr())
        collect(n_batches - 2)
        collect(n_batches - 1)
    for i in range(n_batches):
        assert np.array_equal(got[i], want[i]), i


def test_properties_at_2m_rows_all_paths_agree():
    """Larger than the oracle can check in seconds: size-independent properties instead.  On 2M device-generated
    rows every scan path returns the same ids for the same queries, the fp64 scan (the definition) agrees on a
    sample, scores are sorted, ids are distinct, and tombstoning a query's best row shifts its list up by one."""
    import torch
    import rassengine_b200 as rb
    n, d = 2_000_000, 1024
    with _engine(dim=d, capacity_rows=n) as e:
        g = torch.Generator(device="cuda").manual_seed(99)
        for c0 in range(0, n, 500_000):
            x = torch.randn((500_000, d), generator=g, device="cuda")
            x /= x.norm(dim=1, keepdim=True) + 1e-9
            torch.cuda.synchronize()
            e.append_dev(x.data_ptr(), x.shape[0])
            del x
        q = torch.randn((300, d), generator=g, device="cuda")

        def run(path, B, k):
            e.set_path(path)
            rows = torch.empty((B, k), dtype=torch.int64, device="cuda")
            sc = torch.empty((B, k), dtype=torch.float32, device="cuda")
            st = e.search_knn_dev(q.data_ptr(), B, k, rows.data_ptr(), sc.data_ptr())
            assert st["n_fallback"] == 0 and st["n_certified"] == B, st
            return rows.cpu().numpy(), sc.cpu().numpy()

        for k in (10, 100):
            r_gemm, s_gemm = run(rb.PATH_GEMM, 300, k)
            r_umma, s_umma = run(rb.PATH_UMMA, 130, k)
            r_str, s_str = run(rb.PATH_STREAM, 3, k)
            e.set_path(rb.PATH_EXACT)
            rows = torch.empty((4, k), dtype=torch.int64, device="cuda")
            sc = torch.empty((4, k), dtype=torch.float32, device="cuda")
            e.search_knn_dev(q.data_ptr(), 4, k, rows.data_ptr(), sc.data_ptr())
            assert np.array_equal(r_gemm[:130], r_umma) and np.array_equal(r_gemm[:3], r_str)
            assert np.array_equal(r_gemm[:4], rows.cpu().numpy())
            np.testing.assert_array_equal(s_gemm[:130], s_umma)            # same fp64 rerank -> same float scores
            assert (np.diff(s_gemm, axis=1) <= 0).all()
            assert all(len(set(r.tolist())) == k for r in r_gemm) and r_gemm.min() >= 0 and r_gemm.max() < n
        # the CPU oracle over all 2M rows (read back from the device store) for 8 of the queries, top-100: the merged
        # chain "fast path == fp64 GPU scan == CPU oracle" closed at a size the 100k fixtures do not reach
        qh = q[:8].cpu().numpy()
        want_rows, _, want_scores = knn.knn_exact_stream(
            ((c0, e.read_rows(c0, 250_000)) for c0 in range(0, n, 250_000)), qh, 100)
        _check(r_gemm[:8], s_gemm[:8], want_rows, want_scores)
        best = int(r_gemm[0, 0])
        e.tombstone(best)
        r2, _ = run(rb.PATH_UMMA, 64, 10)
        r_before, _ = r_gemm[:64, :], None
        assert best not in r2[0].tolist() and r2[0, :9].tolist() == r_before[0, 1:10].tolist()
        for b in range(1, 64):
            if best not in r_before[b, :10].tolist():
                assert r2[b].tolist() == r_before[b, :10].tolist()


def test_edge_shapes_and_degenerate_indices():
    """Ragged batch sizes across the path thresholds, k = 1 and k = 128, tiny / emptied indices, filters that pass
    nothing -- through the AUTO path selection, the way a caller reaches them."""
    import rassengine_b200 as rb
    X = synth.embeddings(3000, 256, 91)
    Qall = synth.embeddings(300, 256, 92)
    with _engine(dim=256) as e:
        e.append(X)
        for B, k in ((1, 1), (2, 128), (63, 7), (64, 10), (65, 10), (129, 33), (257, 1), (300, 128)):
            want_rows, _, want_scores = knn.knn_exact(X, Qall[:B], k)
            rows, scores = e.search_knn(Qall[:B], k)
            _check(rows, scores, want_rows, want_scores)
        with pytest.raises(rb.RassError):
            e.search_knn(Qall[:1], 129)                      # k beyond RASS_MAX_K
        # a filter nothing passes, as an exact pre-filter
        e.set_knn_prefilter(True)
        e.set_row_filter(np.zeros(3000, dtype=np.uint8))
        for B in (1, 40, 100):
            rows, scores = e.search_knn(Qall[:B], 5)
            assert (rows == -1).all() and (scores == 0).all()
        e.set_row_filter_rows(np.array([7, 2999, 11], dtype=np.int64), 3000)      # the same filter as a row list
        rows, _ = e.search_knn(Qall[:3], 5)
        assert all(sorted(r[:3].tolist()) == [7, 11, 2999] and (r[3:] == -1).all() for r in rows)
        e.set_row_filter(None)
        e.set_knn_prefilter(False)
        for r in range(3000):
            if r % 1000 != 5:
                e.tombstone(r)                               # three live rows left
        for B in (1, 30, 200):
            rows, _ = e.search_knn(Qall[:B], 10)
            assert all(sorted(r[:3].tolist()) == [5, 1005, 2005] and (r[3:] == -1).all() for r in rows)
    with _engine(dim=256) as e:                              # fewer rows than one tile, more queries than rows
        e.append(X[:5])
        want_rows, _, want_scores = knn.knn_exact(X[:5], Qall[:70], 5)
        rows, scores = e.search_knn(Qall[:70], 8)
        _check(rows[:, :5], scores[:, :5], want_rows, want_scores)
        assert (rows[:, 5:] == -1).all()
