"""BASELINE.json configs[3]: hybrid BM25 multi_match + vector fusion over 5M synthetic FHIR-narrative-shaped chunks
(~30k-term Zipf vocabulary), top-10 -- `python bench.py --workload cfg4`, and the `hybrid` extra of the default line.

One step = one batch of 64 hybrid queries (app/main.py:1574-1598 for chunk documents: S(d) = 4.5 * BM25(unstructuredText)
+ 2.0 * [d in kNN_10] * knn_score) answered exactly: the kNN clause is one corpus pass of the tcgen05 scan (10.24 GB of
bf16 rows), the text clauses one hybrid_tile_fast_kernel launch over the CSR postings, then the per-query select.

`value` = queries/s with the query vectors resident in HBM and results left on the device (rass_search_knn_dev_async +
rass_fuse_hybrid_dev, two batches in flight: the corpus pass of batch i+1 is queued before the host turns to the text
clauses of batch i; the term-id lists, a few hundred bytes per query, come from the host in both arms);
`e2e` = the same batch through rass_search_hybrid: host vectors in, host (row, score) lists out.
`parity`: fused ids and float32 scores against oracle.bm25 + oracle.fusion over the same postings, with the kNN clause
of the oracle taken from oracle.knn over all rows read back from the device store (nothing from the GPU's own search).
"""
from __future__ import annotations

import json
import os
import time

import numpy as np

V, DIM, K = 30000, 1024, 10
W_TEXT, W_KNN = 4.5, 2.0
SEED_TEXT, SEED_CORPUS, SEED_QUERIES = 4242, 1234, 5678


def build_text_corpus(dev, n_docs, engine=None, ingest=None):
    """Zipf(1.07) term ids over a 30k vocabulary, clipped-lognormal lengths (median 120, max 512 = CHUNK_SIZE,
    app/main.py:79), generated on the device (SURVEY.md 8d).  With an engine, every 250k-row slice of the token stream
    goes through the product's ingest (rass_text_add_rows_dev: a device-side segment per bulk; the caller commits).
    Independently of that the same tokens are sorted into CSR with torch ops -- the host arrays the oracle scores and the
    cross-check of the ingest."""
    import torch
    g = torch.Generator(device=dev).manual_seed(SEED_TEXT)
    p = 1.0 / torch.arange(1, V + 1, device=dev, dtype=torch.float64) ** 1.07
    p = (p / p.sum()).float()
    doclen = torch.empty(n_docs, dtype=torch.int32, device=dev)
    keys = []
    step = 250_000
    for c0 in range(0, n_docs, step):
        m = min(step, n_docs - c0)
        ln = torch.exp(torch.randn(m, generator=g, device=dev) * 0.6 + np.log(120.0)).round().clamp_(1, 512).to(torch.int64)
        doclen[c0:c0 + m] = ln.to(torch.int32)
        terms = torch.multinomial(p, int(ln.sum()), replacement=True, generator=g)
        if engine is not None:
            rows = torch.arange(c0, c0 + m, device=dev, dtype=torch.int64)
            tok_indptr = torch.zeros(m + 1, dtype=torch.int64, device=dev)
            tok_indptr[1:] = torch.cumsum(ln, 0)
            t32 = terms.to(torch.int32)
            torch.cuda.synchronize()
            t_i = time.perf_counter()
            engine.text_add_rows_dev(0, rows.data_ptr(), m, tok_indptr.data_ptr(), t32.data_ptr())
            if ingest is not None:
                ingest["add_rows_s"] = ingest.get("add_rows_s", 0.0) + time.perf_counter() - t_i
                ingest["tokens"] = ingest.get("tokens", 0) + int(t32.numel())
                ingest["bulks"] = ingest.get("bulks", 0) + 1
            del rows, tok_indptr, t32
        docs = torch.repeat_interleave(torch.arange(c0, c0 + m, device=dev), ln)
        k_, cnt = torch.unique(terms * n_docs + docs, return_counts=True)
        keys.append((k_, cnt.clamp_(max=65535).to(torch.int16)))
        del terms, docs
    key = torch.cat([k for k, _ in keys])
    tfv = torch.cat([c for _, c in keys])
    del keys
    order = torch.argsort(key)           # term-major, doc ascending within a term
    key, tfv = key[order], tfv[order]
    del order
    term_of = key // n_docs
    doc_of = (key - term_of * n_docs).to(torch.int32)
    indptr = torch.zeros(V + 1, dtype=torch.int64, device=dev)
    indptr[1:] = torch.cumsum(torch.bincount(term_of, minlength=V), 0)
    del key, term_of
    out = (indptr.cpu().numpy(), doc_of.cpu().numpy(), tfv.cpu().numpy().view(np.uint16),
           doclen.cpu().numpy().astype(np.uint32))
    del doc_of, tfv, indptr, doclen
    torch.cuda.empty_cache()
    return out


def build_engine(dev, n_docs, csr=None):
    """csr = None: the postings come through the device-side ingest (build_index)."""
    import torch
    import rassengine_b200 as rb
    e = rb.Engine(dim=DIM, device=dev.index or 0, capacity_rows=n_docs)
    e.set_stream(torch.cuda.current_stream().cuda_stream)      # the CUDA events of the timed loops see the engine's work
    for c0 in range(0, n_docs, 500_000):
        m = min(500_000, n_docs - c0)
        gg = torch.Generator(device=dev).manual_seed(SEED_CORPUS + c0 // 500_000)
        x = torch.randn((m, DIM), generator=gg, device=dev)
        x /= x.norm(dim=1, keepdim=True) + 1e-9
        torch.cuda.synchronize()
        e.append_dev(x.data_ptr(), m)
        del x
    if csr is not None:
        e.bm25_build(*csr)
    return e


def build_index(dev, n_docs):
    """-> (engine, host csr, ingest report).  The engine's postings are built by the product's own device-side ingest
    from the raw token stream and committed once (what a bulk load followed by a refresh does); the torch-sorted CSR of
    the same tokens must match it array for array."""
    e = build_engine(dev, n_docs)
    ingest = {}
    csr = build_text_corpus(dev, n_docs, engine=e, ingest=ingest)
    t_c = time.perf_counter()
    e.text_commit([V], n_docs)
    ingest["commit_s"] = time.perf_counter() - t_c
    t_q = time.perf_counter()
    e.search_hybrid(None, [[1, 2, 3]], W_TEXT, 0.0, K)
    ingest["first_text_query_s"] = time.perf_counter() - t_q
    indptr, doc, tf, doclen, _ = e.text_export()
    ingest["equals_torch_sorted_csr"] = bool(np.array_equal(indptr, csr[0]) and np.array_equal(doc, csr[1]) and
                                             np.array_equal(tf, csr[2]) and np.array_equal(doclen[0], csr[3]))
    ingest["tokens_per_s"] = ingest["tokens"] / max(ingest["add_rows_s"] + ingest["commit_s"], 1e-9)
    ingest["note"] = ("raw token ids -> rass_text_add_rows_dev per 250k-row bulk (radix sort by term + run-length on the "
                      "device) -> one rass_text_commit; first_text_query_s is the first hybrid call after the commit")
    del indptr, doc, tf, doclen
    return e, csr, ingest


def text_queries(nq, seed):
    """3-12 term ids per query, Zipf(1.07) with the 50 most frequent terms down-weighted 10x (SURVEY.md 8d) -- the same
    distribution as oracle.synth.text_queries, restated here because the product path does not import oracle/."""
    rng = np.random.default_rng(seed)
    pr = 1.0 / np.power(np.arange(1, V + 1, dtype=np.float64), 1.07)
    pr[:50] *= 0.1
    cdf = np.cumsum(pr / pr.sum())
    out = []
    for _ in range(nq):
        m = int(rng.integers(3, 13))
        t = np.minimum(np.searchsorted(cdf, rng.random(m), side="left"), V - 1)
        out.append([int(v) for v in t])
    return out


def pack_terms(qterms):
    indptr = np.zeros(len(qterms) + 1, dtype=np.int32)
    indptr[1:] = np.cumsum([len(t) for t in qterms])
    return indptr, np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.int32) for t in qterms]), dtype=np.int32)


def measure(e, dev, csr, n_docs, B, steps, warmup, n_check, cpu_baseline=True, cpu_parity=True):
    import torch
    indptr = csr[0]
    n_sets = 4
    gq = torch.Generator(device=dev).manual_seed(SEED_QUERIES)
    q_dev = [torch.randn((B, DIM), generator=gq, device=dev) for _ in range(n_sets)]
    q_host = [q.cpu().pin_memory() for q in q_dev]
    qterms = [text_queries(B, SEED_TEXT + 1 + i) for i in range(n_sets)]
    packed = [pack_terms(t) for t in qterms]
    postings = [float(sum(int(indptr[t + 1] - indptr[t]) for q in qs for t in q)) for qs in qterms]
    knn_rows = torch.empty((B, K), dtype=torch.int64, device=dev)
    knn_scores = torch.empty((B, K), dtype=torch.float32, device=dev)
    out_rows = torch.empty((B, K), dtype=torch.int64, device=dev)
    out_scores = torch.empty((B, K), dtype=torch.float32, device=dev)
    acc = {"scan_ms": 0.0, "text_ms": 0.0, "launches": 0, "n": 0, "order_free": 0, "scan_bytes": 0}

    # two batches in flight, like the kNN loop of bench.py: the kNN clause of batch i is enqueued (rass_search_knn_dev_async,
    # its own stream and workspace) before the host turns to the text clauses of batch i-1, so the corpus pass of the
    # next batch is already queued when the text kernel ends -- no host round trip between the two big kernels
    e.set_async_overlap(True)
    knn_rows2 = [knn_rows, torch.empty_like(knn_rows)]
    knn_scores2 = [knn_scores, torch.empty_like(knn_scores)]

    def finish(j):
        s, slot = j % n_sets, j & 1
        final, st = e.search_knn_dev_wait(slot)
        if not final:                      # a certificate failed (none on this corpus): the blocking call re-scans
            st = e.search_knn_dev(q_dev[s].data_ptr(), B, K, knn_rows2[slot].data_ptr(), knn_scores2[slot].data_ptr())
        acc["scan_ms"] += st["scan_ms"]
        acc["scan_bytes"] += st["bytes_streamed"]      # the engine's count: 1 or 2 bytes per element, by the pass it ran
        acc["launches"] += st["launches"]
        e.fuse_hybrid_dev(B, packed[s], W_TEXT, knn_rows2[slot].data_ptr(), knn_scores2[slot].data_ptr(), W_KNN, K,
                          out_rows.data_ptr(), out_scores.data_ptr())
        st = e.last_hybrid_stats
        acc["text_ms"] += st["finish_ms"]
        acc["launches"] += st["launches"]
        acc["order_free"] += int(bool(st["path"] & 0x100))
        acc["n"] += 1

    def step_dev(i):
        s, slot = i % n_sets, i & 1
        e.search_knn_dev_async(q_dev[s].data_ptr(), B, K, knn_rows2[slot].data_ptr(), knn_scores2[slot].data_ptr(), 0, slot, 0)
        if i > 0:
            finish(i - 1)

    def step_e2e(i):
        s = i % n_sets
        return e.search_hybrid(q_host[s].numpy(), packed[s], W_TEXT, W_KNN, K)

    def step_text(i):
        s = i % n_sets
        e.fuse_hybrid_dev(B, packed[s], W_TEXT, 0, 0, 0.0, K, out_rows.data_ptr(), out_scores.data_ptr())
        acc["text_ms"] += e.last_hybrid_stats["finish_ms"]
        acc["n"] += 1

    def timed(fn, n, w, flush=None):
        for i in range(w):
            fn(i)
        if flush:
            flush(w - 1)
        for kk in acc:
            acc[kk] = 0.0 if kk.endswith("_ms") else 0
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for i in range(n):
            fn(i)
        if flush:
            flush(n - 1)                   # the last batch completes inside the timed region
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), t0, time.time()

    ms_dev, t0, t1 = timed(step_dev, steps, warmup, flush=finish)
    last = {"rows": out_rows.cpu().numpy(), "scores": out_scores.cpu().numpy()}     # the fused lists of the last step
    dev_acc = dict(acc)

    # the text kernel's own duration: inside the pipelined loop its events also span the next batch's corpus pass (queued
    # first, it takes the SMs first), so it is timed in a short serialised pass -- same kernels, same inputs
    def step_serial(i):
        s = i % n_sets
        e.search_knn_dev(q_dev[s].data_ptr(), B, K, knn_rows.data_ptr(), knn_scores.data_ptr())
        e.fuse_hybrid_dev(B, packed[s], W_TEXT, knn_rows.data_ptr(), knn_scores.data_ptr(), W_KNN, K,
                          out_rows.data_ptr(), out_scores.data_ptr())
        acc["text_ms"] += e.last_hybrid_stats["finish_ms"]
        acc["n"] += 1

    timed(step_serial, min(steps, 10), 2)
    dev_acc["text_ms"], dev_acc["text_n"] = acc["text_ms"], acc["n"]
    ms_e2e, _, _ = timed(step_e2e, steps, warmup)
    ms_text, _, _ = timed(step_text, steps, min(warmup, 3))
    text_acc = dict(acc)
    # one query per call (what /ask issues), host buffers
    one = (q_host[0][:1].numpy(), pack_terms(qterms[0][:1]))
    ms_one, _, _ = timed(lambda i: e.search_hybrid(one[0], one[1], W_TEXT, W_KNN, K), min(steps, 50), 3)
    n_one = min(steps, 50)

    res = {"B": B, "k": K, "steps": steps, "warmup": warmup, "ms_dev": ms_dev, "ms_e2e": ms_e2e, "t0": t0, "t1": t1,
           "qps": steps * B / (ms_dev * 1e-3), "qps_e2e": steps * B / (ms_e2e * 1e-3),
           "qps_text_only": steps * B / (ms_text * 1e-3), "qps_one_query_per_call": n_one / (ms_one * 1e-3),
           "scan_ms": dev_acc["scan_ms"] / max(1, dev_acc["n"]),
           "scan_bytes": dev_acc["scan_bytes"] / max(1, dev_acc["n"]), "text_ms": dev_acc["text_ms"] / max(1, dev_acc["text_n"]),
           "text_only_kernel_ms": text_acc["text_ms"] / max(1, text_acc["n"]),
           "launches": int(dev_acc["launches"]), "order_free_batches": int(dev_acc["order_free"]),
           "mean_postings_per_query": float(np.mean(postings)) / B, "postings_per_batch": float(np.mean(postings)),
           "term_bytes": int(np.mean([p[0].nbytes + p[1].nbytes for p in packed])), "last_outputs": last}

    # ---- parity against the CPU oracle at full size (test infrastructure, outside the timed region) ----
    if cpu_parity:
        import bench
        from oracle import bm25, fusion
        t_p = time.perf_counter()
        n_check = min(n_check, B)
        rows_g, scores_g = step_e2e(0)
        rows_t, scores_t = e.search_hybrid(None, (packed[0][0][:n_check + 1].copy(), packed[0][1]), W_TEXT, W_KNN, K)
        idx = bm25.BM25Index(*csr)
        Qc = q_dev[0][:n_check].cpu().numpy()
        workers = max(1, min(6, (os.cpu_count() or 4) - 1))
        kr, kcos = bench.cpu_oracle_topk(e, 0, n_docs, Qc, K, workers)
        from oracle import knn as oknn
        ids_ok = scores_ok = text_ok = 0
        for b in range(n_check):
            ks = oknn.score_from_cos(kcos[b])
            wr, ws = fusion.hybrid(idx, qterms[0][b], kr[b], ks, W_TEXT, W_KNN, K)
            ids_ok += int(rows_g[b, :len(wr)].tolist() == wr.tolist())
            scores_ok += int(np.allclose(scores_g[b, :len(wr)], ws, rtol=2e-6, atol=0))
            tr, ts = bm25.topk(idx.score(qterms[0][b], boost=W_TEXT), K)
            text_ok += int(rows_t[b].tolist() == tr.tolist() and scores_t[b].tolist() == ts.tolist())
        res["parity"] = {"oracle": "oracle.bm25 + oracle.fusion over the same postings; kNN clause from oracle.knn over all "
                                   f"{n_docs} rows read back from the device store",
                         "queries_checked_cpu": n_check, "fused_ids_equal_cpu_oracle": ids_ok == n_check,
                         "fused_scores_within_2e-6": scores_ok == n_check, "text_only_bit_identical": text_ok == n_check,
                         "seconds": round(time.perf_counter() - t_p, 1)}
        # ---- CPU baseline: the oracle port of the same step on a bounded sample ----
        if cpu_baseline:
            res["cpu_baseline"] = cpu_step_qps(e, idx, qterms[0], q_dev[0].cpu().numpy(), n_docs, B)
    return res


def cpu_step_qps(e, idx, qterms, Q, n_docs, B, sample_rows=1_000_000, sample_queries=8):
    """numpy port of one hybrid batch: fp32 sgemm + argpartition kNN over `sample_rows` rows (scaled to n_docs) plus
    oracle BM25 scoring + fusion top-k of `sample_queries` queries (scaled to B)."""
    import bench
    from oracle import bm25, fusion, knn
    sample_rows = min(sample_rows, n_docs)
    Xs = e.read_rows(0, sample_rows)
    bench.cpu_scan_time(Xs[:20000], Q, K)
    t_knn = bench.cpu_scan_time(Xs, Q, K, repeats=2) * (n_docs / float(sample_rows))
    rows, scores = knn.knn_fp32_baseline(Xs, Q[:sample_queries], K)
    t0 = time.perf_counter()
    for b in range(sample_queries):
        fusion.hybrid(idx, qterms[b], rows[b], scores[b], W_TEXT, W_KNN, K)
    t_text = (time.perf_counter() - t0) * (B / float(sample_queries))
    return {"value": B / (t_knn + t_text), "unit": "queries/s", "cores": bench.blas_threads(), "kind": "port",
            "sample": f"numpy port of one {B}-query hybrid batch: kNN clause = fp32 sgemm + argpartition over the first "
                      f"{sample_rows} of {n_docs} rows scaled x{n_docs / float(sample_rows):g} ({t_knn:.2f} s), text + "
                      f"fusion = oracle.bm25 / oracle.fusion for {sample_queries} queries scaled x"
                      f"{B / float(sample_queries):g} ({t_text:.2f} s)"}


def roofline_block(res, n_docs):
    import bench
    peak_hbm, _, src = bench.peaks()
    scan_bytes = float(res["scan_bytes"])
    text_bytes = res["postings_per_batch"] * 7.0            # doc id 4 B + tf 2 B + norm byte per posting (SURVEY.md 8d)
    scan = {"kernel": "scan_umma_kernel", "ms": res["scan_ms"], "algorithmic_bytes_per_launch": scan_bytes,
            "achieved_gbs": scan_bytes / (res["scan_ms"] * 1e-3) / 1e9 if res["scan_ms"] else None}
    text = {"kernel": "hybrid_tile_fast_kernel + hybrid_select_kernel", "ms": res["text_ms"],
            "timed": "serialised pass after the timed loop (in the pipelined loop the kernel waits behind the next batch's "
                     "corpus pass)",
            "algorithmic_bytes_per_launch": text_bytes, "postings_per_launch": res["postings_per_batch"],
            "achieved_gbs": text_bytes / (res["text_ms"] * 1e-3) / 1e9 if res["text_ms"] else None,
            "postings_per_s": res["postings_per_batch"] / (res["text_ms"] * 1e-3) if res["text_ms"] else None}
    dom = scan if res["scan_ms"] >= res["text_ms"] else text
    return {"bound": "hbm", "achieved": dom["achieved_gbs"], "peak": peak_hbm, "unit": "GB/s",
            "frac": dom["achieved_gbs"] / peak_hbm if dom["achieved_gbs"] else None, "traffic": None,
            "peak_source": src, "kernel": dom["kernel"], "kernel_ms": dom["ms"],
            "algorithmic_bytes_per_launch": dom["algorithmic_bytes_per_launch"],
            "kernels": {"knn_scan": dict(scan, frac=scan["achieved_gbs"] / peak_hbm if scan["achieved_gbs"] else None),
                        "bm25_fusion": dict(text, frac=text["achieved_gbs"] / peak_hbm if text["achieved_gbs"] else None)},
            "step_frac_of_knn_ceiling": (scan_bytes / (peak_hbm * 1e9)) / ((res["ms_dev"] / res["steps"]) * 1e-3)}


def workload_name(n_docs, B):
    return (f"cfg4: hybrid BM25 multi_match + knn fusion (4.5 * BM25(unstructuredText) + 2.0 * knn), {n_docs} synthetic "
            f"chunks x {DIM}, vocab {V} Zipf(1.07), top-{K}, query batch {B}")


def run_ours(a, world, rank, dev):
    import bench
    if world > 1:
        raise SystemExit("--workload cfg4 runs on one GPU (row-sharded hybrid: tests/sharded_worker.py)")
    sampler = bench.ClockSampler(dev.index or 0)
    n_docs, B = a.rows, a.batch
    t0 = time.time()
    e, csr, ingest = build_index(dev, n_docs)
    setup_s = time.time() - t0
    res = measure(e, dev, csr, n_docs, B, a.steps, a.warmup, 8, cpu_baseline=not a.no_cpu_baseline,
                  cpu_parity=not a.no_cpu_parity)
    sampler.stop()
    if a.dump_outputs:
        bench.dump_outputs(a.dump_outputs, res["last_outputs"])
    out = {"metric": "exact hybrid (BM25 multi_match + kNN fusion) top-10 QPS @5M chunks (ids identical to the CPU oracle)",
           "value": res["qps"], "unit": "queries/s", "n_gpus": 1, "steps": a.steps, "warmup": a.warmup,
           "ms_per_step": res["ms_dev"] / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "bf16 scan + fp64 rerank (kNN), f32 BM25 ops summed in f64 (text)", "data": "synthetic",
           "config": {"workload": workload_name(n_docs, B), "rows": n_docs, "dim": DIM, "batch": B, "k": K,
                      "nnz": int(csr[0][-1]), "mean_postings_per_query": res["mean_postings_per_query"],
                      "l2": "inputs larger than L2: every step streams the 10.24 GB bf16 shard and ~2 GB of postings"},
           "e2e": {"value": res["qps_e2e"], "unit": "queries/s", "h2d_bytes_per_step": B * DIM * 4 + res["term_bytes"],
                   "d2h_bytes_per_step": B * K * 12, "ms_per_step": res["ms_e2e"] / a.steps},
           "gpu_launches": res["launches"], "roofline": roofline_block(res, n_docs),
           "text_only_qps": res["qps_text_only"], "text_only_kernel_ms": res["text_only_kernel_ms"],
           "one_query_per_call_qps": res["qps_one_query_per_call"], "order_free_batches": res["order_free_batches"],
           "parity": res.get("parity"), "ingest": ingest, "setup_s": round(setup_s, 1),
           "clocks": bench.ClockSampler.summarise(sampler.window(res["t0"], res["t1"]), "timed region")}
    if "cpu_baseline" in res:
        out["cpu_baseline"] = res["cpu_baseline"]
    print(json.dumps(out), flush=True)
    e.close()


def run_extra(dev, n_docs=5_000_000, B=64, steps=20, warmup=5):
    """The `hybrid` extra of the default bench line: configuration 4 at full size, short."""
    t0 = time.time()
    e, csr, ingest = build_index(dev, n_docs)
    setup_s = time.time() - t0
    res = measure(e, dev, csr, n_docs, B, steps, warmup, 8, cpu_baseline=False)
    e.close()
    rl = roofline_block(res, n_docs)
    return {"workload": workload_name(n_docs, B), "qps": res["qps"], "qps_e2e": res["qps_e2e"],
            "ms_per_batch": res["ms_dev"] / steps, "qps_text_only": res["qps_text_only"],
            "qps_one_query_per_call": res["qps_one_query_per_call"], "knn_scan_ms": res["scan_ms"],
            "bm25_fusion_ms": res["text_ms"], "text_only_kernel_ms": res["text_only_kernel_ms"],
            "postings_per_s": rl["kernels"]["bm25_fusion"]["postings_per_s"],
            "bm25_gbs": rl["kernels"]["bm25_fusion"]["achieved_gbs"],
            "frac_of_knn_ceiling": rl["step_frac_of_knn_ceiling"], "order_free_batches": res["order_free_batches"],
            "parity": res.get("parity"), "ingest": ingest, "setup_s": round(setup_s, 1)}


def run_reference(a):
    """CPU arm of cfg4: the oracle port of one hybrid batch on a bounded sample (numpy kNN + oracle BM25 + fusion)."""
    import bench
    from oracle import bm25, fusion, knn, synth
    t_start = time.perf_counter()
    n_docs, B = a.rows, a.batch
    n_text = min(n_docs, 500_000)                      # postings scale linearly with the documents
    csr = synth.text_corpus(n_text, vocab=V, seed=SEED_TEXT)
    idx = bm25.BM25Index(*csr)
    qterms = text_queries(B, SEED_TEXT + 1)
    n_rows = min(n_docs, 500_000)
    X = synth.embeddings(n_rows, DIM, SEED_CORPUS)
    Q = synth.embeddings(B, DIM, SEED_QUERIES)
    nq = 8

    def step():
        t0 = time.perf_counter()
        rows, scores = knn.knn_fp32_baseline(X, Q, K)
        t_knn = (time.perf_counter() - t0) * (n_docs / float(n_rows))
        t0 = time.perf_counter()
        for b in range(nq):
            fusion.hybrid(idx, qterms[b], rows[b], scores[b], W_TEXT, W_KNN, K)
        return t_knn + (time.perf_counter() - t0) * (B / float(nq)) * (n_docs / float(n_text))

    for _ in range(a.warmup):
        step()
    t_step = float(np.mean([step() for _ in range(a.steps)]))
    qps = B / t_step
    cores = bench.blas_threads()
    out = {"impl": "reference", "metric": "exact hybrid (BM25 multi_match + kNN fusion) top-10 QPS @5M chunks (ids "
           "identical to the CPU oracle)", "value": qps, "unit": "queries/s", "n_gpus": a.gpus, "steps": a.steps,
           "warmup": a.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload_name(n_docs, B), "rows": n_docs, "dim": DIM, "batch": B, "k": K},
           "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
                            "sample": f"per step: numpy fp32 sgemm + argpartition over {n_rows} of {n_docs} rows (scaled) + "
                                      f"oracle.bm25 / oracle.fusion of {nq} of {B} queries over {n_text} of {n_docs} "
                                      f"documents (scaled); {time.perf_counter() - t_start:.0f} s in all"},
           "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)
