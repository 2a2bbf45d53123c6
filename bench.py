#!/usr/bin/env python
"""Headline benchmark: exact top-10 QPS over a 10M x 1024 corpus (BASELINE.json configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg2|cfg3|cfg4|cfg5] [--rows R] [--batch B] [--k K] [--dump-outputs DIR]
    torchrun --nproc-per-node N ... bench.py --gpus N ...          (one rank per GPU, NCCL)

--workload selects the BASELINE.json configuration: cfg2 (default, the one the metric is quoted on: 10M x 1024,
batch 64, top-10, HBM roofline), cfg3 (10M x 1024, batch 8192, top-100, tensor roofline), cfg4 (hybrid BM25 + kNN
over 5M chunks, bench_hybrid.py) or cfg5 (100M x 1024 bf16 corpus row-sharded over >= 2 GPUs, batch 1024, top-10,
tensor roofline).  The default run also reports, as extras of the same JSON line, the batch-1, batch-1024 and
batch-8192/top-100 regimes of the same corpus (`batch1` / `batched`), a >= 2 s `sustained` loop, the hybrid
configuration at reduced scale (`hybrid`, N = 1) and configuration 5 (`cfg5`, N >= 2).

One step = one query batch (default 64 queries) answered exactly against the whole corpus.  The corpus is
synthetic (seeded N(0,1) rows, L2-normalised as app/main.py:1250-1251 does), generated on the device and
ingested through the engine's append path before the timed region.  With N GPUs the SAME 10M-row corpus is
row-sharded (strong scaling): local exact top-k, one NCCL all-gather of k candidates per query, device merge.

Prints ONE JSON line (rank 0).  `value` = queries/s with queries resident in HBM; `e2e` = the same through the
host-buffer API (pinned host queries in, host results out, copies inside the timed region); `roofline` = the
scan kernel's algorithmic bytes / its CUDA-event time against the measured HBM copy peak; `cpu_baseline` = the
numpy port of the reference's exact CPU scan on a bounded sample of the same workload; `parity` = the MERGED result
the timed loop returned against the fp64 CPU oracle run over the whole corpus (rows read back from every shard).

--dump-outputs DIR writes what the last timed step returned to its caller as DIR/rows.npy (global row ids, float64)
and DIR/scores.npy (float32), one row per query of that batch.  Corpus and queries are seeded, so two builds run with
the same arguments can be compared output for output.
"""
from __future__ import annotations

import os
import sys


def _early_env():
    """Thread / NCCL environment that has to be in place before numpy and torch load.  The CPU arm must not inherit
    torchrun's OMP_NUM_THREADS=1: it is the reference's CPU path with every host thread it can use."""
    argv = sys.argv
    ref = any(a == "--impl=reference" for a in argv) or any(
        a == "--impl" and i + 1 < len(argv) and argv[i + 1] == "reference" for i, a in enumerate(argv))
    if ref:
        n = str(os.cpu_count() or 1)
        for v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
            os.environ[v] = n
    elif int(os.environ.get("WORLD_SIZE", "1")) > 1:
        # communicator setup (rank / nranks lines) to stderr, so stdout stays the one JSON line -- whatever level the
        # environment asked for (at WARN / VERSION NCCL prints its version banner on stdout); RASS_NCCL_DEBUG overrides
        os.environ["NCCL_DEBUG"] = os.environ.get("RASS_NCCL_DEBUG", "INFO")
        os.environ["NCCL_DEBUG_SUBSYS"] = os.environ.get("RASS_NCCL_DEBUG_SUBSYS", "INIT")
        os.environ["NCCL_DEBUG_FILE"] = "/dev/stderr"


_early_env()

import argparse  # noqa: E402
import json  # noqa: E402
import subprocess  # noqa: E402
import threading  # noqa: E402
import time  # noqa: E402

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "exact top-10 QPS @10M x 1024 (cosine, ids identical to the fp64 CPU oracle)"
DIM = 1024
CHUNK = 500_000
SEED_CORPUS, SEED_QUERIES = 1234, 5678
N_CHECK = 8                      # queries per regime compared with the CPU oracle over the whole corpus
ARM_IDLE_S = 0.5                 # pause before the warm-up of the device-resident arm and of the e2e arm: both timed
                                 # regions are short bursts, and the second one must not inherit the first one's heat


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4", "cfg5"])
    ap.add_argument("--rows", type=int, default=None)
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--cpu-sample-rows", type=int, default=None)
    ap.add_argument("--cpu-budget-s", type=float, default=75.0, help="wall-clock budget of the reference arm")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-parity", action="store_true", help="skip the CPU-oracle check over the whole corpus")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (batch1, batched, hybrid, cfg5)")
    ap.add_argument("--sustained-s", type=float, default=2.5)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm scans a sample of the corpus")
    rows, batch, k = {"cfg2": (10_000_000, 64, 10), "cfg3": (10_000_000, 8192, 100), "cfg4": (5_000_000, 64, 10),
                      "cfg5": (100_000_000, 1024, 10)}[a.workload]
    a.rows = a.rows if a.rows is not None else rows
    a.batch = a.batch if a.batch is not None else batch
    a.k = a.k if a.k is not None else k
    a.bf16_only = a.workload == "cfg5"
    return a


def workload_name(a):
    store = ("bf16 corpus (the bf16 values are the data)" if a.bf16_only
             else "synthetic fp32 unit rows (bf16 scan shadow + fp64 rerank)")
    return f"{a.workload}: exact cosine top-{a.k}, {a.rows} x {DIM} {store}, query batch {a.batch}"


def scan_kernel_name(B):
    if B <= 1:
        return "scan_stream_kernel (128-bit streaming GEMV + warp select)"
    if B <= 64:
        return "scan_umma_kernel (TMA + tcgen05, 64 queries/pass)"
    return "scan_gemm_kernel (TMA + tcgen05 cta_group::2, 256 queries/pass)"


def make_config(a, world):
    """The `config` object of the JSON line -- the same dict for the GPU arm and the reference arm."""
    per = -(-a.rows // world)
    return {"workload": workload_name(a), "rows": a.rows, "dim": DIM, "batch": a.batch, "k": a.k,
            "sharding": f"row-sharded x{world}, one NCCL all-gather of k candidates per query" if world > 1
            else "single shard",
            "l2": "inputs larger than L2: every step streams the whole bf16 shard "
                  f"({per * DIM * 2 / 1e9:.2f} GB per GPU)",
            "scan_kernel": scan_kernel_name(a.batch),
            "loop": "each timed arm starts after 0.5 s of idle and its own warm-up; two batches in flight "
                    "(search_dev_async / wait): the exchange and host work of batch i "
                    "overlap the scan of batch i+1; the e2e arm is the same loop with pinned host queries in "
                    "and host results out"}


def peaks():
    """(HBM GB/s, bf16 TFLOP/s sustained, source)"""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), float(j.get("bf16_tflops_sustained", j["bf16_tflops"])), \
            "measured (MEASURED_PEAKS.json hbm_gbs / bf16_tflops_sustained)"
    return 6650.0, 1400.0, "fallback (B200_PROFILING.md)"


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(directory, arrays):
    """arrays: name -> [B, ...] host array, one row per query.  Written as <directory>/<name>.npy, float32 arrays as
    they are and everything else (row ids) as float64, which holds every row id exactly.  Above DUMP_LIMIT_BYTES in all,
    a fixed seeded sample of the queries is written instead, their indices in query_index.npy."""
    out = {n: np.asarray(v, dtype=np.float32 if v.dtype == np.float32 else np.float64) for n, v in arrays.items()}
    n_queries = next(iter(out.values())).shape[0]
    per_query = sum(v.nbytes for v in out.values()) // max(1, n_queries) + 8
    if per_query * n_queries > DUMP_LIMIT_BYTES:
        pick = np.sort(np.random.default_rng(0).choice(n_queries, DUMP_LIMIT_BYTES // per_query, replace=False))
        out = {n: v[pick] for n, v in out.items()}
        out["query_index"] = pick.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for n, v in out.items():
        np.save(os.path.join(directory, n + ".npy"), v)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons, sampled over the whole run; windows are cut out afterwards."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0, t1):
        return [r for t, r in self.rows if t0 <= t <= t1]

    def stop(self):
        if self.proc:
            self.proc.terminate()

    @staticmethod
    def summarise(lines, note=None):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in lines:
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except Exception:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0, "window": note}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm), "window": note}


# ---------------------------------------------------------------------------------------------------
# CPU arm: the numpy port of the reference's exact CPU scan (oracle.knn.knn_fp32_baseline)
# ---------------------------------------------------------------------------------------------------
def cpu_scan_time(X, Q, k, repeats=1):
    """Best wall time of fp32 sgemm + argpartition + sort of Q against X (oracle.knn.knn_fp32_baseline)."""
    from oracle import knn
    best = float("inf")
    for _ in range(repeats):
        t0 = time.perf_counter()
        knn.knn_fp32_baseline(X, Q, k)
        best = min(best, time.perf_counter() - t0)
    return best


def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([int(p.get("num_threads", 1)) for p in threadpool_info()] or [1])
    except Exception:
        return int(os.environ.get("OMP_NUM_THREADS", os.cpu_count() or 1))


def run_reference(a):
    """The reference's CPU path for this metric, every host thread in use, on a bounded sample of the same workload:
    each step scans `sample` of the rows (the time is scaled by rows / sample: the scan is linear in rows)."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    if a.workload == "cfg4":
        import bench_hybrid
        return bench_hybrid.run_reference(a)
    from oracle import knn, synth
    t_start = time.perf_counter()
    Q = synth.embeddings(a.batch, DIM, SEED_QUERIES)
    # size the sample so that warmup + steps fit the budget: calibrate on a small piece first
    cal_rows = min(a.rows, 100_000 if a.batch <= 64 else 10_000)
    Xc = synth.embeddings(cal_rows, DIM, SEED_CORPUS)
    knn.knn_fp32_baseline(Xc[: min(20000, cal_rows)], Q, a.k)                  # warm the BLAS threads
    rate = cal_rows / cpu_scan_time(Xc, Q, a.k, repeats=2)                     # rows/s at this batch
    n_pass = max(1, a.steps + a.warmup)
    if a.cpu_sample_rows is not None:
        sample = min(a.cpu_sample_rows, a.rows)
    else:
        sample = int(rate * a.cpu_budget_s / n_pass)
        sample = max(min(cal_rows, a.rows), min(sample, 2_000_000, a.rows))     # <= 8 GB of host rows
    X = Xc if sample == cal_rows else synth.embeddings(sample, DIM, SEED_CORPUS)
    for _ in range(a.warmup):
        cpu_scan_time(X, Q, a.k)
    times = [cpu_scan_time(X, Q, a.k) for _ in range(a.steps)]
    scale = a.rows / float(sample)
    t_step = float(np.mean(times)) * scale
    qps = a.batch / t_step
    cores = blas_threads()
    sample_desc = (f"numpy fp32 sgemm + argpartition (oracle.knn.knn_fp32_baseline, OpenBLAS on {cores} threads of "
                   f"{os.cpu_count()} cores) over {sample} of {a.rows} rows x {a.batch} queries per step, step time "
                   f"scaled x{scale:g} (the scan is linear in rows); {a.steps} steps after {a.warmup} warm-ups in "
                   f"{time.perf_counter() - t_start:.0f} s; oracle port of the exact CPU scan -- OpenSearch/HNSW "
                   "needs a JVM and FAISS is not installed, neither can be installed offline")
    out = {"impl": "reference", "metric": METRIC, "value": qps, "unit": "queries/s", "n_gpus": a.gpus,
           "steps": a.steps, "warmup": a.warmup, "ms_per_step": t_step * 1e3, "higher_is_better": True,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": make_config(a, max(world, a.gpus)),
           "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample_desc},
           "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


# ---------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------
def fill_shard(index, lo, hi, seed=SEED_CORPUS):
    """Device-side synthetic rows [lo, hi): chunk c of the global corpus is seeded seed + c, so the data is
    the same for every GPU count."""
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    c0 = lo // CHUNK
    while c0 * CHUNK < hi:
        g = torch.Generator(device=dev).manual_seed(seed + c0)
        x = torch.randn((CHUNK, DIM), generator=g, device=dev, dtype=torch.float32)
        x = x / (x.norm(dim=1, keepdim=True) + 1e-9)
        s = max(lo, c0 * CHUNK) - c0 * CHUNK
        e = min(hi, (c0 + 1) * CHUNK) - c0 * CHUNK
        part = x[s:e].contiguous()
        torch.cuda.synchronize()
        index.append_dev(part)
        del x, part
        c0 += 1


def cpu_oracle_topk(eng, lo, hi, Q, k, workers):
    """fp64 CPU oracle (oracle.knn.knn_exact) over THIS rank's rows [lo, hi), read back from the device store in
    pinned chunks: -> (global rows [B, k], key64 [B, k]).  Test infrastructure, outside every timed region."""
    import torch
    from concurrent.futures import ThreadPoolExecutor
    from oracle import knn
    step = 250_000
    n_buf = workers + 1
    bufs = [torch.empty((step, DIM), dtype=torch.float32).pin_memory() for _ in range(n_buf)]

    def work(X, base):
        r, key, _ = knn.knn_exact(X, Q, k)
        return np.where(r >= 0, r + base, -1), key

    futs = []
    with ThreadPoolExecutor(max_workers=workers) as ex:
        for i, c0 in enumerate(range(0, hi - lo, step)):
            if i >= n_buf:
                futs[i - n_buf].result()             # that chunk is done with the buffer about to be refilled
            n = min(step, hi - lo - c0)
            eng.read_rows_into(c0, n, bufs[i % n_buf].data_ptr())
            futs.append(ex.submit(work, bufs[i % n_buf].numpy()[:n], lo + c0))
        parts = [f.result() for f in futs]
    if not parts:
        return np.full((Q.shape[0], 0), -1, np.int64), np.zeros((Q.shape[0], 0))
    r, key, _ = knn.merge_topk(parts, k)
    return r, key


def oracle_parity(eng, lo, hi, world, rank, checks, workers):
    """checks: [(name, Q numpy [n, dim], k, gpu_rows numpy [n, k], gpu_scores numpy [n, k])] -- the MERGED results the
    timed loops returned.  Every rank runs the CPU oracle over its own rows, rank 0 merges the per-shard lists (the
    top-k of a union is the top-k of the per-part top-k) and compares.  -> dict on rank 0, None elsewhere."""
    import torch.distributed as dist
    from oracle import knn
    t0 = time.perf_counter()
    Qall = np.concatenate([c[1] for c in checks], axis=0)
    kmax = max(c[2] for c in checks)
    r_loc, key_loc = cpu_oracle_topk(eng, lo, hi, Qall, kmax, workers)
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, (r_loc, key_loc))
    else:
        gathered = [(r_loc, key_loc)]
    if rank != 0:
        return None
    rows, keys, scores = knn.merge_topk(gathered, kmax)
    out = {"oracle": "oracle.knn.knn_exact (fp64 keys of the stored fp32 values, (key desc, row asc)) over all "
                     f"{hi - lo if world == 1 else 'shards'} rows read back from the device store, per-shard lists "
                     "merged on rank 0", "ids_equal_cpu_oracle": True, "queries_checked_cpu": 0,
           "max_score_rel_err": 0.0, "regimes": {}}
    o = 0
    for name, Q, k, g_rows, g_scores in checks:
        n = Q.shape[0]
        want_r, want_s = rows[o:o + n, :k], scores[o:o + n, :k]
        o += n
        ids_ok = bool(np.array_equal(want_r, g_rows))
        rel = float(np.max(np.abs(g_scores.astype(np.float64) - want_s) / np.abs(want_s))) if want_s.size else 0.0
        out["regimes"][name] = {"queries": n, "k": k, "ids_equal": ids_ok, "max_score_rel_err": rel}
        out["ids_equal_cpu_oracle"] &= ids_ok
        out["queries_checked_cpu"] += n
        out["max_score_rel_err"] = max(out["max_score_rel_err"], rel)
    out["scores_within_1e-5"] = out["max_score_rel_err"] <= 1e-5
    out["seconds"] = round(time.perf_counter() - t0, 1)
    return out


class KnnLoop:
    """The serving loop of one index: two batches in flight, device-event timing, max over ranks."""

    def __init__(self, index, world, dev):
        self.index, self.eng, self.world, self.dev = index, index.engine, world, dev
        self.reset()

    def reset(self):
        self.stats = {"scan_ms": 0.0, "launches": 0, "fallback": 0, "certified": 0, "bytes": 0, "n": 0}
        self.index.merge_launches = 0

    def account(self):
        st = self.eng.last_stats
        s = self.stats
        s["scan_ms"] += st["scan_ms"]
        s["launches"] += st["launches"]
        s["fallback"] += st["n_fallback"]
        s["certified"] += st["n_certified"]
        s["bytes"] += st["bytes_streamed"]
        s["n"] += 1

    def barrier(self):
        import torch
        import torch.distributed as dist
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps, warmup, flush=None, idle_s=0.0):
        import torch
        import torch.distributed as dist
        if idle_s:                  # every arm starts from the same power state: a pause, then its own warm-up
            self.barrier()
            time.sleep(idle_s)
        for i in range(warmup):
            fn(i)
        if flush:
            flush()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.time()
        e0.record()
        for i in range(steps):
            fn(i)
        if flush:
            flush()          # the last batches in flight complete inside the timed region
        e1.record()
        self.barrier()
        t1 = time.time()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev, dtype=torch.float64)
        if self.world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), t0, t1

    def pipelined(self, pick, kx, capture=None, n_capture=N_CHECK):
        """(step, flush) closures of a loop that keeps two batches of pick(i) in flight.  capture: dict that receives
        the merged (rows, scores) of the first n_capture queries of the first batch-0 result the loop collects."""
        tickets = []

        def collect():
            t, i = tickets.pop(0)
            rows, scores = self.index.wait(t)
            self.account()
            self.last = (rows, scores)          # the index's work buffers: valid until its next search
            if capture is not None and "rows" not in capture and capture["want"](i):
                capture["rows"] = rows[:n_capture].clone()
                capture["scores"] = scores[:n_capture].clone()

        def step(i):
            tickets.append((self.index.search_dev_async(pick(i), kx), i))
            if len(tickets) == 2:
                collect()

        def flush():
            while tickets:
                collect()
        return step, flush


def run_ours(a):
    import torch
    import torch.distributed as dist
    import rassengine_b200 as rb
    from rassengine_b200.sharded import ShardedIndex, shard_bounds

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    if a.workload == "cfg4":
        import bench_hybrid
        return bench_hybrid.run_ours(a, world, rank, dev)

    sampler = ClockSampler(local) if rank == 0 else None
    lo, hi = shard_bounds(a.rows, world, rank)
    index = ShardedIndex(dim=DIM, capacity_rows=hi - lo, flags=rb.BF16_ONLY if a.bf16_only else 0)
    index.set_row_base(lo)
    fill_shard(index, lo, hi)
    eng = index.engine
    B, k = a.batch, a.k
    loop = KnnLoop(index, world, dev)
    stats = loop.stats

    gq = torch.Generator(device=dev).manual_seed(SEED_QUERIES)
    n_batches = 8 if B <= 1024 else 2
    q_dev = [torch.randn((B, DIM), generator=gq, device=dev) for _ in range(n_batches)]
    q_host = [q.cpu().pin_memory() for q in q_dev]
    n_chk = min(N_CHECK, B)

    # ---- parity spot-check outside the timed region: fast path ids == fp64 full scan ids on this shard ----
    nb = min(B, 256)          # every query of a 64-query batch; a 256-query sample (one pass of the pair kernel) above
    rows_f = torch.empty((nb, k), dtype=torch.int64, device=dev)
    sc_f = torch.empty((nb, k), dtype=torch.float32, device=dev)
    eng.search_knn_dev(q_dev[0].data_ptr(), nb, k, rows_f.data_ptr(), sc_f.data_ptr())
    eng.set_path(rb.PATH_EXACT)
    rows_x = torch.empty_like(rows_f)
    sc_x = torch.empty_like(sc_f)
    eng.search_knn_dev(q_dev[0].data_ptr(), nb, k, rows_x.data_ptr(), sc_x.data_ptr())
    eng.set_path(rb.PATH_AUTO)
    parity_fp64_ok = bool((rows_f == rows_x).all())

    # ---- device-resident arm ----
    # the serving loop keeps two batches in flight: batch i+1 is enqueued before batch i is collected, so the
    # exchange (all-gather + merge, on a side stream) and the host work of a batch hide behind the next scan
    cap_main = {"want": lambda i: i % n_batches == 0}
    step_dev, flush_dev = loop.pipelined(lambda i: q_dev[i % n_batches], k, capture=cap_main, n_capture=n_chk)
    loop.barrier()
    time.sleep(ARM_IDLE_S)          # (the fp64 parity scan above ran the GPU hot)
    for i in range(a.warmup):
        step_dev(i)
    flush_dev()
    loop.reset()
    cap_main.pop("rows", None)
    cap_main.pop("scores", None)
    ms_dev, t0, t1 = loop.timed(step_dev, a.steps, 0, flush=flush_dev)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"rows": loop.last[0].cpu().numpy(), "scores": loop.last[1].cpu().numpy()})
    stats = loop.stats
    scan_ms_avg = stats["scan_ms"] / max(1, stats["n"])
    bytes_per_step = stats["bytes"] / max(1, stats["n"])
    launches = stats["launches"] + index.merge_launches
    fallback = stats["fallback"]
    win_timed = (t0, t1)
    if "rows" not in cap_main:      # fewer timed steps than it takes to collect a batch-0 result
        r_, s_ = index.search_dev(q_dev[0], k)
        cap_main["rows"], cap_main["scores"] = r_[:n_chk].clone(), s_[:n_chk].clone()

    # ---- end-to-end arm: pinned host queries in, host results out, every step (same two-in-flight loop) ----
    e2e_tickets = []

    def step_e2e(i):
        e2e_tickets.append(index.search_async(q_host[i % n_batches], k))
        if len(e2e_tickets) == 2:
            index.wait_host(e2e_tickets.pop(0))

    def flush_e2e():
        while e2e_tickets:
            index.wait_host(e2e_tickets.pop(0))

    ms_e2e, _, _ = loop.timed(step_e2e, a.steps, a.warmup, flush=flush_e2e, idle_s=ARM_IDLE_S)

    # ---- sustained: the same device-resident loop for >= a.sustained_s seconds (the driver's 20 steps are a burst) ----
    sustained = None
    t_sus = None
    if a.sustained_s > 0:
        n_sus = max(a.steps, int(np.ceil(a.sustained_s * 1e3 / max(ms_dev / a.steps, 1e-3))))
        loop.reset()
        ms_s, ts0, ts1 = loop.timed(step_dev, n_sus, 0, flush=flush_dev)
        st = loop.stats
        scan_s = st["scan_ms"] / max(1, st["n"])
        sustained = {"qps": n_sus * B / (ms_s * 1e-3), "ms_per_step": ms_s / n_sus, "steps": n_sus,
                     "seconds": ms_s * 1e-3, "scan_ms": scan_s,
                     "scan_gbs": (st["bytes"] / max(1, st["n"])) / (scan_s * 1e-3) / 1e9 if scan_s and B <= 64 else None,
                     "scan_tflops": 2.0 * B * (hi - lo) * DIM / (scan_s * 1e-3) / 1e12 if scan_s and B > 64 else None,
                     "certificate_fallbacks": int(st["fallback"])}
        t_sus = (ts0, ts1)

    # ---- batch-1 latency regime (same corpus), for the record ----
    checks = [("batch%d_top%d" % (B, k), q_dev[0][:n_chk].cpu().numpy(), k, cap_main["rows"].cpu().numpy(),
               cap_main["scores"].cpu().numpy())]
    b1 = None
    extras = a.workload == "cfg2" and not a.no_extras
    if B != 1 and extras:
        q1 = [q[:1].contiguous() for q in q_dev]
        loop.reset()

        # one blocking call per query: the latency regime (the streaming scan fills every SM, so a second batch in
        # flight would only delay the exchange of the first)
        def step_b1(i):
            index.search_dev(q1[i % n_batches], k)
            loop.account()

        for i in range(a.warmup):
            step_b1(i)
        loop.reset()
        ms_b1, _, _ = loop.timed(step_b1, a.steps, 0)
        st = loop.stats
        b1_scan = st["scan_ms"] / max(1, st["n"])
        b1 = {"qps": a.steps / (ms_b1 * 1e-3), "ms_per_query": ms_b1 / a.steps,
              "scan_gbs": (st["bytes"] / max(1, st["n"])) / (b1_scan * 1e-3) / 1e9 if b1_scan else None}
        r1, s1 = index.search_dev(q1[1 % n_batches], k)
        checks.append(("batch1_top%d" % k, q1[1 % n_batches].cpu().numpy(), k, r1.cpu().numpy().copy(),
                       s1.cpu().numpy().copy()))
    # ---- large-batch regimes of the same corpus (tensor-core contraction), for the record ----
    batched = None
    if extras:
        batched = {}
        for name, Bx, kx, nsteps in (("batch1024_top10", 1024, 10, 10), ("batch8192_top100", 8192, 100, 3)):
            qx = torch.randn((Bx, DIM), generator=gq, device=dev)
            loop.reset()
            cap = {"want": lambda i: True}
            step_x, flush_x = loop.pipelined(lambda i, qx=qx: qx, kx, capture=cap)
            for i in range(3):
                step_x(i)
            flush_x()
            loop.reset()
            cap.pop("rows", None)
            cap.pop("scores", None)
            ms_x, _, _ = loop.timed(step_x, nsteps, 0, flush=flush_x)
            st = loop.stats
            scan_x = st["scan_ms"] / max(1, st["n"])
            flops = 2.0 * Bx * (hi - lo) * DIM
            batched[name] = {"qps": nsteps * Bx / (ms_x * 1e-3), "ms_per_batch": ms_x / nsteps, "k": kx,
                             "scan_kernel": scan_kernel_name(Bx), "scan_ms": scan_x,
                             "scan_tflops_per_gpu": flops / (scan_x * 1e-3) / 1e12 if scan_x else None,
                             "certificate_fallbacks": int(st["fallback"])}
            checks.append((name, qx[:N_CHECK].cpu().numpy(), kx, cap["rows"].cpu().numpy(), cap["scores"].cpu().numpy()))
            del qx
    t_gpu_end = time.time()

    # ---- CPU-oracle parity of the merged results, over the whole corpus (outside every timed region) ----
    parity_cpu = None
    if not a.no_cpu_parity:
        workers = max(1, min(6, (os.cpu_count() or 4) // max(1, world) - 1))
        parity_cpu = oracle_parity(eng, lo, hi, world, rank, checks, workers)

    # ---- CPU baseline on the same rows (rank 0 at N = 1 only) ----
    cpu_baseline = None
    if not a.no_cpu_baseline and world == 1:
        cores = blas_threads()
        sample = min(a.cpu_sample_rows or (2_000_000 if B <= 64 else 200_000), a.rows)
        Xs = eng.read_rows(0, sample)            # the same rows the GPU scanned
        Qs = q_dev[0].cpu().numpy()
        cpu_scan_time(Xs[: min(20000, sample)], Qs, k)
        t = cpu_scan_time(Xs, Qs, k, repeats=5)
        scale = a.rows / float(sample)
        cpu_baseline = {"value": B / (t * scale), "unit": "queries/s", "cores": cores, "kind": "port",
                        "sample": f"numpy fp32 sgemm + argpartition (oracle.knn.knn_fp32_baseline) over the "
                                  f"first {sample} of {a.rows} rows x {B} queries ({t:.2f} s, best of 5), scaled "
                                  f"x{scale:g}"}
        del Xs

    # ---- extras that need their own index: hybrid at N = 1, configuration 5 at N >= 2 ----
    index.close()
    del index, eng
    torch.cuda.empty_cache()
    hybrid = cfg5 = None
    if extras and world == 1:
        try:
            import bench_hybrid
            hybrid = bench_hybrid.run_extra(dev)
        except Exception as e:            # an extra must not take the headline line down with it
            hybrid = {"error": f"{type(e).__name__}: {e}"}
    if extras and world > 1:
        try:
            cfg5 = run_cfg5_extra(world, rank, dev, a)
        except Exception as e:
            cfg5 = {"error": f"{type(e).__name__}: {e}"}
    if sampler:
        sampler.stop()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # clocks: the driver-stepped region first; a 60 ms burst can fall between two samples, then the sustained loop
    clocks = None
    if sampler:
        lines = sampler.window(*win_timed)
        note = "timed region"
        if len(lines) < 3 and t_sus:
            lines = sampler.window(*t_sus)
            note = "sustained loop (the timed region is shorter than the sampling period)"
        if len(lines) < 3:
            lines = sampler.window(win_timed[0], t_gpu_end)
            note = "first timed step .. last GPU measurement"
        clocks = ClockSampler.summarise(lines, note)

    peak_hbm, peak_tf, peak_src = peaks()
    tensor_bound = B > 64
    if tensor_bound:
        flops_per_step = 2.0 * B * (hi - lo) * DIM
        achieved = flops_per_step / (scan_ms_avg * 1e-3) / 1e12 if scan_ms_avg else 0.0
        peak = peak_tf
    else:
        achieved = bytes_per_step / (scan_ms_avg * 1e-3) / 1e9 if scan_ms_avg else 0.0
        peak = peak_hbm
    if batched:
        for v in batched.values():
            v["frac_of_tensor_peak"] = v["scan_tflops_per_gpu"] / peak_tf if v["scan_tflops_per_gpu"] else None
    traffic = traffic_src = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp) and not tensor_bound:
        try:
            t = json.load(open(tp))
            traffic = t.get("dram_bytes_per_row", 0) * (hi - lo) or None
            traffic_src = ("profiles/traffic.json: dram__bytes_read+write of one `ncu --set full` capture of this "
                           "kernel, per row, x the rows of this run -- a cross-reference, not measured in this run")
        except Exception:
            traffic = None
    out = {
        "metric": METRIC, "value": a.steps * B / (ms_dev * 1e-3), "unit": "queries/s", "n_gpus": world,
        "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_dev / a.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "bf16 scan (fp32 accumulate) + fp64 rerank",
        "data": "synthetic",
        "config": make_config(a, world),
        "e2e": {"value": a.steps * B / (ms_e2e * 1e-3), "unit": "queries/s", "h2d_bytes_per_step": B * DIM * 4,
                "d2h_bytes_per_step": B * k * 12, "ms_per_step": ms_e2e / a.steps},
        "gpu_launches": int(launches),
        "roofline": ({"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s",
                      "frac": achieved / peak if peak else None, "traffic": None, "peak_source": peak_src,
                      "kernel": "scan_gemm_kernel", "algorithmic_flops_per_launch": 2.0 * B * (hi - lo) * DIM,
                      "kernel_ms": scan_ms_avg, "frac_of_nominal_2250TF": achieved / 2250.0} if tensor_bound else
                     {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                      "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
                      "peak_source": peak_src,
                      "kernel": "scan_umma_kernel" if B > 1 else "scan_stream_kernel",
                      "algorithmic_bytes_per_launch": bytes_per_step, "kernel_ms": scan_ms_avg,
                      "frac_of_nominal_8TBs": achieved / 8000.0}),
        "parity": dict({"fast_path_ids_equal_fp64_scan": parity_fp64_ok, "queries_checked": int(nb),
                        "certificate_fallbacks_in_timed_region": int(fallback)}, **(parity_cpu or {})),
        "sustained": sustained,
        "batch1": b1,
        "batched": batched,
        "hybrid": hybrid,
        "cfg5": cfg5,
        "clocks": clocks,
    }
    if cpu_baseline:
        out["cpu_baseline"] = cpu_baseline
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_cfg5_extra(world, rank, dev, a):
    """BASELINE.json configs[4] beside the headline: 100M x 1024 bf16 rows over the same ranks, batch 1024, top-10."""
    import torch
    import rassengine_b200 as rb
    from rassengine_b200.sharded import ShardedIndex, shard_bounds
    rows, B, k, nsteps = 100_000_000, 1024, 10, 5
    lo, hi = shard_bounds(rows, world, rank)
    need = (hi - lo) * (DIM * 2 + 24) + (6 << 30)
    free, _ = torch.cuda.mem_get_info()
    if need > free:
        return {"skipped": f"{(hi - lo)} bf16 rows per GPU need {need / 1e9:.0f} GB, {free / 1e9:.0f} GB free"}
    index = ShardedIndex(dim=DIM, capacity_rows=hi - lo, flags=rb.BF16_ONLY)
    index.set_row_base(lo)
    fill_shard(index, lo, hi)
    loop = KnnLoop(index, world, dev)
    gq = torch.Generator(device=dev).manual_seed(SEED_QUERIES + 5)
    qx = torch.randn((B, DIM), generator=gq, device=dev)
    cap = {"want": lambda i: True}
    step_x, flush_x = loop.pipelined(lambda i: qx, k, capture=cap)
    for i in range(3):
        step_x(i)
    flush_x()
    loop.reset()
    cap.pop("rows", None)
    cap.pop("scores", None)
    ms_x, _, _ = loop.timed(step_x, nsteps, 0, flush=flush_x)
    st = loop.stats
    scan_x = st["scan_ms"] / max(1, st["n"])
    _, peak_tf, _ = peaks()
    tf = 2.0 * B * (hi - lo) * DIM / (scan_x * 1e-3) / 1e12 if scan_x else None
    out = {"workload": f"cfg5: exact cosine top-{k}, {rows} x {DIM} bf16 corpus row-sharded x{world}, query batch {B}",
           "qps": nsteps * B / (ms_x * 1e-3), "ms_per_batch": ms_x / nsteps, "steps": nsteps,
           "scan_kernel": scan_kernel_name(B), "scan_ms": scan_x, "scan_tflops_per_gpu": tf,
           "frac_of_tensor_peak": tf / peak_tf if tf else None, "certificate_fallbacks": int(st["fallback"])}
    if not a.no_cpu_parity:
        workers = max(1, min(6, (os.cpu_count() or 4) // max(1, world) - 1))
        checks = [("cfg5_batch1024_top10", qx[:N_CHECK].cpu().numpy(), k, cap["rows"].cpu().numpy(),
                   cap["scores"].cpu().numpy())]
        out["parity"] = oracle_parity(index.engine, lo, hi, world, rank, checks, workers)
    index.close()
    return out


def main():
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
