"""Python handle over the C-ABI engine (include/rass_b200.h): numpy in / numpy out for the host-pointer calls,
raw device pointers (e.g. ``torch.Tensor.data_ptr()``) for the ``*_dev`` calls."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi as capi
from ._capi import RassError, RassStats


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _pack_terms(qterms, B: int):
    """qterms: B term-id lists, or an already packed (indptr int32 [B+1], terms int32 [nnz]) pair."""
    if isinstance(qterms, tuple) and len(qterms) == 2 and isinstance(qterms[0], np.ndarray):
        indptr = np.ascontiguousarray(qterms[0], dtype=np.int32)
        terms = np.ascontiguousarray(qterms[1], dtype=np.int32)
        if indptr.size != B + 1:
            raise ValueError("packed qterms: indptr must have B + 1 entries")
        return indptr, (terms if terms.size else np.zeros(1, dtype=np.int32))
    if len(qterms) != B:
        raise ValueError("qterms must hold one list per query")
    indptr = np.zeros(B + 1, dtype=np.int32)
    indptr[1:] = np.cumsum([len(t) for t in qterms])
    terms = np.ascontiguousarray(np.concatenate([np.asarray(t, dtype=np.int32) for t in qterms])
                                 if indptr[-1] else np.zeros(1, dtype=np.int32), dtype=np.int32)
    return indptr, terms


class Engine:
    """One device-resident shard of the vector store + its postings (rass_create ... rass_destroy)."""

    def __init__(self, dim: int = 1024, metric: int = capi.METRIC_COSINE, device: int = 0, capacity_rows: int = 0,
                 flags: int = 0, devices=None):
        """devices: a list of CUDA ordinals -> ONE handle whose rows are spread over those GPUs (rass_create_sharded;
        devices[0] is the coordinator).  Every method below works unchanged on such a handle."""
        self._lib = capi.lib()
        self._h = C.c_void_p()
        if devices is not None and len(devices) > 1:
            ids = (C.c_int * len(devices))(*[int(d) for d in devices])
            rc = self._lib.rass_create_sharded(dim, metric, len(devices), ids, capacity_rows, flags, C.byref(self._h))
            device = int(devices[0])
        else:
            if devices:
                device = int(devices[0])
            rc = self._lib.rass_create(dim, metric, device, capacity_rows, flags, C.byref(self._h))
        if rc:
            msg = self._lib.rass_last_error(None).decode()
            self._h = None
            raise RassError(rc, msg)
        self.devices = [int(d) for d in devices] if devices else [device]
        self.dim, self.metric, self.device, self.flags = dim, metric, device, flags or capi.KEEP_FP32
        self.last_stats: dict = {}

    # -- plumbing ---------------------------------------------------------------------------------------
    def _check(self, rc: int):
        if rc:
            raise RassError(rc, self._lib.rass_last_error(self._h).decode())

    def close(self):
        if getattr(self, "_h", None):
            self._lib.rass_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def set_path(self, path: int):
        self._check(self._lib.rass_set_option(self._h, capi.OPT_PATH, path))

    def set_stream(self, cuda_stream: int):
        self._check(self._lib.rass_set_option(self._h, capi.OPT_STREAM, cuda_stream))

    def set_knn_prefilter(self, on: bool):
        """When on, search_knn returns the exact top-k of the rows passing set_row_filter (pre-filter)."""
        self._check(self._lib.rass_set_option(self._h, capi.OPT_KNN_PREFILTER, 1 if on else 0))

    def set_hybrid_ordered(self, on: bool):
        """Force the ordered (one barrier per term) text kernel for hybrid calls; results are bit-identical either way."""
        self._check(self._lib.rass_set_option(self._h, capi.OPT_HYBRID_ORDERED, 1 if on else 0))

    def set_hybrid_maxscore(self, on: bool):
        """MaxScore-style essential / non-essential term split in the order-free text kernel (identical results)."""
        self._check(self._lib.rass_set_option(self._h, capi.OPT_HYBRID_MAXSCORE, 1 if on else 0))

    def set_row_base(self, base: int):
        self._check(self._lib.rass_set_row_base(self._h, base))

    def sync(self):
        self._check(self._lib.rass_sync(self._h))

    def save(self, path: str):
        """Snapshot of the stored rows + tombstones (rass_save)."""
        self._check(self._lib.rass_save(self._h, path.encode()))

    def load(self, path: str):
        """Restore into an empty engine of the same dim / metric / corpus type (rass_load)."""
        self._check(self._lib.rass_load(self._h, path.encode()))

    # -- store ------------------------------------------------------------------------------------------
    def store_info(self) -> dict:
        """{"capacity_rows", "grows_in_place"}: see rass_store_info."""
        cap, vm = C.c_int64(), C.c_int()
        self._check(self._lib.rass_store_info(self._h, C.byref(cap), C.byref(vm)))
        return {"capacity_rows": cap.value, "grows_in_place": bool(vm.value)}

    def append(self, rows: np.ndarray) -> int:
        rows = np.ascontiguousarray(rows, dtype=np.float32).reshape(-1, self.dim)
        first = C.c_int64(-1)
        self._check(self._lib.rass_append(self._h, _ptr(rows), rows.shape[0], C.byref(first)))
        return first.value

    def append_dev(self, dev_ptr: int, n: int) -> int:
        first = C.c_int64(-1)
        self._check(self._lib.rass_append_dev(self._h, C.c_void_p(dev_ptr), n, C.byref(first)))
        return first.value

    def overwrite(self, row: int, v: np.ndarray):
        v = np.ascontiguousarray(v, dtype=np.float32).reshape(self.dim)
        self._check(self._lib.rass_overwrite(self._h, row, _ptr(v)))

    def tombstone(self, row: int):
        self._check(self._lib.rass_tombstone(self._h, row))

    def count(self) -> int:
        n = C.c_int64()
        self._check(self._lib.rass_count(self._h, C.byref(n)))
        return n.value

    def rows(self) -> int:
        n = C.c_int64()
        self._check(self._lib.rass_rows(self._h, C.byref(n)))
        return n.value

    def read_rows(self, first: int, n: int) -> np.ndarray:
        out = np.empty((n, self.dim), dtype=np.float32)
        self._check(self._lib.rass_read_rows(self._h, first, n, _ptr(out)))
        return out

    def read_rows_into(self, first: int, n: int, out_ptr: int):
        """Same into caller memory ([n, dim] fp32, e.g. a pinned buffer: the copy then runs at PCIe rate)."""
        self._check(self._lib.rass_read_rows(self._h, first, n, C.c_void_p(out_ptr)))

    def read_rows_list(self, rows) -> np.ndarray:
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        out = np.empty((rows.size, self.dim), dtype=np.float32)
        self._check(self._lib.rass_read_rows_list(self._h, _ptr(rows), rows.size, _ptr(out)))
        return out

    def set_row_filter_rows(self, rows, total_rows: int):
        """The bool.filter as the list of rows that pass; rows >= total_rows fail."""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        self._check(self._lib.rass_set_row_filter_rows(self._h, _ptr(rows), rows.size, total_rows))

    # -- search -----------------------------------------------------------------------------------------
    def search_knn(self, q: np.ndarray, k: int, want_keys: bool = False):
        """q: [B, dim] fp32 (host).  Returns rows int64 [B, k] (-1 = no hit), scores fp32 [B, k]
        (and keys fp64 [B, k] = cos or squared distance when want_keys)."""
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
        B = q.shape[0]
        rows = np.empty((B, k), dtype=np.int64)
        scores = np.empty((B, k), dtype=np.float32)
        keys = np.empty((B, k), dtype=np.float64) if want_keys else None
        st = RassStats()
        self._check(self._lib.rass_search_knn(self._h, _ptr(q), B, k, _ptr(rows), _ptr(scores),
                                              _ptr(keys) if want_keys else None, C.byref(st)))
        self.last_stats = st.as_dict()
        return (rows, scores, keys) if want_keys else (rows, scores)

    def search_knn_dev(self, q_ptr: int, B: int, k: int, rows_ptr: int, scores_ptr: int, keys_ptr: int = 0) -> dict:
        st = RassStats()
        self._check(self._lib.rass_search_knn_dev(self._h, C.c_void_p(q_ptr), B, k, C.c_void_p(rows_ptr),
                                                  C.c_void_p(scores_ptr), C.c_void_p(keys_ptr) if keys_ptr else None,
                                                  C.byref(st)))
        self.last_stats = st.as_dict()
        return self.last_stats

    def search_knn_dev_async(self, q_ptr: int, B: int, k: int, rows_ptr: int, scores_ptr: int, keys_ptr: int = 0,
                             slot: int = 0, flag_ptr: int = 0):
        """Enqueue only (no host synchronisation); pair with search_knn_dev_wait(slot)."""
        self._check(self._lib.rass_search_knn_dev_async(self._h, C.c_void_p(q_ptr), B, k, C.c_void_p(rows_ptr),
                                                        C.c_void_p(scores_ptr),
                                                        C.c_void_p(keys_ptr) if keys_ptr else None, slot,
                                                        C.c_void_p(flag_ptr) if flag_ptr else None))

    def set_async_overlap(self, on: bool = True):
        """Each async slot on its own stream and workspace (RASS_OPT_ASYNC_OVERLAP): the fixed costs of batch i run
        under the corpus pass of batch i+1.  Order readers of the outputs with async_join / search_knn_dev_wait."""
        self._check(self._lib.rass_set_option(self._h, capi.OPT_ASYNC_OVERLAP, 1 if on else 0))

    def set_scan_reserve_sms(self, n: int):
        """SMs the 64-query corpus pass leaves to the kernels beside it (RASS_OPT_SCAN_RESERVE_SMS)."""
        self._check(self._lib.rass_set_option(self._h, capi.OPT_SCAN_RESERVE_SMS, int(n)))

    def async_join(self, slot: int, cuda_stream: int):
        """Make `cuda_stream` wait (on the device) for the search enqueued in `slot`."""
        self._check(self._lib.rass_async_join(self._h, slot, C.c_void_p(cuda_stream) if cuda_stream else None))

    def search_knn_dev_wait(self, slot: int = 0) -> tuple[bool, dict]:
        """(final, stats): final is False when some query failed its certificate and the batch must be repeated with
        the blocking call."""
        st = RassStats()
        rc = self._lib.rass_search_knn_dev_wait(self._h, slot, C.byref(st))
        if rc not in (0, capi.RASS_E_AGAIN):
            self._check(rc)
        self.last_stats = st.as_dict()
        return rc == 0, self.last_stats

    def merge_topk_dev(self, keys_ptr: int, rows_ptr: int, G: int, B: int, k: int, out_rows_ptr: int,
                       out_scores_ptr: int, out_keys_ptr: int = 0, shard_stride: int = 0):
        """Enqueued on the engine stream; call sync() (or synchronise that stream) before reading the outputs."""
        self._check(self._lib.rass_merge_topk_dev(self._h, C.c_void_p(keys_ptr), C.c_void_p(rows_ptr), shard_stride,
                                                  G, B, k,
                                                  C.c_void_p(out_rows_ptr), C.c_void_p(out_scores_ptr),
                                                  C.c_void_p(out_keys_ptr) if out_keys_ptr else None))

    def merge_scores_dev(self, scores_ptr: int, rows_ptr: int, G: int, B: int, k: int, out_rows_ptr: int,
                         out_scores_ptr: int, out_keys_ptr: int = 0, shard_stride: int = 0):
        """merge_topk_dev for fused hybrid lists: raw scores, larger is better whatever the vector metric."""
        self._check(self._lib.rass_merge_scores_dev(self._h, C.c_void_p(scores_ptr), C.c_void_p(rows_ptr),
                                                    shard_stride, G, B, k, C.c_void_p(out_rows_ptr),
                                                    C.c_void_p(out_scores_ptr),
                                                    C.c_void_p(out_keys_ptr) if out_keys_ptr else None))

    # -- text -------------------------------------------------------------------------------------------
    def bm25_build(self, indptr, doc, tf, doclen, global_doc_count: int = 0, global_sum_ttf: int = 0,
                   global_df=None):
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        doc = np.ascontiguousarray(doc, dtype=np.int32)
        tf = np.ascontiguousarray(tf, dtype=np.uint16)
        doclen = np.ascontiguousarray(doclen, dtype=np.uint32)
        gdf = None if global_df is None else np.ascontiguousarray(global_df, dtype=np.int64)
        self._check(self._lib.rass_bm25_build(self._h, _ptr(indptr), _ptr(doc), _ptr(tf), _ptr(doclen),
                                              indptr.size - 1, doclen.size, global_doc_count, global_sum_ttf,
                                              _ptr(gdf) if gdf is not None else None))

    def bm25_build_fields(self, indptr, doc, tf, term_field, doclen):
        """Several analysed fields in one CSR: term_field int32 [V], doclen uint32 [F, N]."""
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        doc = np.ascontiguousarray(doc, dtype=np.int32)
        tf = np.ascontiguousarray(tf, dtype=np.uint16)
        term_field = np.ascontiguousarray(term_field, dtype=np.int32)
        doclen = np.ascontiguousarray(doclen, dtype=np.uint32)
        if doclen.ndim != 2 or term_field.size != indptr.size - 1:
            raise ValueError("doclen must be [F, N] and term_field [V]")
        self._check(self._lib.rass_bm25_build_fields(self._h, _ptr(indptr), _ptr(doc), _ptr(tf), _ptr(term_field),
                                                     _ptr(doclen), indptr.size - 1, doclen.shape[1], doclen.shape[0]))

    def text_add_rows(self, field: int, rows, tok_indptr, tok_terms):
        """Device-side ingest of one field of a bulk of NEW rows (rass_text_add_rows): rows int64 [n] ascending,
        tok_indptr int64 [n + 1], tok_terms int32 term ids local to the field, token order, repeats included.
        Searchable after text_commit."""
        rows = np.ascontiguousarray(rows, dtype=np.int64)
        tok_indptr = np.ascontiguousarray(tok_indptr, dtype=np.int64)
        tok_terms = np.ascontiguousarray(tok_terms, dtype=np.int32)
        if tok_indptr.size != rows.size + 1:
            raise ValueError("tok_indptr must have len(rows) + 1 entries")
        self._check(self._lib.rass_text_add_rows(self._h, int(field), _ptr(rows), rows.size, _ptr(tok_indptr),
                                                 _ptr(tok_terms) if tok_terms.size else None))

    def text_add_rows_dev(self, field: int, rows_ptr: int, n_rows: int, tok_indptr_ptr: int, tok_terms_ptr: int):
        """The same with device pointers (int64 rows, int64 offsets, int32 term ids)."""
        self._check(self._lib.rass_text_add_rows_dev(self._h, int(field), C.c_void_p(rows_ptr), int(n_rows),
                                                     C.c_void_p(tok_indptr_ptr), C.c_void_p(tok_terms_ptr)))

    def text_omit_norms(self, field: int, omit: bool = True):
        """The field's documents all count as length 1 (a `keyword` field): rass_text_omit_norms."""
        self._check(self._lib.rass_text_omit_norms(self._h, int(field), 1 if omit else 0))

    def text_commit(self, field_vocab, n_rows: int):
        """Fold the pending segments into the searchable CSR (rass_text_commit): field_vocab = terms per field now."""
        fv = np.ascontiguousarray(field_vocab, dtype=np.int64)
        self._check(self._lib.rass_text_commit(self._h, _ptr(fv), fv.size, int(n_rows)))

    def text_size(self) -> dict:
        V, N, nnz, F = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int()
        self._check(self._lib.rass_text_size(self._h, C.byref(V), C.byref(N), C.byref(nnz), C.byref(F)))
        return {"V": V.value, "N": N.value, "nnz": nnz.value, "F": F.value}

    def text_stats(self):
        """(indptr int64 [V + 1], doc_count int64 [F]) of the committed index -- host copies, no device traffic."""
        sz = self.text_size()
        indptr = np.zeros(sz["V"] + 1, dtype=np.int64)
        dc = np.zeros(max(sz["F"], 1), dtype=np.int64)
        self._check(self._lib.rass_text_stats(self._h, _ptr(indptr), _ptr(dc), None))
        return indptr, dc[:sz["F"]]

    def text_export(self, postings: bool = True):
        """The committed index read back: (indptr int64 [V+1], doc int32 [nnz], tf uint16 [nnz], doclen uint32 [F, N],
        norm uint8 [F, N]); doc / tf are None with postings=False."""
        sz = self.text_size()
        indptr = np.zeros(sz["V"] + 1, dtype=np.int64)
        doc = np.zeros(sz["nnz"], dtype=np.int32) if postings else None
        tf = np.zeros(sz["nnz"], dtype=np.uint16) if postings else None
        doclen = np.zeros((sz["F"], sz["N"]), dtype=np.uint32)
        norm = np.zeros((sz["F"], sz["N"]), dtype=np.uint8)
        self._check(self._lib.rass_text_export(self._h, _ptr(indptr), _ptr(doc) if postings and doc.size else None,
                                               _ptr(tf) if postings and tf.size else None,
                                               _ptr(doclen) if doclen.size else None,
                                               _ptr(norm) if norm.size else None))
        return indptr, doc, tf, doclen, norm

    def set_row_filter(self, mask):
        """mask: uint8/bool [rows] (1 = passes the query's bool.filter) or None to clear."""
        if mask is None:
            self._check(self._lib.rass_set_row_filter(self._h, None, 0))
            return
        m = np.ascontiguousarray(mask, dtype=np.uint8)
        self._check(self._lib.rass_set_row_filter(self._h, _ptr(m), m.size))

    def set_vocab(self, terms: list[str]):
        """The text field's term dictionary in term-id order (needed by fuzzy_expand)."""
        enc = [t.encode("utf-8", "replace") for t in terms]
        off = np.zeros(len(enc) + 1, dtype=np.int64)
        if enc:
            off[1:] = np.cumsum([len(e) for e in enc])
        self._check(self._lib.rass_text_set_vocab(self._h, b"".join(enc), _ptr(off), len(enc)))
        self._vocab_size = len(enc)

    def set_vocab_raw(self, blob: bytes, offsets):
        """set_vocab from prepared arrays: the terms' utf-8 bytes back to back, int64 byte offsets [V + 1]."""
        off = np.ascontiguousarray(offsets, dtype=np.int64)
        self._check(self._lib.rass_text_set_vocab(self._h, blob, _ptr(off), off.size - 1))
        self._vocab_size = off.size - 1

    def fuzzy_expand(self, token: str, max_edits: int, term_lo: int = 0, term_hi: int = -1):
        """Dictionary terms of [term_lo, term_hi) within max_edits (optimal string alignment) of the token:
        (term ids, edits), unordered."""
        n_cap = max(getattr(self, "_vocab_size", 0), 1)
        terms = np.empty(n_cap, dtype=np.int32)
        edits = np.empty(n_cap, dtype=np.int32)
        n = C.c_int64(0)
        tok = token.encode("utf-8", "replace")
        self._check(self._lib.rass_fuzzy_expand(self._h, tok, len(tok), max_edits, term_lo, term_hi, n_cap,
                                                _ptr(terms), _ptr(edits), C.byref(n)))
        return terms[: n.value].copy(), edits[: n.value].copy()

    def search_hybrid(self, q, qterms, w_text: float, w_knn: float, k: int, qweights=None, qflags=None):
        """q: [B, dim] fp32 or None (text only); qterms: list of B term-id lists or None (vector only); qweights:
        optional list of B float32 lists, the weight of every term occurrence (replaces w_text * idf); qflags:
        optional list of B uint8 lists (bit 0 = last term of its field group, bit 1 = last term of its clause)."""
        packed = isinstance(qterms, tuple)
        if q is not None:
            q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
            B = q.shape[0]
        else:
            B = qterms[0].size - 1 if packed else len(qterms)
        indptr = terms = None
        if qterms is not None:
            indptr, terms = _pack_terms(qterms, B)
        rows = np.empty((B, k), dtype=np.int64)
        scores = np.empty((B, k), dtype=np.float32)
        st = RassStats()
        if qweights is not None and qterms is not None:
            w = np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.float32) for x in qweights])
                                     if indptr[-1] else np.zeros(1, dtype=np.float32), dtype=np.float32)
            if w.size != max(int(indptr[-1]), 1):
                raise ValueError("qweights must hold one weight per query term")
            fl = None
            if qflags is not None:
                fl = np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.uint8) for x in qflags])
                                          if indptr[-1] else np.zeros(1, dtype=np.uint8), dtype=np.uint8)
                if fl.size != w.size:
                    raise ValueError("qflags must hold one byte per query term")
            self._check(self._lib.rass_search_hybrid_weighted(self._h, _ptr(q) if q is not None else None, B,
                                                              _ptr(indptr), _ptr(terms), _ptr(w),
                                                              _ptr(fl) if fl is not None else None, w_knn, k,
                                                              _ptr(rows), _ptr(scores), C.byref(st)))
            self.last_stats = st.as_dict()
            return rows, scores
        self._check(self._lib.rass_search_hybrid(self._h, _ptr(q) if q is not None else None, B,
                                                 _ptr(indptr) if indptr is not None else None,
                                                 _ptr(terms) if terms is not None else None,
                                                 w_text, w_knn, k, _ptr(rows), _ptr(scores), C.byref(st)))
        self.last_stats = st.as_dict()
        return rows, scores

    @staticmethod
    def _pack_rows(row_lists):
        """B lists of passing rows -> (indptr int64 [B + 1], rows int64 [total])."""
        indptr = np.zeros(len(row_lists) + 1, dtype=np.int64)
        indptr[1:] = np.cumsum([len(r) for r in row_lists])
        rows = np.ascontiguousarray(np.concatenate([np.asarray(r, dtype=np.int64).reshape(-1) for r in row_lists])
                                    if indptr[-1] else np.zeros(1, dtype=np.int64), dtype=np.int64)
        return indptr, rows

    def search_knn_filtered(self, q: np.ndarray, k: int, row_lists, want_keys: bool = False):
        """Exact top-k among each query's OWN list of passing rows (per-query bool.filter, one call for the batch)."""
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
        B = q.shape[0]
        if len(row_lists) != B:
            raise ValueError("row_lists must hold one list per query")
        fip, frows = self._pack_rows(row_lists)
        rows = np.empty((B, k), dtype=np.int64)
        scores = np.empty((B, k), dtype=np.float32)
        keys = np.empty((B, k), dtype=np.float64) if want_keys else None
        self._check(self._lib.rass_search_knn_filtered(self._h, _ptr(q), B, k, _ptr(fip), _ptr(frows), _ptr(rows),
                                                       _ptr(scores), _ptr(keys) if want_keys else None))
        return (rows, scores, keys) if want_keys else (rows, scores)

    def search_hybrid_filtered(self, q, qterms, w_text: float, w_knn: float, k: int, row_lists, knn_pre: bool = False,
                               qweights=None, qflags=None):
        """search_hybrid with a DIFFERENT bool.filter per query, given as each query's list of passing rows; the knn
        clause is the k nearest of the whole corpus (one shared pass) unless knn_pre (k nearest among the list)."""
        if q is not None:
            q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
            B = q.shape[0]
        else:
            B = len(row_lists)
        if len(row_lists) != B:
            raise ValueError("row_lists must hold one list per query")
        fip, frows = self._pack_rows(row_lists)
        indptr = terms = w = fl = None
        if qterms is not None:
            indptr, terms = _pack_terms(qterms, B)
            cat = lambda xs, dt: np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=dt) for x in xs])
                                                      if indptr[-1] else np.zeros(1, dtype=dt), dtype=dt)
            w = cat(qweights, np.float32) if qweights is not None else None
            fl = cat(qflags, np.uint8) if qflags is not None else None
        rows = np.empty((B, k), dtype=np.int64)
        scores = np.empty((B, k), dtype=np.float32)
        st = RassStats()
        self._check(self._lib.rass_search_hybrid_filtered(
            self._h, _ptr(q) if q is not None else None, B, _ptr(indptr) if indptr is not None else None,
            _ptr(terms) if terms is not None else None, _ptr(w) if w is not None else None,
            _ptr(fl) if fl is not None else None, w_text, w_knn, k, _ptr(fip), _ptr(frows), 1 if knn_pre else 0,
            _ptr(rows), _ptr(scores), C.byref(st)))
        self.last_stats = st.as_dict()
        return rows, scores

    def fuse_hybrid(self, qterms, w_text: float, knn_rows, knn_scores, w_knn: float, k: int, qweights=None,
                    qflags=None):
        """Text clauses + bool.filter of this request fused with a knn list obtained earlier (host arrays [B, k], or
        None for text only).  Returns (rows, scores) like search_hybrid."""
        B = len(qterms) if qterms is not None else np.asarray(knn_rows).shape[0]
        indptr = terms = w = fl = None
        if qterms is not None:
            indptr = np.zeros(B + 1, dtype=np.int32)
            indptr[1:] = np.cumsum([len(t) for t in qterms])
            cat = lambda xs, dt: np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=dt) for x in xs])
                                                      if indptr[-1] else np.zeros(1, dtype=dt), dtype=dt)
            terms = cat(qterms, np.int32)
            w = cat(qweights, np.float32) if qweights is not None else None
            fl = cat(qflags, np.uint8) if qflags is not None else None
        kr = ks = None
        if knn_rows is not None:
            kr = np.ascontiguousarray(knn_rows, dtype=np.int64).reshape(B, k)
            ks = np.ascontiguousarray(knn_scores, dtype=np.float32).reshape(B, k)
        rows = np.empty((B, k), dtype=np.int64)
        scores = np.empty((B, k), dtype=np.float32)
        self._check(self._lib.rass_fuse_hybrid(
            self._h, B, _ptr(indptr) if indptr is not None else None, _ptr(terms) if terms is not None else None,
            _ptr(w) if w is not None else None, _ptr(fl) if fl is not None else None, w_text,
            _ptr(kr) if kr is not None else None, _ptr(ks) if ks is not None else None, w_knn, k, _ptr(rows),
            _ptr(scores)))
        return rows, scores

    def fuse_hybrid_dev(self, B: int, qterms, w_text: float, knn_rows_ptr: int, knn_scores_ptr: int, w_knn: float, k: int,
                        out_rows_ptr: int, out_scores_ptr: int, out_keys_ptr: int = 0, qweights=None, qflags=None):
        """Text clauses fused with an external (global) knn list; this shard's top-k stays on the device."""
        indptr = terms = w = fl = None
        if qterms is not None:
            indptr, terms = _pack_terms(qterms, B)
            cat = lambda xs, dt: np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=dt) for x in xs])
                                                      if indptr[-1] else np.zeros(1, dtype=dt), dtype=dt)
            w = cat(qweights, np.float32) if qweights is not None else None
            fl = cat(qflags, np.uint8) if qflags is not None else None
        vp = lambda p: C.c_void_p(p) if p else None
        self._check(self._lib.rass_fuse_hybrid_dev(
            self._h, B, _ptr(indptr) if indptr is not None else None, _ptr(terms) if terms is not None else None,
            _ptr(w) if w is not None else None, _ptr(fl) if fl is not None else None, w_text, vp(knn_rows_ptr),
            vp(knn_scores_ptr), w_knn, k, vp(out_rows_ptr), vp(out_scores_ptr), vp(out_keys_ptr)))
        self.last_hybrid_stats = self.stats()

    def stats(self) -> dict:
        """rass_last_stats: of the last blocking search / hybrid / fuse call."""
        st = RassStats()
        self._check(self._lib.rass_last_stats(self._h, C.byref(st)))
        return st.as_dict()

    def debug_umma_scores(self, q: np.ndarray) -> np.ndarray:
        """Raw tensor-core dot products bf16(q_hat) . bf16(x) of up to 64 queries against every row: [rows, 64]."""
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
        out = np.zeros((self.rows(), 64), dtype=np.float32)
        self._check(self._lib.rass_debug_umma_scores(self._h, _ptr(q), q.shape[0], _ptr(out)))
        return out

    def debug_umma8_scores(self, q: np.ndarray):
        """The int8 pass's exact int32 accumulators of up to 64 queries against every row, [rows, 128] (column j < 64:
        x8 . q1 of query j, 64 + j: x8 . q2), with the int8 operands it read: x8 [rows, dim_pad], q8 [128, dim_pad]."""
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
        dim_pad = (self.dim + 255) // 256 * 256
        acc = np.zeros((self.rows(), 128), dtype=np.int32)
        x8 = np.zeros((self.rows(), dim_pad), dtype=np.int8)
        q8 = np.zeros((128, dim_pad), dtype=np.int8)
        self._check(self._lib.rass_debug_umma8_scores(self._h, _ptr(q), q.shape[0], _ptr(acc), _ptr(x8), _ptr(q8)))
        return acc, x8, q8

    def debug_gemm_scores(self, q: np.ndarray) -> np.ndarray:
        """Same through the CTA-pair (cta_group::2) kernel: up to 256 queries, [rows, 256]."""
        q = np.ascontiguousarray(q, dtype=np.float32).reshape(-1, self.dim)
        out = np.zeros((self.rows(), 256), dtype=np.float32)
        self._check(self._lib.rass_debug_gemm_scores(self._h, _ptr(q), q.shape[0], _ptr(out)))
        return out
