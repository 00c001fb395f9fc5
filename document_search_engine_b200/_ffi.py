"""ctypes binding of ``libbm25f.so`` (C ABI declared in ``include/bm25f.h``).

The library is built in-tree by ``__graft_entry__.build()`` (or ``make -C
document_search_engine_b200/csrc``).  There is no CPU fallback: if the library is
missing or no B200 is visible, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Optional, Sequence, Tuple

import numpy as np

ABI_VERSION = 3
MAX_K = 1024
MAX_LEAVES_PER_QUERY = 256
TERM_UNKNOWN = 0xFFFFFFFF
TERM_EVERY_BASE = 0xFFFFFF00       # + field index: Every(field)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libbm25f.so")

#: every symbol ``include/bm25f.h`` declares
EXPORTS = (
    "bm25f_abi_version", "bm25f_last_error", "bm25f_create", "bm25f_destroy", "bm25f_set_weighting",
    "bm25f_prepare", "bm25f_prepare_arena", "bm25f_execute", "bm25f_fetch", "bm25f_plan_device_results", "bm25f_synchronize",
    "bm25f_set_stream", "bm25f_plan_destroy", "bm25f_search_batch", "bm25f_merge_keys", "bm25f_decode_keys", "bm25f_get_stats",
    "bm25f_reset_stats", "bm25f_submit", "bm25f_collect", "bm25f_set_final_date", "bm25f_fetch_final",
    "bm25f_plan_device_final", "bm25f_merge_final_lists", "bm25f_plan_gather_span", "bm25f_merge_gathered", "bm25f_put_lists",
    "bm25f_put_positions", "bm25f_phrase_lists",
)


class EngineError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__("libbm25f error %d: %s" % (code, message))
        self.code = code


class IndexDesc(C.Structure):
    _fields_ = [("abi_version", C.c_uint32), ("n_fields", C.c_uint32), ("n_docs_all", C.c_uint64),
                ("n_terms", C.c_uint64), ("n_postings", C.c_uint64), ("doc_base", C.c_uint64),
                ("term_offsets", C.c_void_p), ("term_field", C.c_void_p), ("docids", C.c_void_p),
                ("tfs", C.c_void_p), ("len_bytes", C.c_void_p), ("deleted", C.c_void_p)]


class Options(C.Structure):
    _fields_ = [("tile_docs", C.c_uint32), ("threads", C.c_uint32), ("split_postings", C.c_uint32),
                ("variant", C.c_uint32), ("chunk_postings", C.c_uint32), ("stages", C.c_uint32),
                ("subtile_docs", C.c_uint32), ("warp_split", C.c_uint32), ("stream_warps", C.c_uint32),
                ("prefetch_postings", C.c_uint32), ("cta_warps", C.c_uint32), ("cta_prefetch", C.c_uint32),
                ("cta_split", C.c_uint32), ("cta_slice_docs", C.c_uint32), ("isect_ratio", C.c_uint32),
                ("isect_split", C.c_uint32), ("isect_or_limit", C.c_uint32), ("serial_streams", C.c_uint32),
                ("host_plan", C.c_uint32), ("compact_store", C.c_uint32),
                ("filter_postings", C.c_uint32)]


#: engine options a caller may pass (``bm25f_options`` field names; 0 = library default)
OPTION_NAMES = tuple(n for n, _ in Options._fields_)


class QueryBatchDesc(C.Structure):
    _fields_ = [("n_queries", C.c_uint32), ("n_leaves", C.c_uint32), ("query_leaf_offsets", C.c_void_p),
                ("query_n_groups", C.c_void_p), ("leaf_term", C.c_void_p), ("leaf_weight", C.c_void_p),
                ("leaf_group", C.c_void_p), ("after_keys", C.c_void_p), ("after_lo", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("postings_touched", C.c_uint64), ("n_items", C.c_uint64), ("n_launches", C.c_uint64),
                ("n_executes", C.c_uint64), ("ms_bounds", C.c_float), ("ms_score", C.c_float), ("ms_merge", C.c_float), ("ms_total", C.c_float),
                ("tile_docs", C.c_uint32), ("threads", C.c_uint32), ("ctas_per_sm", C.c_uint32),
                ("packed_payload", C.c_uint32), ("device_bytes", C.c_uint64), ("postings_stream", C.c_uint64),
                ("postings_team", C.c_uint64), ("postings_cta", C.c_uint64), ("postings_lookup", C.c_uint64),
                ("postings_topk", C.c_uint64), ("ms_stream", C.c_float), ("reserved1", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_lib = None


def load_library(path: Optional[str] = None):
    """Load ``libbm25f.so`` and declare the prototypes.  Raises if it is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    path = path or os.environ.get("BM25F_LIB", LIB_PATH)
    if not os.path.exists(path):
        raise RuntimeError("libbm25f.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "or `make -C document_search_engine_b200/csrc`. There is no CPU fallback." % path)
    lib = C.CDLL(path)
    vp, i32, u32 = C.c_void_p, C.c_int, C.c_uint32
    lib.bm25f_abi_version.restype = i32
    lib.bm25f_last_error.restype = C.c_char_p
    lib.bm25f_create.argtypes = [C.POINTER(IndexDesc), i32, C.POINTER(Options), C.POINTER(vp)]
    lib.bm25f_destroy.argtypes = [vp]
    lib.bm25f_destroy.restype = None
    lib.bm25f_set_weighting.argtypes = [vp, vp]
    lib.bm25f_prepare.argtypes = [vp, C.POINTER(QueryBatchDesc), i32, C.POINTER(vp)]
    lib.bm25f_prepare_arena.argtypes = [vp, C.POINTER(QueryBatchDesc), i32, C.POINTER(vp)]
    lib.bm25f_execute.argtypes = [vp, vp]
    lib.bm25f_fetch.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.bm25f_plan_device_results.argtypes = [vp, C.POINTER(vp), C.POINTER(vp)]
    lib.bm25f_synchronize.argtypes = [vp]
    lib.bm25f_set_stream.argtypes = [vp, vp, i32]
    lib.bm25f_put_lists.argtypes = [vp, u32, vp, vp, C.POINTER(u32)]
    lib.bm25f_put_positions.argtypes = [vp, u32, vp, vp]
    lib.bm25f_phrase_lists.argtypes = [vp, u32, vp, vp, vp, C.POINTER(u32)]
    lib.bm25f_plan_destroy.argtypes = [vp]
    lib.bm25f_plan_destroy.restype = None
    lib.bm25f_search_batch.argtypes = [vp, C.POINTER(QueryBatchDesc), i32, vp, vp, vp, vp]
    lib.bm25f_merge_keys.argtypes = [vp, vp, i32, u32, i32, vp, vp]
    lib.bm25f_decode_keys.argtypes = [vp, vp, u32, i32, vp, vp, vp, vp]
    lib.bm25f_get_stats.argtypes = [vp, C.POINTER(Stats)]
    lib.bm25f_reset_stats.argtypes = [vp]
    lib.bm25f_submit.argtypes = [vp, C.POINTER(QueryBatchDesc), i32, C.POINTER(vp)]
    lib.bm25f_collect.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.bm25f_set_final_date.argtypes = [vp, vp]
    lib.bm25f_fetch_final.argtypes = [vp, vp, vp, vp, vp, vp]
    lib.bm25f_plan_device_final.argtypes = [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]
    lib.bm25f_merge_final_lists.argtypes = [vp, vp, vp, i32, u32, i32, vp, vp, vp, vp]
    lib.bm25f_plan_gather_span.argtypes = [vp, C.POINTER(vp), C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    lib.bm25f_merge_gathered.argtypes = [vp, vp, i32, C.c_uint64, C.c_uint64, u32, i32, vp, vp, vp, vp, vp, vp]
    if lib.bm25f_abi_version() != ABI_VERSION:
        raise RuntimeError("libbm25f ABI %d != binding ABI %d" % (lib.bm25f_abi_version(), ABI_VERSION))
    if path == os.environ.get("BM25F_LIB", LIB_PATH):
        _lib = lib
    return lib


def _check(lib, rc: int):
    if rc != 0:
        raise EngineError(rc, (lib.bm25f_last_error() or b"").decode("utf-8", "replace"))


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class PackedBatch:
    """A lowered query batch in the layout of ``bm25f_query_batch`` (host arrays)."""

    def __init__(self, query_leaf_offsets, query_n_groups, leaf_term, leaf_weight, leaf_group, after_keys=None, after_lo=None):
        self.query_leaf_offsets = np.ascontiguousarray(query_leaf_offsets, dtype=np.uint32)
        self.query_n_groups = np.ascontiguousarray(query_n_groups, dtype=np.uint8)
        self.leaf_term = np.ascontiguousarray(leaf_term, dtype=np.uint32)
        self.leaf_weight = np.ascontiguousarray(leaf_weight, dtype=np.float32)
        self.leaf_group = np.ascontiguousarray(leaf_group, dtype=np.uint8)
        self.after_keys = None if after_keys is None else np.ascontiguousarray(after_keys, dtype=np.uint64)
        self.after_lo = None if after_lo is None else np.ascontiguousarray(after_lo, dtype=np.uint32)
        self.n_queries = int(self.query_n_groups.size)
        self.n_leaves = int(self.leaf_term.size)
        if self.query_leaf_offsets.size != self.n_queries + 1:
            raise ValueError("query_leaf_offsets must have n_queries + 1 entries")

    def desc(self) -> QueryBatchDesc:
        return QueryBatchDesc(self.n_queries, self.n_leaves, _ptr(self.query_leaf_offsets),
                              _ptr(self.query_n_groups), _ptr(self.leaf_term), _ptr(self.leaf_weight),
                              _ptr(self.leaf_group), _ptr(self.after_keys), _ptr(self.after_lo))

    def slice(self, a: int, b: int) -> "PackedBatch":
        o = self.query_leaf_offsets
        la, lb = int(o[a]), int(o[b])
        return PackedBatch(o[a:b + 1] - o[a], self.query_n_groups[a:b], self.leaf_term[la:lb],
                           self.leaf_weight[la:lb], self.leaf_group[la:lb],
                           None if self.after_keys is None else self.after_keys[a:b],
                           None if self.after_lo is None else self.after_lo[a:b])

    @property
    def nbytes(self) -> int:
        n = (self.query_leaf_offsets.nbytes + self.query_n_groups.nbytes + self.leaf_term.nbytes
             + self.leaf_weight.nbytes + self.leaf_group.nbytes)
        return n + (0 if self.after_keys is None else self.after_keys.nbytes)


class Plan:
    def __init__(self, engine: "Engine", handle, n_queries: int, k: int):
        self.engine = engine
        self._p = handle
        self.n_queries = n_queries
        self.k = k

    def execute(self):
        _check(self.engine.lib, self.engine.lib.bm25f_execute(self.engine._h, self._p))

    def fetch(self):
        q, k = self.n_queries, self.k
        scores = np.empty((q, k), dtype=np.float32)
        docids = np.empty((q, k), dtype=np.uint32)
        counts = np.empty(q, dtype=np.uint32)
        totals = np.empty(q, dtype=np.uint64)
        _check(self.engine.lib, self.engine.lib.bm25f_fetch(self.engine._h, self._p, _ptr(scores), _ptr(docids),
                                                              _ptr(counts), _ptr(totals)))
        return scores, docids, counts, totals

    def fetch_final(self):
        """``fetch`` for a plan prepared under a final() weighting: float64 final values instead of scores."""
        q, k = self.n_queries, self.k
        final = np.empty((q, k), dtype=np.float64)
        docids = np.empty((q, k), dtype=np.uint32)
        counts = np.empty(q, dtype=np.uint32)
        totals = np.empty(q, dtype=np.uint64)
        _check(self.engine.lib, self.engine.lib.bm25f_fetch_final(self.engine._h, self._p, _ptr(final), _ptr(docids),
                                                                    _ptr(counts), _ptr(totals)))
        return final, docids, counts, totals

    def device_results(self) -> Tuple[int, int]:
        """Raw device pointers ``(keys [Q*k] u64, totals [Q] u64)``."""
        dk, dt = C.c_void_p(), C.c_void_p()
        _check(self.engine.lib, self.engine.lib.bm25f_plan_device_results(self._p, C.byref(dk), C.byref(dt)))
        return dk.value, dt.value

    def gather_span(self) -> Tuple[int, int, int]:
        """``(device pointer, words, offset of the totals)`` of the span that holds this workspace plan's keys and
        match counts: what one all-gather of the sharded exchange step moves."""
        base, span, off = C.c_void_p(), C.c_uint64(), C.c_uint64()
        _check(self.engine.lib, self.engine.lib.bm25f_plan_gather_span(self._p, C.byref(base), C.byref(span), C.byref(off)))
        return base.value, int(span.value), int(off.value)

    def device_final(self) -> Tuple[int, int, int]:
        """Raw device pointers ``(final values [Q*k] f64, docids [Q*k] u32, totals [Q] u64)`` of a plan prepared
        under a final() weighting."""
        df, dd, dt = C.c_void_p(), C.c_void_p(), C.c_void_p()
        _check(self.engine.lib, self.engine.lib.bm25f_plan_device_final(self._p, C.byref(df), C.byref(dd), C.byref(dt)))
        return df.value, dd.value, dt.value

    def close(self):
        if self._p is not None:
            self.engine.lib.bm25f_plan_destroy(self._p)
            self._p = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Pending:
    """A batch submitted with ``Engine.submit``: its kernels and the copy of its results are in flight."""

    def __init__(self, engine: "Engine", handle, n_queries: int, k: int):
        self.engine = engine
        self._p = handle
        self.n_queries = n_queries
        self.k = k

    def collect(self):
        """Wait for the batch; ``(scores, docids, counts, totals)`` as ``Engine.search_batch`` returns them."""
        if self._p is None:
            raise RuntimeError("batch already collected")
        q, k = self.n_queries, self.k
        scores = np.empty((q, k), dtype=np.float32)
        docids = np.empty((q, k), dtype=np.uint32)
        counts = np.empty(q, dtype=np.uint32)
        totals = np.empty(q, dtype=np.uint64)
        rc = self.engine.lib.bm25f_collect(self.engine._h, self._p, _ptr(scores), _ptr(docids), _ptr(counts),
                                           _ptr(totals))
        if rc != -1:                        # a refused call (BM25F_EINVAL) leaves the batch in flight;
            self._p = None                  # otherwise bm25f_collect has freed the plan
        _check(self.engine.lib, rc)
        return scores, docids, counts, totals


class Engine:
    """One uploaded index shard on one GPU."""

    def __init__(self, ix, device: int = 0, **options):
        """``options``: ``bm25f_options`` fields by name (``OPTION_NAMES``); anything left out is the library default."""
        unknown = sorted(set(options) - set(OPTION_NAMES))
        if unknown:
            raise TypeError("unknown engine option(s): %s" % ", ".join(unknown))
        self.lib = load_library()
        #: a handle serves one call at a time (include/bm25f.h); host layers that share an engine take this lock
        self.lock = threading.RLock()
        self._h = None
        desc = IndexDesc(ABI_VERSION, len(ix.field_names), ix.n_docs_all, ix.n_terms, ix.n_postings, ix.doc_base,
                         _ptr(ix.term_offsets), _ptr(ix.term_field), _ptr(ix.docids), _ptr(ix.tfs),
                         _ptr(ix.len_bytes), _ptr(ix.deleted))
        opts = Options(**{n: int(v) for n, v in options.items()})
        h = C.c_void_p()
        _check(self.lib, self.lib.bm25f_create(C.byref(desc), device, C.byref(opts), C.byref(h)))
        self._h = h
        self.n_docs_all = int(ix.n_docs_all)
        self._final_key = None            # which final() step the handle currently applies (None: none)
        self.device = device
        self.n_fields = len(ix.field_names)
        self._weighting_key = None
        #: fields whose word order is on the device (``put_positions``)
        self.positions_fields = set()

    def set_weighting(self, norm: np.ndarray, key=None):
        norm = np.ascontiguousarray(norm, dtype=np.float32)
        if norm.shape != (self.n_fields, 256):
            raise ValueError("norm tables must be [n_fields, 256]")
        _check(self.lib, self.lib.bm25f_set_weighting(self._h, _ptr(norm)))
        self._weighting_key = key

    def set_final_date(self, date_add: Optional[np.ndarray]):
        """Per-document date term of a DateBM25F-style final() step (NaN: no date); ``None`` switches it off."""
        if date_add is None:
            _check(self.lib, self.lib.bm25f_set_final_date(self._h, None))
            return
        a = np.ascontiguousarray(date_add, dtype=np.float64)
        if a.shape != (self.n_docs_all,):
            raise ValueError("date_add must have one entry per document (%d), got %r" % (self.n_docs_all, a.shape))
        _check(self.lib, self.lib.bm25f_set_final_date(self._h, _ptr(a)))

    def search_batch_final(self, batch: PackedBatch, k: int):
        """prepare + execute + fetch_final with the handle's reusable workspaces."""
        plan = self.prepare(batch, k, arena=True)
        try:
            plan.execute()
            return plan.fetch_final()
        finally:
            plan.close()

    def prepare(self, batch: PackedBatch, k: int, arena: bool = False) -> Plan:
        """``arena=True``: the plan lives in the handle's reusable workspaces (no allocation) and is
        valid until the next arena plan / ``search_batch`` on this engine."""
        d = batch.desc()
        p = C.c_void_p()
        fn = self.lib.bm25f_prepare_arena if arena else self.lib.bm25f_prepare
        _check(self.lib, fn(self._h, C.byref(d), k, C.byref(p)))
        return Plan(self, p, batch.n_queries, k)

    def search_batch(self, batch: PackedBatch, k: int):
        """One synchronous C-ABI call with host buffers in and out."""
        q = batch.n_queries
        scores = np.empty((q, k), dtype=np.float32)
        docids = np.empty((q, k), dtype=np.uint32)
        counts = np.empty(q, dtype=np.uint32)
        totals = np.empty(q, dtype=np.uint64)
        d = batch.desc()
        _check(self.lib, self.lib.bm25f_search_batch(self._h, C.byref(d), k, _ptr(scores), _ptr(docids),
                                                     _ptr(counts), _ptr(totals)))
        return scores, docids, counts, totals

    def submit(self, batch: PackedBatch, k: int) -> Pending:
        """Plan, upload and launch a batch without waiting for it (``bm25f_submit``).  At most two batches
        may be in flight; collect them in submission order."""
        d = batch.desc()
        p = C.c_void_p()
        _check(self.lib, self.lib.bm25f_submit(self._h, C.byref(d), k, C.byref(p)))
        return Pending(self, p, batch.n_queries, k)

    def merge_keys(self, d_keys: int, n_lists: int, n_queries: int, k: int, d_out: int):
        """Runs on the handle's stream (see ``set_stream``)."""
        _check(self.lib, self.lib.bm25f_merge_keys(self._h, d_keys, n_lists, n_queries, k, d_out, None))

    def merge_gathered(self, d_gathered: int, n_lists: int, span: int, totals_offset: int, n_queries: int, k: int,
                       d_keys: int, d_scores: int, d_docids: int, d_counts: int, d_totals: int):
        """Merge + count + decode of an all-gathered exchange buffer; runs on the handle's stream."""
        _check(self.lib, self.lib.bm25f_merge_gathered(self._h, d_gathered, n_lists, span, totals_offset, n_queries, k,
                                                       d_keys, d_scores, d_docids, d_counts, d_totals, None))

    def merge_final_lists(self, d_vals: int, d_docids: int, n_lists: int, n_queries: int, k: int, d_out_final: int,
                          d_out_docids: int, d_out_counts: int):
        """Merge per-shard (final value, docnum) result lists; runs on the handle's stream."""
        _check(self.lib, self.lib.bm25f_merge_final_lists(self._h, d_vals, d_docids, n_lists, n_queries, k, d_out_final,
                                                          d_out_docids, d_out_counts, None))

    def decode_keys(self, d_keys: int, n_queries: int, k: int, d_scores: int, d_docids: int, d_counts: int):
        _check(self.lib, self.lib.bm25f_decode_keys(self._h, d_keys, n_queries, k, d_scores or None,
                                                    d_docids or None, d_counts or None, None))

    def synchronize(self):
        _check(self.lib, self.lib.bm25f_synchronize(self._h))

    def set_stream(self, stream: Optional[int]):
        """Launch on the given ``cudaStream_t`` (e.g. ``torch.cuda.current_stream().cuda_stream``;
        0 is the legacy default stream).  ``None`` restores the library's own stream."""
        if stream is None:
            _check(self.lib, self.lib.bm25f_set_stream(self._h, None, 1))
        else:
            _check(self.lib, self.lib.bm25f_set_stream(self._h, C.c_void_p(stream), 0))

    def put_lists(self, lists) -> int:
        """Hand the library per-batch document lists (``bm25f_put_lists``: phrase filters); ``lists`` are ascending
        local docnum arrays.  Returns the ``leaf_term`` id of the first one; they replace the previous call's lists."""
        offs = np.zeros(len(lists) + 1, dtype=np.uint64)
        if lists:
            np.cumsum([len(x) for x in lists], out=offs[1:])
        docs = (np.ascontiguousarray(np.concatenate([np.asarray(x, dtype=np.uint32) for x in lists]))
                if lists else np.zeros(0, np.uint32))
        first = C.c_uint32()
        _check(self.lib, self.lib.bm25f_put_lists(self._h, len(lists), _ptr(offs), _ptr(docs), C.byref(first)))
        return int(first.value)

    def put_positions(self, field: int, offs: np.ndarray, ids: np.ndarray):
        """Upload one field's word order (``FlatIndex.positions[field]``: document offsets, token ids in document order)
        for the positional filter of ``phrase_lists``; replaces an earlier upload of the field."""
        offs = np.ascontiguousarray(offs, dtype=np.int64)
        if offs.shape != (self.n_docs_all + 1,):
            raise ValueError("offsets must have n_docs_all + 1 = %d entries, got %r" % (self.n_docs_all + 1, offs.shape))
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        if ids.size != int(offs[-1]) or int(offs[0]) != 0:
            raise ValueError("the offsets must run from 0 to the number of tokens (%d)" % ids.size)
        _check(self.lib, self.lib.bm25f_put_positions(self._h, int(field), _ptr(offs.view(np.uint64)), _ptr(ids.view(np.uint32))))
        self.positions_fields.add(int(field))

    def phrase_lists(self, words: Sequence[Sequence[int]], slops: Sequence[int]) -> int:
        """The positional filter on the device (``bm25f_phrase_lists``): phrase ``i`` is the posting-list ids ``words[i]``
        (``TERM_UNKNOWN`` for a word the index does not have) with ``slops[i]``.  Its live matching documents become
        per-batch list ``i``, as ``put_lists`` makes them; returns the ``leaf_term`` id of the first one."""
        wo = np.zeros(len(words) + 1, dtype=np.uint32)
        if words:
            np.cumsum([len(w) for w in words], out=wo[1:])
        flat = np.ascontiguousarray(np.concatenate([np.asarray(w, dtype=np.uint32) for w in words]) if words
                                    else np.zeros(0, np.uint32))
        sl = np.ascontiguousarray(slops, dtype=np.uint32)
        first = C.c_uint32()
        _check(self.lib, self.lib.bm25f_phrase_lists(self._h, len(words), _ptr(wo), _ptr(flat), _ptr(sl), C.byref(first)))
        return int(first.value)

    def stats(self) -> dict:
        s = Stats()
        _check(self.lib, self.lib.bm25f_get_stats(self._h, C.byref(s)))
        return s.as_dict()

    def reset_stats(self):
        _check(self.lib, self.lib.bm25f_reset_stats(self._h))

    def close(self):
        if self._h is not None:
            self.lib.bm25f_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
