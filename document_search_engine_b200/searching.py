"""``Searcher`` / ``Results`` / ``ResultsPage`` / ``Hit`` with the Whoosh contract the
reference's front ends consume (SURVEY.md §8 a9, b).

Call sites served (reference file:line):

* ``with ix.searcher(weighting=weighting) as searcher``            my_flask.py:184
* ``searcher.search_page(qp, pagenum=..., pagelen=...)``            my_flask.py:208, :211
* ``searcher.search(qp, limit=MAXIMUM_SAME_SESSION_HITS + 1)``      my_flask.py:304
* ``results.scored_length()``, ``results[0]['session']``, iteration  my_flask.py:306, :315
* ``page.total / .offset / .pagelen / .pagenum / len(page)``        my_flask.py:212, :287-293
* ``hit.docnum``, ``hit['field']``, ``hit.results.q``, ``hit.searcher``  my_flask.py:326-380
* ``searcher.ixreader.frequency('exact', word)``                    my_flask.py:254
* ``searcher.stored_fields(docnum)``                                my_whoosh.py:131

New: ``search_batch(queries, limit)`` — the batched entry the GPU wants.  Scoring and
top-k always run on the GPU through ``libbm25f``; there is no CPU path here.
"""
from __future__ import annotations

import gc
import struct
import time
from math import ceil, log
from collections.abc import Sequence as _SequenceABC
from typing import Iterable, List, Optional, Sequence

import numpy as np

from . import _ffi
from .query import (FILTER_FIELD, And, Or, Query, Term, UnsupportedQuery, expand_multiterms, expand_phrases, has_multiterm,
                    has_phrase, lower)
from .scoring import BM25F, instantiate

#: one lowered leaf as ``Searcher.pack`` keeps it: posting-list id (or -1 / -2 - field), boost, group
_LEAF_REC = np.dtype([("tid", "<i8"), ("boost", "<f8"), ("group", "u1"), ("pad", "V7")])
_LEAF_STRUCT = struct.Struct("<qdB7x")
_LEAF_STRUCTS = {}


def _leaf_struct(n: int) -> struct.Struct:
    """``n`` leaf records in one ``struct`` call."""
    st = _LEAF_STRUCTS.get(n)
    if st is None:
        st = _LEAF_STRUCTS[n] = struct.Struct("<" + "qdB7x" * n)
    return st


#: ``tid`` of the leaf that stands for per-batch document list ``i`` (a phrase's positional test): ``_FILTER_TID - i``
_FILTER_TID = -1000
#: its weight: positive for the library, invisible next to any float32 score
FILTER_WEIGHT = 1e-29

#: bound on the per-call tile-boundary table (bytes); larger batches are split
BOUNDS_BYTES_PER_CALL = 1 << 30
DEFAULT_TILE_DOCS = 8192
#: largest limit the device serves under a final() weighting (the warp kernels keep up to 8 keys per lane;
#: the reference's listing page asks for 150, my_flask.py:208)
FINAL_MAX_K = 256


def make_keys(scores: np.ndarray, docids: np.ndarray) -> np.ndarray:
    """The engine's 64-bit W11 ordering key (score desc, docnum asc), host version."""
    u = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32).astype(np.uint64)
    neg = (u & np.uint64(0x80000000)) != 0
    u = np.where(neg, (~u) & np.uint64(0xFFFFFFFF), u | np.uint64(0x80000000))
    return (u << np.uint64(32)) | (np.uint64(0xFFFFFFFF) - docids.astype(np.uint64))


def orderable_f64(v: np.ndarray) -> np.ndarray:
    """float64 -> uint64 with the same order (the high part of the engine's 96-bit final() keys, csrc/final.cuh)."""
    u = np.ascontiguousarray(v, dtype=np.float64).view(np.uint64)
    neg = (u >> np.uint64(63)) != 0
    return np.where(neg, ~u, u | np.uint64(0x8000000000000000))


class Hit:
    def __init__(self, results: "Results", docnum: int, pos: int, score: float):
        self.results = results
        self.searcher = results.searcher
        self.docnum = docnum
        self.pos = self.rank = pos
        self.score = score
        self._fields = None

    def fields(self):
        if self._fields is None:
            self._fields = self.searcher.stored_fields(self.docnum)
        return self._fields

    def __getitem__(self, name):
        return self.fields()[name]

    def __contains__(self, name):
        return name in self.fields()

    def get(self, name, default=None):
        return self.fields().get(name, default)

    def keys(self):
        return self.fields().keys()

    def __iter__(self):
        return iter(self.fields())

    def __len__(self):
        return len(self.fields())

    def __repr__(self):
        return "<Hit %r>" % (dict(self.fields()),)

    def highlights(self, fieldname, text=None, top=3, minscore=1):
        raise NotImplementedError("highlighting is outside the scoring path (SURVEY.md §2: out of scope)")


class Results:
    """Scored top-N plus the exact match count (``len(results)``, W13)."""

    def __init__(self, searcher: "Searcher", q: Query, top_n, total: int, runtime: float = 0.0, rows=None):
        self.searcher = searcher
        self.q = q
        #: ``[(score, docnum)]`` in W11 order; built on first use from the engine's result rows when the batch
        #: entry made this object (``rows = (scores row, docids row, count)``)
        self._top_n = None if top_n is None else list(top_n)
        self._rows = rows
        self._total = int(total)
        self.runtime = runtime
        # settable presentation hooks the reference assigns (my_flask.py:349-352)
        self.fragmenter = None
        self.order = None
        self.scorer = None
        self.formatter = None

    @property
    def top_n(self):
        t = self._top_n
        if t is None:
            sc, dc, n = self._rows
            t = self._top_n = list(zip(sc[:n].tolist(), dc[:n].tolist()))
        return t

    @top_n.setter
    def top_n(self, value):
        self._top_n = list(value)

    def __len__(self):
        return self._total

    def __repr__(self):
        return "<Top %s Results for %r runtime=%s>" % (len(self.top_n), self.q, self.runtime)

    def scored_length(self):
        return len(self.top_n)

    def has_exact_length(self):
        return True

    def estimated_length(self):
        return self._total

    def estimated_min_length(self):
        return self._total

    def is_empty(self):
        return self._total == 0

    def score(self, n):
        return self.top_n[n][0]

    def docnum(self, n):
        return self.top_n[n][1]

    def docs(self):
        return set(d for _, d in self.top_n)

    def fields(self, n):
        return self.searcher.stored_fields(self.top_n[n][1])

    def __getitem__(self, n):
        if isinstance(n, slice):
            start, stop, step = n.indices(len(self.top_n))
            return [Hit(self, self.top_n[i][1], i, self.top_n[i][0]) for i in range(start, stop, step)]
        if n < 0:
            n += len(self.top_n)
        if n >= len(self.top_n) or n < 0:
            raise IndexError("results[%r]: Results only has %s hits" % (n, len(self.top_n)))
        return Hit(self, self.top_n[n][1], n, self.top_n[n][0])

    def __iter__(self):
        for i in range(len(self.top_n)):
            yield Hit(self, self.top_n[i][1], i, self.top_n[i][0])


class BatchResults(_SequenceABC):
    """What ``search_batch`` returns: a read-only sequence of ``Results``, one per query, over the engine's result
    arrays.  A ``Results`` object is built when its position is read (a 10k-query batch is returned in the time
    the GPU needs, not in the time Python needs to make 10k objects)."""

    def __init__(self, searcher, queries, scores, docids, counts, totals, runtime):
        self.searcher, self.queries = searcher, queries
        self.scores, self.docids, self.counts, self.totals = scores, docids, counts, totals
        self.runtime = runtime
        self._made = {}

    def __len__(self):
        return len(self.queries)

    def __getitem__(self, i):
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(len(self.queries)))]
        if i < 0:
            i += len(self.queries)
        if not 0 <= i < len(self.queries):
            raise IndexError(i)
        r = self._made.get(i)
        if r is None:
            r = self._made[i] = Results(self.searcher, self.queries[i], None, int(self.totals[i]), runtime=self.runtime,
                                        rows=(self.scores[i], self.docids[i], int(self.counts[i])))
        return r

    def __eq__(self, other):
        return list(self) == list(other)

    def __repr__(self):
        return "<BatchResults of %d queries>" % len(self.queries)


class ResultsPage:
    """W13: a page view over ``search(q, limit=pagenum * pagelen)``."""

    def __init__(self, results: Results, pagenum: int, pagelen: int = 10):
        self.results = results
        self.total = len(results)
        if pagenum < 1:
            raise ValueError("pagenum must be >= 1")
        self.pagecount = int(ceil(self.total / pagelen))
        self.pagenum = min(self.pagecount, pagenum)
        offset = (self.pagenum - 1) * pagelen
        if (offset + pagelen) > self.total:
            pagelen = self.total - offset
        self.offset = offset
        self.pagelen = pagelen

    def __getitem__(self, n):
        offset = self.offset
        if isinstance(n, slice):
            start, stop, step = n.indices(self.pagelen)
            return self.results.__getitem__(slice(start + offset, stop + offset, step))
        return self.results.__getitem__(n + offset)

    def __iter__(self):
        return iter(self.results[self.offset:self.offset + self.pagelen])

    def __len__(self):
        return self.total          # the reference relies on this (my_flask.py:212)

    def scored_length(self):
        return self.results.scored_length()

    def score(self, n):
        return self.results.score(n + self.offset)

    def docnum(self, n):
        return self.results.docnum(n + self.offset)

    def is_last_page(self):
        return self.pagecount == 0 or self.pagenum == self.pagecount


class Searcher:
    """Whoosh-shaped searcher over a ``FlatIndex`` whose postings live in HBM."""

    def __init__(self, ix, weighting=None, device: int = 0, stats_ix=None, **engine_options):
        """``engine_options``: ``bm25f_options`` fields by name (``_ffi.OPTION_NAMES``), e.g. ``variant=3``."""
        self.ix = ix
        #: index the corpus statistics come from (the whole corpus when ``ix`` is a shard, W8)
        self.stats_ix = stats_ix or ix
        self.weighting = instantiate(weighting)
        if not isinstance(self.weighting, BM25F):
            raise NotImplementedError("only BM25F weightings run on the GPU path")
        if self.weighting.use_final and not hasattr(self.weighting, "doc_final_terms"):
            raise NotImplementedError(
                "a weighting with use_final=True must provide doc_final_terms(ix) (see scoring.DateBM25F): "
                "final() is applied to every match before the top-k (W14), which only the device can do")
        self.device = device
        self.ixreader = self.stats_ix.reader()
        engine_options = {n: int(v) for n, v in engine_options.items() if v}
        key = (device,) + tuple(sorted(engine_options.items()))
        with ix._engine_cache_lock:
            eng = ix._engine_cache.get(key)
            if eng is None:
                eng = _ffi.Engine(ix, device=device, **engine_options)
                ix._engine_cache[key] = eng
        self.engine = eng
        # The engine (the uploaded index) is shared by every searcher of this index, but its weighting (impact
        # pairs) and final() table are handle state: every search call re-binds them under the engine's lock
        # (the reference opens a searcher per request with the weighting of the requested hit order, my_flask.py:183-184).
        self._wkey = self.weighting.norm_key() + (self.stats_ix.doc_count_all(),)
        self._fkey = self.weighting.key() if self.weighting.use_final else None
        with eng.lock:
            self._bind()
        self._idf_cache = {}
        self._term_w = None
        self.closed = False

    def _bind(self):
        """Make the shared engine score with this searcher's weighting (call with ``engine.lock`` held)."""
        eng = self.engine
        if eng._weighting_key != self._wkey:
            eng.set_weighting(self.weighting.norm_tables(self.stats_ix), key=self._wkey)
        if eng._final_key != self._fkey:
            # a final() step (DateBM25F: my_whoosh.py:127-154) runs on the device, over every match (W14)
            eng.set_final_date(None if self._fkey is None else self.weighting.doc_final_terms(self.ix))
            eng._final_key = self._fkey

    # -- context manager / lifetime (my_flask.py:184) ---------------------------
    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def close(self):
        self.closed = True       # the uploaded index stays cached on the FlatIndex

    # -- statistics ---------------------------------------------------------------
    def doc_count_all(self):
        return self.stats_ix.doc_count_all()

    def doc_count(self):
        return self.stats_ix.doc_count()

    def doc_frequency(self, fieldname, text):
        tid = self.stats_ix.term_id(fieldname, text)
        return 0 if tid < 0 else int(self.stats_ix.df[tid])

    def idf(self, fieldname, text):
        k = (fieldname, text)
        v = self._idf_cache.get(k)
        if v is None:
            v = self.weighting.idf(self, fieldname, text)
            self._idf_cache[k] = v
        return v

    def avg_field_length(self, fieldname):
        return self.stats_ix.avg_field_length(fieldname)

    def stored_fields(self, docnum):
        return self.stats_ix.stored_fields(docnum)

    def reader(self):
        return self.ixreader

    def get_parent(self):
        return self

    # -- lowering -------------------------------------------------------------------
    def _term_weights(self) -> np.ndarray:
        """float64 ``[n_terms]``: ``idf * (K1 + 1)`` of every posting list (W3 with the corpus-wide df / dc), or 1
        for a term of a field that is not scorable (W15: WeightScorer, the leaf weight is the boost alone)."""
        tw = self._term_w
        if tw is None:
            sx = self.stats_ix
            dc = float(sx.doc_count_all())
            tw = (np.log(dc / (sx.df.astype(np.float64) + 1.0)) + 1.0) * (self.weighting.K1 + 1.0)
            for f, name in enumerate(sx.field_names):
                if not sx.is_scorable(name):
                    tw[sx.term_field == f] = 1.0
            self._term_w = tw
        return tw

    def _make_tid_of(self):
        """``(fieldname, text) -> posting-list id or -1`` as a closure over the index's dictionary (``FlatIndex.term_id``
        without the per-call field search)."""
        ix = self.ix
        fmap = {name: f for f, name in enumerate(ix.field_names)}
        terms, vs, slow = ix.terms, ix.vocab_size, ix.term_id

        if terms is not None:
            def tid_of(fieldname, text):
                f = fmap.get(fieldname)
                return -1 if f is None else terms.get((f, text), -1)
        else:
            def tid_of(fieldname, text):
                if type(text) is int:
                    f = fmap.get(fieldname)
                    return f * vs + text if f is not None and 0 <= text < vs else -1
                return slow(fieldname, text)
        self.__dict__["_tid_of"] = tid_of
        return tid_of

    def _lower_one(self, q: Query, register=None):
        """``(index, n_leaves, n_groups, packed leaf records, query)`` of one query: what ``pack`` needs, remembered
        on the query object.  A leaf record is ``_LEAF_REC``: posting-list id (-1: unknown term or field, W10;
        ``-2 - f``: ``Every`` on field ``f``), boost, group."""
        ix = self.ix
        cls = type(q)
        cacheable = True
        tid_of = self.__dict__.get("_tid_of") or self._make_tid_of()
        if cls is Term:
            return (ix.token, 1, 1, _LEAF_STRUCT.pack(tid_of(q.fieldname, q.text), q.boost, 0), True)
        elif (cls is And or cls is Or) and 0 < len(q.subqueries) <= 32 and all([type(t) is Term for t in q.subqueries]):
            # the common shapes (the reference's form: words joined by AND / OR) skip the general lowering; one
            # struct call packs all the leaves
            subs = q.subqueries
            n = len(subs)
            qb = q.boost
            flat = []
            if cls is And:
                for i, t in enumerate(subs):
                    flat += (tid_of(t.fieldname, t.text), t.boost * qb, i)
            else:
                for t in subs:
                    flat += (tid_of(t.fieldname, t.text), t.boost * qb, 0)
            return (ix.token, n, n if cls is And else 1, _leaf_struct(n).pack(*flat), True)
        else:
            if has_phrase(q):
                # a phrase is And(its words, the documents that pass the positional test): the latter is a per-batch
                # list (bm25f_phrase_lists), numbered by ``register``; such a lowering is not remembered on the query
                if register is None:
                    raise UnsupportedQuery("phrase queries are served by search() / search_page() / search_batch(), "
                                           "not by pre-packed batches: %r" % (q,))
                q = expand_phrases(q, register)
                cacheable = False
            if has_multiterm(q):
                # Prefix / Wildcard: Whoosh's MultiTerm.matcher expands the pattern over the field's lexicon into an
                # Or of Terms (reference UI: book:tes?, search-form.html:20-40); same rewrite here, on the host
                q = expand_multiterms(q, ix.lexicon)
            low, g, kind = lower(q)
            if kind == "every":
                # Whoosh's Every(field): every live document that has the field, constant score = boost
                # (reference cli.py:9).  The library keeps one posting list per field for it.
                f = ix.field_index(low[0].fieldname)
                leaves = [(-1 if f < 0 else -2 - f, float(low[0].boost), 0)]
            elif kind == "null":
                leaves, g = [], 0
            else:
                if len(low) > _ffi.MAX_LEAVES_PER_QUERY:
                    raise UnsupportedQuery("more than %d leaves in one query" % _ffi.MAX_LEAVES_PER_QUERY)
                if g > 32:
                    raise UnsupportedQuery("more than 32 AND-groups in one query")
                leaves = [((_FILTER_TID - lf.text) if lf.fieldname == FILTER_FIELD else ix.term_id(lf.fieldname, lf.text), lf.boost, lf.group)
                          for lf in low]
        return (ix.token, len(leaves), g, b"".join([_LEAF_STRUCT.pack(tid, boost, group) for tid, boost, group in leaves]), cacheable)

    def pack(self, queries: Sequence[Query], after_keys: Optional[np.ndarray] = None,
             after_lo: Optional[np.ndarray] = None, filters_ok: bool = False) -> _ffi.PackedBatch:
        """Lower query trees to the ``bm25f_query_batch`` layout.  Leaf weights ``idf * (K1 + 1) * boost`` are
        evaluated in float64 and rounded once (numpy gathers over a per-term table).  The lowered form of a query
        is remembered on the query object (query trees are values: the reference builds one per request,
        ``my_flask.py:189-193``, and never edits it), so packing the same objects again costs three list appends
        per query."""
        token = self.ix.token
        counts: List[int] = []
        ngroups: List[int] = []
        blobs: List[bytes] = []
        lower1 = self._lower_one
        phrases: List[Query] = []             # the batch's distinct phrases = its per-batch document lists

        def register(p):
            try:
                return phrases.index(p)
            except ValueError:
                phrases.append(p)
                return len(phrases) - 1
        reg = register if filters_ok else None
        gc_was_on = gc.isenabled()
        gc.disable()                             # thousands of small objects: a collection in here costs more than the loop
        try:
            for q in queries:
                c = q.__dict__.get("_lowered")
                if c is None or c[0] != token:
                    c = lower1(q, reg)
                    if c[4]:
                        q.__dict__["_lowered"] = c
                counts.append(c[1])
                ngroups.append(c[2])
                blobs.append(c[3])
        finally:
            if gc_was_on:
                gc.enable()
        offs = np.zeros(len(counts) + 1, dtype=np.uint32)
        np.cumsum(counts, out=offs[1:])
        rec = np.frombuffer(b"".join(blobs), dtype=_LEAF_REC)
        tids = rec["tid"]
        known = tids >= 0
        w = np.zeros(rec.size, dtype=np.float64)
        if rec.size:
            w[known] = self._term_weights()[tids[known]]
            w *= rec["boost"]
        terms = np.where(known, tids, _ffi.TERM_UNKNOWN).astype(np.uint32)
        if phrases:
            # [W] Phrase: the positions decide whether a document matches, the score is the words' alone.  The
            # documents that pass (the positional filter runs on the device) become per-batch posting lists; their
            # leaves get a weight far below float32 resolution of any score (and above the library's "positive
            # weight" bar)
            first = self._phrase_lists(phrases)
            flt = tids <= _FILTER_TID
            terms[flt] = (first + (_FILTER_TID - tids[flt])).astype(np.uint32)
            w[flt] = FILTER_WEIGHT
        ev = (tids <= -2) & (tids > _FILTER_TID)      # Every(field): constant-score pseudo lists, weight = boost
        if ev.any():
            terms[ev] = (_ffi.TERM_EVERY_BASE + (-2 - tids[ev])).astype(np.uint32)
            w[ev] = rec["boost"][ev]
        return _ffi.PackedBatch(offs, np.asarray(ngroups, dtype=np.uint8), terms, w, rec["group"], after_keys, after_lo)

    def _phrase_lists(self, phrases: Sequence[Query]) -> int:
        """Run the positional filter of the batch's phrases on the device (``Engine.phrase_lists``; the same documents
        as ``FlatIndex.phrase_docs`` minus the deleted ones).  A field's word order is uploaded the first time a phrase
        on it reaches the engine."""
        ix, eng = self.ix, self.engine
        words, slops = [], []
        for p in phrases:
            f = ix.field_index(p.fieldname)
            if f >= 0:
                if f not in ix.positions:
                    raise NotImplementedError("field %r was flattened without positions: no phrase queries on it" % p.fieldname)
                with eng.lock:
                    if f not in eng.positions_fields:
                        eng.put_positions(f, *ix.positions[f])
            tids = [ix.term_id(p.fieldname, w) for w in p.words]
            words.append([_ffi.TERM_UNKNOWN if t < 0 else t for t in tids])
            slops.append(min(max(p.slop, 0), 0xFFFFFFFF))          # slop <= 0: no position follows another by <= 0
        return eng.phrase_lists(words, slops)

    # -- searching ----------------------------------------------------------------
    def _run_packed(self, batch: _ffi.PackedBatch, k: int):
        """Run a packed batch, splitting it so the boundary table stays bounded."""
        T = max(1, -(-self.ix.n_docs_all // (self.engine.stats()["tile_docs"] or DEFAULT_TILE_DOCS)))
        max_leaves = max(_ffi.MAX_LEAVES_PER_QUERY, BOUNDS_BYTES_PER_CALL // (4 * (T + 1)))
        if batch.n_leaves <= max_leaves:
            return self.engine.search_batch(batch, k)
        outs = []
        a = 0
        offs = batch.query_leaf_offsets
        while a < batch.n_queries:
            b = int(np.searchsorted(offs, offs[a] + max_leaves, side="right")) - 1
            b = min(max(b, a + 1), batch.n_queries)
            outs.append(self.engine.search_batch(batch.slice(a, b), k))
            a = b
        return tuple(np.concatenate([o[i] for o in outs]) for i in range(4))

    def search_packed(self, batch: _ffi.PackedBatch, limit: int = 10):
        """``(scores [Q,k] f32, docids [Q,k] u32, counts [Q], totals [Q])`` for a packed batch (float64 final
        values instead of scores under a final() weighting)."""
        if limit < 1 or limit > _ffi.MAX_K:
            raise ValueError("limit must be 1..%d for search_packed" % _ffi.MAX_K)
        with self.engine.lock:
            self._bind()
            if self.weighting.use_final:
                if limit > FINAL_MAX_K:
                    raise NotImplementedError("a final() weighting is served for limit <= %d" % FINAL_MAX_K)
                return self.engine.search_batch_final(batch, limit)
            return self._run_packed(batch, limit)

    def search_packed_stream(self, batches, limit: int = 10):
        """``search_packed`` over an iterable of packed batches, pipelined two deep: while the GPU scores
        batch i, the host plans and uploads batch i + 1 (``bm25f_submit`` / ``bm25f_collect``).  Yields the
        result tuples in order.  This is the throughput form for a server that answers request batches
        back to back; the latency of one batch is that of ``search_packed``."""
        if limit < 1 or limit > _ffi.MAX_K:
            raise ValueError("limit must be 1..%d for search_packed_stream" % _ffi.MAX_K)
        if self.weighting.use_final:                     # float64 results: one blocking call per batch
            for batch in batches:
                yield self.search_packed(batch, limit)
            return
        T = max(1, -(-self.ix.n_docs_all // (self.engine.stats()["tile_docs"] or DEFAULT_TILE_DOCS)))
        max_leaves = max(_ffi.MAX_LEAVES_PER_QUERY, BOUNDS_BYTES_PER_CALL // (4 * (T + 1)))
        pending = None
        self.engine.lock.acquire()                       # the handle is this stream's until the generator ends
        try:
            self._bind()
            for batch in batches:
                if batch.n_leaves > max_leaves:          # needs splitting: not pipelined
                    if pending is not None:
                        p, pending = pending, None
                        yield p.collect()
                    yield self._run_packed(batch, limit)
                    continue
                nxt = self.engine.submit(batch, limit)
                if pending is not None:
                    p, pending = pending, nxt
                    yield p.collect()
                else:
                    pending = nxt
            if pending is not None:
                p, pending = pending, None
                yield p.collect()
        finally:
            try:
                if pending is not None:                  # the consumer stopped early: free the workspace
                    pending.collect()
            finally:
                self.engine.lock.release()

    def search_batch(self, queries: Sequence[Query], limit: Optional[int] = 10) -> List[Results]:
        """Batched ``search``: one GPU pass for all queries (several when ``limit`` is
        ``None`` or exceeds the kernel's top-k capacity: the next pass collects only hits
        ordered strictly after the last one already returned)."""
        with self.engine.lock:
            self._bind()
            return self._search_batch_locked(queries, limit)

    def _search_batch_locked(self, queries: Sequence[Query], limit: Optional[int]) -> List[Results]:
        t_start = time.perf_counter()
        queries = list(queries)
        nq = len(queries)
        if self.weighting.use_final:
            # final values (float64) come straight from the device; one pass serves limit <= 256, deeper pages
            # (search_page(qp, pagenum=26, pagelen=10) on a date-ordered listing, my_flask.py:211) take another pass
            # for the hits ordered strictly after the last one already returned
            tops: List[list] = [[] for _ in range(nq)]
            totals = np.zeros(nq, dtype=np.uint64)
            active = list(range(nq))
            after_hi = after_lo = None
            first = True
            while active:
                k = FINAL_MAX_K if limit is None else min(limit, FINAL_MAX_K)
                batch = self.pack([queries[i] for i in active], after_hi, after_lo, filters_ok=True)
                final, docids, counts, tot = self.engine.search_batch_final(batch, k)
                nxt, nh, nlo = [], [], []
                for j, i in enumerate(active):
                    c = int(counts[j])
                    if first:
                        totals[i] = tot[j]
                    tops[i].extend(zip(final[j, :c].tolist(), docids[j, :c].tolist()))
                    need = int(totals[i]) if limit is None else min(limit, int(totals[i]))
                    if c == k and len(tops[i]) < need:
                        nxt.append(i)
                        nh.append(final[j, c - 1])
                        nlo.append(0xFFFFFFFF - int(docids[j, c - 1]))
                if limit is not None:
                    for i in active:
                        del tops[i][limit:]
                active = nxt
                if nxt:
                    after_hi, after_lo = orderable_f64(np.asarray(nh, dtype=np.float64)), np.asarray(nlo, dtype=np.uint32)
                first = False
            dt = time.perf_counter() - t_start
            return [Results(self, queries[i], tops[i], int(totals[i]), runtime=dt) for i in range(nq)]
        if limit is not None and limit <= _ffi.MAX_K:
            # one pass serves every query: the per-query Results are made when somebody looks at them
            scores, docids, counts, tot = self._run_packed(self.pack(queries, filters_ok=True), limit)
            return BatchResults(self, queries, scores, docids, counts, tot, time.perf_counter() - t_start)
        want = [limit if limit is not None else None] * nq
        tops: List[list] = [[] for _ in range(nq)]
        totals = np.zeros(nq, dtype=np.uint64)
        active = list(range(nq))
        after = None
        first = True
        while active:
            k = _ffi.MAX_K if limit is None else min(limit, _ffi.MAX_K)
            batch = self.pack([queries[i] for i in active], after, filters_ok=True)
            scores, docids, counts, tot = self._run_packed(batch, k)
            nxt, nxt_after = [], []
            for j, i in enumerate(active):
                c = int(counts[j])
                if first:
                    totals[i] = tot[j]
                tops[i].extend(zip(scores[j, :c].tolist(), docids[j, :c].tolist()))
                need = int(totals[i]) if want[i] is None else min(want[i], int(totals[i]))
                if c == k and len(tops[i]) < need:
                    nxt.append(i)
                    nxt_after.append(make_keys(scores[j, c - 1:c], docids[j, c - 1:c])[0])
            if limit is not None:
                for i in active:
                    del tops[i][limit:]
            active = nxt
            after = np.asarray(nxt_after, dtype=np.uint64) if nxt else None
            first = False
        dt = time.perf_counter() - t_start
        return [Results(self, queries[i], tops[i], int(totals[i]), runtime=dt) for i in range(nq)]

    # -- key terms / more-like-this (reference my_flask.py:428-446, my_index.py:100) -------------------------------
    def key_terms_from_text(self, fieldname, text, numterms=5, normalize=True):
        """``[(word, weight)]``: the terms of ``text`` (a token list, or a string split on whitespace: analysis is the
        caller's, SURVEY.md section 2) that best tell it from the collection, by Whoosh's default Bo1 model
        (``classify.Expander`` / ``Bo1Model`` [W])."""
        toks = text.split() if isinstance(text, str) else list(text)
        return self._expanded_terms(fieldname, [(t, 1.0) for t in toks], numterms, normalize)

    def key_terms(self, docnums, fieldname, numterms=5, normalize=True):
        """The same for the term vectors of the given documents (``s.key_terms([doc], field, numterms=10)``,
        reference ``my_index.py:100``)."""
        vec = []
        for d in docnums:
            vec.extend(self.stats_ix.doc_terms(d, fieldname))
        return self._expanded_terms(fieldname, vec, numterms, normalize)

    def _expanded_terms(self, fieldname, vector, numterms, normalize):
        sx = self.stats_ix
        top_total, top_weight = 0.0, {}
        for word, weight in vector:
            top_total += weight
            top_weight[word] = top_weight.get(word, 0.0) + weight
        if not top_weight:
            return []
        N = float(sx.doc_count_all())
        tlist, maxweight = [], 0.0
        for word, weight in top_weight.items():
            if sx.term_id(fieldname, word) < 0:
                continue
            f = sx.term_frequency(fieldname, word) / N
            score = weight * log((1.0 + f) / f, 2) + log(1.0 + f, 2)         # Bo1Model.score
            maxweight = max(maxweight, score)
            tlist.append((score, word))
        if not tlist:
            return []
        if normalize:
            f = maxweight / N
            norm = (maxweight * log((1.0 + f) / f) + log(1.0 + f)) / log(2.0)  # Bo1Model.normalizer
        else:
            norm = maxweight
        tlist = [(weight / norm, t) for weight, t in tlist]
        tlist.sort(key=lambda x: (0 - x[0], x[1]))
        return [(t, weight) for weight, t in tlist[:numterms]]

    def more_like(self, docnum, fieldname, text=None, top=10, numterms=5, normalize=True):
        """Whoosh ``Searcher.more_like`` (reference ``my_flask.py:431-434``: ``more_like(docnum | None, 'exact', text=...,
        top=5)``): the key terms of ``text`` (or of document ``docnum``) become an ``Or`` of boosted terms, scored on
        the GPU like any other query; document ``docnum`` itself is masked out of the hits and of the total."""
        if text:
            kts = self.key_terms_from_text(fieldname, text, numterms=numterms, normalize=normalize)
        else:
            kts = self.key_terms([docnum], fieldname, numterms=numterms, normalize=normalize)
        q = Or([Term(fieldname, word, boost=weight) for word, weight in kts])
        if not kts:
            return Results(self, q, [], 0)
        r = self.search(q, limit=top + (0 if docnum is None else 1))
        if docnum is not None:
            masked = any(t == docnum for t in (d for _, d in r.top_n))
            hits = [(s, d) for s, d in r.top_n if d != docnum][:top]
            sx = self.stats_ix
            in_mask = masked or any(self._doc_has_term(sx, docnum, fieldname, w) for w, _ in kts)
            return Results(self, q, hits, len(r) - (1 if in_mask else 0), runtime=r.runtime)
        return r

    @staticmethod
    def _doc_has_term(ix, docnum, fieldname, word) -> bool:
        tid = ix.term_id(fieldname, word)
        if tid < 0:
            return False
        d, _ = ix.postings(tid)
        i = int(np.searchsorted(d, docnum - ix.doc_base))
        live = ix.deleted is None or not ix.deleted[docnum - ix.doc_base]
        return i < d.size and int(d[i]) == docnum - ix.doc_base and live

    def search(self, q: Query, limit: Optional[int] = 10, **kwargs) -> Results:
        if limit is not None and limit < 1:
            raise ValueError("limit must be >= 1")
        return self.search_batch([q], limit=limit)[0]

    def search_page(self, q: Query, pagenum: int, pagelen: int = 10, **kwargs) -> ResultsPage:
        if pagenum < 1:
            raise ValueError("pagenum must be >= 1")
        return ResultsPage(self.search(q, limit=pagenum * pagelen, **kwargs), pagenum, pagelen)
