"""Exact W11 order (score descending, then docnum ascending) on a corpus whose scores are exact in float32.

The parity gate (tests/parity.py) accepts any document whose score ties with the oracle's at a rank, so it cannot
tell which of several tied documents made the cut.  Here the corpus and the queries are built so that every partial
sum is exact in float32 in any accumulation order:

* B = 0, K1 = 1: the length norm is exactly 1, so a posting's impact ``tf / (tf + 1)`` is 1/2, 3/4 or 7/8 for the
  term counts 1, 3 and 7 the corpus is given;
* every leaf's boost is ``2**e / ((K1 + 1) * idf)``, so its float32 weight ``idf * (K1 + 1) * boost`` is exactly
  ``2**e``.

Every score is then a multiple of 1/8 with a few significant bits, large classes of documents have bit-identical
scores, and every kernel, work split, planner, shard count and page boundary must return the same bits: the
oracle's documents in exact W11 order, its scores snapped to the 1/8 grid, its match counts.  The preconditions
are asserted, so these tests cannot silently decay into the tolerant gate.
"""
from datetime import datetime, timedelta

import numpy as np
import pytest

from document_search_engine_b200 import And, AscDateBM25F, BM25F, DescDateBM25F, Every, FlatIndex, Not, Or, Term
from document_search_engine_b200.corpus import make_corpus
from document_search_engine_b200.distributed import (decode_keys_host, merge_final_host, merge_gathered_host,
                                                      merge_keys_host)
from document_search_engine_b200.numeric import lengths_to_bytes
from document_search_engine_b200.query import GROUP_NOT
from document_search_engine_b200.searching import Searcher, make_keys
from oracle.numpy_oracle import NumpyOracle
from oracle.whoosh_port import OracleSearcher
from tests.test_date_final import FINAL_TOL

K1 = 1.0
TFS = np.array([1, 3, 7], dtype=np.float32)         # impacts tf / (tf + 1) = 1/2, 3/4, 7/8
GRID = 8.0                                          # every score is a multiple of 1 / GRID
UNKNOWN = "no-such-term"
#: top-k sizes around the warp (32), four-keys-per-lane (128), warp-kernel (256) and CTA-kernel (1024) limits
K_ALL = (1, 10, 31, 32, 33, 100, 128, 150, 256, 257, 1024)


# ---- the exact corpus and queries -------------------------------------------------------------------------------

def exact_corpus(n_docs, vocab, seed, deleted=0.2):
    """One ``body`` field, term counts from {1, 3, 7}, a fraction ``deleted`` of the documents deleted."""
    ix = make_corpus(n_docs, vocab, seed, device="cpu")
    rng = np.random.default_rng(seed)
    ix.tfs = np.ascontiguousarray(rng.choice(TFS, ix.tfs.size))
    ix.deleted = (rng.random(n_docs) < deleted).astype(np.uint8)
    return ix


def exact_weighting(cls=BM25F):
    return cls(B=0.0, K1=K1)


def exact_oracle(ix, **kw):
    return NumpyOracle(ix, B=0.0, K1=K1, **kw)


class _Stats:
    """What ``WeightingModel.idf`` reads from a searcher (``Searcher.doc_frequency`` / ``doc_count_all``), without
    an engine, so that queries can be built before any device exists."""

    doc_frequency = Searcher.doc_frequency
    doc_count_all = Searcher.doc_count_all

    def __init__(self, ix):
        self.stats_ix = ix


def pow2_term(ix, t, e):
    """A leaf whose packed float32 weight ``idf * (K1 + 1) * boost`` is exactly ``2**e``."""
    idf = exact_weighting().idf(_Stats(ix), "body", t)
    return Term("body", t, boost=2.0 ** e / ((K1 + 1.0) * idf))


def exact_queries(ix, n, seed, emax=7, max_terms=8, with_not=False):
    """Flat ORs of 1..max_terms terms (some with the densest terms, some with one exponent for every leaf: the
    largest tie classes), ANDs, AND-of-OR variant groups, ``Every``, unknown terms; with ``with_not`` also ``Not``
    clauses.  At most 8 leaves per query, so that the device planner takes a batch without ``Not``."""
    rng = np.random.default_rng(seed)
    V = ix.vocab_size

    def e():
        return int(rng.integers(0, emax + 1))

    def pick(m, dense=False):
        ts = rng.choice(V, size=m, replace=False).tolist()
        if dense:
            ts[0] = int(rng.integers(0, 4))
            ts = list(dict.fromkeys(ts))
        return ts

    def leaves(ts, same=None):
        return [pow2_term(ix, t, e() if same is None else same) for t in ts]

    out = []
    for i in range(n):
        kind = i % (10 if with_not else 8)
        m = int(rng.integers(1, max_terms + 1))
        if kind == 0:
            q = Or(leaves(pick(m)))
        elif kind == 1:
            q = Or(leaves(pick(m, dense=True)))
        elif kind == 2:
            q = Or(leaves(pick(max(2, min(m, 5))), same=e()))
        elif kind == 3:
            q = And(leaves(pick(int(rng.integers(2, 4)))))
        elif kind == 4:
            ts = pick(int(rng.integers(3, min(8, max_terms) + 1)))
            cut = int(rng.integers(1, len(ts)))
            q = And([Or(g) if len(g) > 1 else g[0] for g in (leaves(ts[:cut]), leaves(ts[cut:]))])
        elif kind == 5:
            q = leaves(pick(1, dense=bool(rng.integers(0, 2))))[0]
        elif kind == 6:
            dense = int(rng.integers(0, 4))
            q = And(leaves([dense] + [t for t in pick(2) if t != dense][:1]))
        elif kind == 7:
            q = Or(leaves(pick(max(1, min(m, 4)), dense=True), same=e()))
        elif kind == 8:
            ts = pick(3)
            q = And(leaves(ts[:2]) + [Not(Term("body", ts[2]))])
        else:
            ts = pick(4)
            q = Or(leaves(ts[:2]) + [Not(Or([Term("body", ts[2]), Term("body", ts[3])]))])
        out.append(q)
    t = pick(2)
    out += [Every("body", boost=2.0 ** e()),
            Or([pow2_term(ix, t[0], e()), Term("body", UNKNOWN)]),
            And([pow2_term(ix, t[1], e()), Term("body", UNKNOWN)]),
            Term("body", UNKNOWN)]
    return out


def _positive_terms(q):
    """The scoring leaves of a query tree (``Not`` children excluded) with their boost products."""
    name = type(q).__name__
    if name == "Term":
        return [(q.text, q.boost)]
    if name == "Not":
        return []
    if name in ("And", "Or"):
        return [(t, b * q.boost) for s in q.subqueries for t, b in _positive_terms(s)]
    return []


def host_leaf_weights(ix, queries):
    """float32 weights of the queries' known term leaves, by the arithmetic of ``Searcher.pack`` (float64
    ``(log(dc / (df + 1)) + 1) * (K1 + 1) * boost``, rounded once)."""
    dc = float(ix.doc_count_all())
    tw = (np.log(dc / (ix.df.astype(np.float64) + 1.0)) + 1.0) * (K1 + 1.0)
    out = []
    for q in queries:
        for text, boost in _positive_terms(q):
            tid = ix.term_id("body", text)
            if tid >= 0:
                out.append(tw[tid] * boost)
    return np.asarray(out, dtype=np.float64).astype(np.float32)


def assert_powers_of_two(w):
    w = np.asarray(w, dtype=np.float32)
    mant, _ = np.frexp(w)
    bad = np.nonzero(mant != 0.5)[0]
    assert bad.size == 0, "leaf weights that are not powers of two: %r" % (w[bad[:5]].tolist(),)


def snap(s, ctx=""):
    """Oracle float64 scores on the 1/8 grid (asserted to within 1e-9), as float64."""
    g = np.round(s * GRID) / GRID
    off = np.abs(s - g)
    assert off.size == 0 or off.max() <= 1e-9, "%s score %r is off the 1/8 grid" % (ctx, float(s[np.argmax(off)]))
    return g


def expected(oracle, q, ctx=""):
    """``(docids u32, scores f32)`` of every match in exact W11 order."""
    d, s = oracle.match_all(q)
    g = snap(s, ctx)
    order = np.lexsort((d, -g))
    return d[order].astype(np.uint32), g[order].astype(np.float32)


def assert_rows(want, scores, docids, count, total, k, ctx):
    """One query's result row equals the expected order: docnums exactly, float32 scores bit for bit."""
    wd, ws = want
    n = wd.size if k is None else min(k, wd.size)
    assert int(total) == wd.size, "%s total %d != %d" % (ctx, int(total), wd.size)
    assert int(count) == n, "%s count %d != %d" % (ctx, int(count), n)
    gd = np.asarray(docids[:n], dtype=np.uint32)
    gs = np.asarray(scores[:n], dtype=np.float32)
    if not np.array_equal(gd, wd[:n]) or not np.array_equal(gs.view(np.uint32), ws[:n].view(np.uint32)):
        r = int(np.nonzero((gd != wd[:n]) | (gs.view(np.uint32) != ws[:n].view(np.uint32)))[0][0])
        raise AssertionError("%s rank %d: doc %d score %r, expected doc %d score %r" % (
            ctx, r, int(gd[r]), float(gs[r]), int(wd[r]), float(ws[r])))


def assert_exact(wants, out, k, ctx):
    scores, docids, counts, totals = out
    for i, w in enumerate(wants):
        assert_rows(w, scores[i], docids[i], counts[i], totals[i], k, "%s query %d:" % (ctx, i))


def assert_results_exact(wants, results, k, ctx):
    for i, (w, r) in enumerate(zip(wants, results)):
        top = r.top_n
        assert_rows(w, [s for s, _ in top], [d for _, d in top], len(top), len(r), k, "%s query %d:" % (ctx, i))


# ---- CPU: the generator meets its own preconditions ---------------------------------------------------------------

@pytest.fixture(scope="module")
def small_exact():
    ix = exact_corpus(20_000, 200, 3)
    return ix, exact_queries(ix, 120, 4, with_not=True)


def test_generator_preconditions(small_exact):
    ix, qs = small_exact
    assert_powers_of_two(host_leaf_weights(ix, qs))
    o = exact_oracle(ix)
    sizes = []
    for i, q in enumerate(qs):
        d, _ = expected(o, q, ctx="query %d" % i)
        sizes.append(d.size)
    assert max(sizes) > 10_000 and sizes[-1] == 0 and sizes[-2] == 0
    # the ties the tests are about: a single dense term has three score classes of thousands of documents
    d, s = expected(o, pow2_term(ix, 0, 3))
    vals, counts = np.unique(s, return_counts=True)
    assert vals.tolist() == [4.0, 6.0, 7.0] and counts.min() > 1000


def test_preconditions_fire_when_broken(small_exact):
    """The strict comparison is only as good as its preconditions: each check fails on inputs that break it."""
    ix, qs = small_exact
    with pytest.raises(AssertionError, match="grid"):
        for q in qs[:8]:
            expected(NumpyOracle(ix, B=0.75, K1=K1), q)          # length norms off the grid
    with pytest.raises(AssertionError, match="powers of two"):
        assert_powers_of_two(host_leaf_weights(ix, [Or([Term("body", 5), Term("body", 9)])]))   # plain idf weights
    tfs = ix.tfs
    try:
        ix.tfs = tfs + np.float32(1.0)                            # impacts 2/3, 4/5, 8/9
        with pytest.raises(AssertionError, match="grid"):
            for q in qs[:8]:
                expected(exact_oracle(ix), q)
    finally:
        ix.tfs = tfs


def test_oracles_agree_on_exact_order():
    """The vectorised oracle and the doc-at-a-time Whoosh port give the identical exact order on this corpus.  Both
    add float64 leaf scores, in different orders, so their raw sums differ in the last bits and order tied documents
    by that noise; snapped to the grid, matches, scores and order must be identical."""
    ix = exact_corpus(3000, 80, 5)
    qs = exact_queries(ix, 40, 6, with_not=True)
    o = exact_oracle(ix)
    port = OracleSearcher(ix, B=0.0, K1=K1)
    for i, q in enumerate(qs):
        wd, ws = expected(o, q, "query %d" % i)
        top_p, total_p = port.search(q, limit=None)
        assert total_p == wd.size, "query %d" % i
        d = np.array([d for _, d in top_p], dtype=np.uint32)
        g = snap(np.array([s for s, _ in top_p], dtype=np.float64), "port query %d" % i)
        order = np.lexsort((d, -g))
        assert np.array_equal(d[order], wd), "query %d" % i
        assert np.array_equal(g[order].astype(np.float32), ws), "query %d" % i


# ---- GPU ------------------------------------------------------------------------------------------------------------

N_DOCS, VOCAB = 200_000, 300


class Exact:
    """The exact corpus with its query batches and their expected orders."""

    def __init__(self):
        self.ix = ix = exact_corpus(N_DOCS, VOCAB, 20261020)
        self.oracle = o = exact_oracle(ix)
        self.big = exact_queries(ix, 300, 11)                  # >= 256 queries, no Not: the device planner's batch
        self.small = exact_queries(ix, 50, 12, with_not=True)
        self.want_big = [expected(o, q, "big %d" % i) for i, q in enumerate(self.big)]
        self.want_small = [expected(o, q, "small %d" % i) for i, q in enumerate(self.small)]
        # limit=None / deep pages: queries with more matches than one kernel pass returns, but not the whole corpus
        tot = [w[0].size for w in self.want_big]
        self.deep = [i for i in range(len(self.big)) if 1024 < tot[i] < 30_000][:10] + \
                    [i for i in range(len(self.big)) if 0 < tot[i] <= 1024][:3] + [len(self.big) - 3]

    def searcher(self, **opts):
        return Searcher(self.ix, weighting=exact_weighting(), **opts)

    def close_engines(self):
        for eng in self.ix._engine_cache.values():
            eng.close()
        self.ix._engine_cache.clear()


@pytest.fixture(scope="module")
def ex():
    e = Exact()
    yield e
    e.close_engines()


#: small work items: many items per query, hence many partial lists and merge steps
SMALL = dict(tile_docs=1024, split_postings=2048, subtile_docs=128, warp_split=2048, cta_slice_docs=128, cta_split=2048,
             isect_split=128)
CONFIGS = [("auto", {}), ("host_plan", dict(host_plan=1)), ("pipe", dict(variant=1)), ("cta", dict(variant=2)),
           ("stream", dict(variant=3)), ("team", dict(variant=4)), ("isect", dict(variant=5)),
           ("auto_small", SMALL)] + [("%s_small" % n, dict(SMALL, variant=v))
                                     for n, v in (("pipe", 1), ("cta", 2), ("stream", 3), ("team", 4), ("isect", 5))]


@pytest.mark.gpu
def test_leaf_weights_are_exact_powers_of_two(ex):
    s = ex.searcher()
    for qs in (ex.big, ex.small):
        b = s.pack(qs)
        known = (b.leaf_term != 0xFFFFFFFF) & (b.leaf_group != GROUP_NOT)     # a Not child scores nothing
        assert known.sum() > len(qs)
        assert_powers_of_two(b.leaf_weight[known])


@pytest.mark.gpu
@pytest.mark.parametrize("name,opts", CONFIGS, ids=[c[0] for c in CONFIGS])
def test_exact_order_every_kernel_and_split(ex, name, opts):
    """Every kernel family and work split returns the expected order bit for bit, for every k; the batch with
    ``Not`` clauses for every k the NOT path serves; ``limit=None`` and limits past 1024 through the paging bound."""
    s = ex.searcher(**opts)
    big, small = s.pack(ex.big), s.pack(ex.small)
    for k in K_ALL:
        assert_exact(ex.want_big, s.search_packed(big, k), k, "%s k=%d big" % (name, k))
        if k <= 256:
            assert_exact(ex.want_small, s.search_packed(small, k), k, "%s k=%d small" % (name, k))
    deep = [ex.big[i] for i in ex.deep]
    want = [ex.want_big[i] for i in ex.deep]
    for limit in (None, 2500):
        assert_results_exact(want, s.search_batch(deep, limit=limit), limit, "%s limit=%s" % (name, limit))
    ex.close_engines()


@pytest.mark.gpu
def test_device_planner_takes_the_big_batch(ex):
    """The batch of >= 256 queries is planned on the device: three more launches than with ``host_plan``."""
    launches = {}
    for name, opts in (("dev", {}), ("host", dict(host_plan=1))):
        s = ex.searcher(**opts)
        b = s.pack(ex.big)
        s.search_packed(b, 10)
        s.engine.reset_stats()
        s.search_packed(b, 10)
        launches[name] = s.engine.stats()["n_launches"]
        ex.close_engines()
    assert launches["dev"] >= launches["host"] + 3


@pytest.mark.gpu
def test_every_limit_none(ex):
    """``Every`` (one constant score: a single tie class of every live document) through all the paging passes."""
    s = ex.searcher()
    q = [ex.big[-4]]
    assert type(q[0]).__name__ == "Every"
    assert_results_exact([ex.want_big[-4]], s.search_batch(q, limit=None), None, "Every limit=None")


@pytest.mark.gpu
@pytest.mark.parametrize("pagelen", [10, 150])
def test_pages_split_tie_classes(ex, pagelen):
    """``search_page`` pages whose boundaries fall inside tie classes of thousands of documents, up to and past the
    1024 hits of one kernel pass: concatenated, they are the expected order, no duplicates, no gaps."""
    s = ex.searcher()
    qs = [pow2_term(ex.ix, 0, 2), Or([pow2_term(ex.ix, 1, 0), pow2_term(ex.ix, 2, 0)]), ex.big[ex.deep[0]]]
    pages = list(range(1, 13)) + ([110, 111] if pagelen == 10 else [])
    for j, q in enumerate(qs):
        wd, ws = expected(ex.oracle, q)
        for p in pages:
            page = s.search_page(q, p, pagelen)
            lo = (p - 1) * pagelen
            if lo >= wd.size:
                continue
            hits = list(page)
            assert page.total == wd.size and page.offset == lo
            assert [h.docnum for h in hits] == wd[lo:lo + pagelen].tolist(), "query %d page %d" % (j, p)
            assert np.array_equal(np.array([h.score for h in hits], np.float32).view(np.uint32),
                                  ws[lo:lo + pagelen].view(np.uint32)), "query %d page %d" % (j, p)


def lagging_warp_index(n_warps, slice_docs, n_top=32):
    """A corpus laid out for ``k_score_team`` with ``n_warps`` warps and slices of ``slice_docs`` documents: terms
    0..6 are in every document of slice 0 (tf 1), term 7 in ``n_top`` documents of slice ``n_warps`` and
    ``n_top`` documents of slice ``n_warps + 1`` (tf 7), nothing else.  Slices go round-robin to the warps, so
    warp 0 is busy with 7 * slice_docs postings while warp 1 skips its empty first slice, scores its second and
    publishes its k-th best score; warp 0 then scores its second slice, whose documents tie with that threshold
    exactly and have the lower docnums."""
    n = (n_warps + 2) * slice_docs
    heavy = np.arange(slice_docs, dtype=np.uint32)
    top = np.concatenate([n_warps * slice_docs + 100 + 7 * np.arange(n_top),
                          (n_warps + 1) * slice_docs + 50 + 5 * np.arange(n_top)]).astype(np.uint32)
    lists = [heavy] * 7 + [top]
    tfs = [np.ones(heavy.size, np.float32)] * 7 + [np.full(top.size, 7.0, np.float32)]
    offs = np.concatenate([[0], np.cumsum([x.size for x in lists])]).astype(np.uint64)
    return FlatIndex(field_names=["body"], n_docs_all=n, term_offsets=offs, docids=np.concatenate(lists),
                     tfs=np.concatenate(tfs), term_field=np.zeros(len(lists), np.uint8),
                     len_bytes=lengths_to_bytes(np.full(n, 100))[None, :],
                     field_length_total=np.array([100 * n], np.uint64), vocab_size=len(lists))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 10, 32])
def test_team_threshold_tie_across_warps(k):
    """The warp-team kernel shares one admission threshold per CTA (the largest k-th best score of any warp).  A
    document whose score equals that threshold can still belong in the top k when its docnum is lower than the
    documents that set it; here a warp that lags behind meets exactly such documents."""
    NW, SW = 3, 12288
    ix = lagging_warp_index(NW, SW)
    q = Or([pow2_term(ix, t, 0) for t in range(7)] + [pow2_term(ix, 7, 7)])
    want = expected(exact_oracle(ix), q)
    assert want[1][0] == 112.0 and (want[1] == 112.0).sum() == 64
    for opts in (dict(variant=4, cta_warps=NW, cta_slice_docs=SW, cta_split=1 << 30), {}):
        s = Searcher(ix, weighting=exact_weighting(), **opts)
        out = s.search_packed(s.pack([q]), k)
        if opts:
            assert s.engine.stats()["postings_team"] > 0
        assert_exact([want], out, k, "%r k=%d" % (opts, k))
        s.engine.close()
        ix._engine_cache.clear()


# ---- date-ordered weightings: final() values under exact ties ------------------------------------------------------

def whole_day_dates(ix, seed, n_days=40):
    """Stored fields with a date at a whole day (no time, no chapter) shared by thousands of documents, one
    document in ten without a date."""
    rng = np.random.default_rng(seed)
    day = rng.integers(0, n_days, ix.n_docs_all)
    undated = rng.random(ix.n_docs_all) < 0.1
    base = datetime(1964, 1, 6)
    ix.stored = [{"heading": "Session %d" % day[i]} if undated[i] else
                 {"heading": "Session %d" % day[i], "date": base + timedelta(days=7 * int(day[i]))}
                 for i in range(ix.n_docs_all)]
    return ix


def expected_final(oracle, add, q, ctx=""):
    """``(docids u32, final values f64)`` of every match in exact order, from the grid scores; distinct
    (date, score) classes must be far apart compared with FINAL_TOL, so the order is not a matter of rounding."""
    d, s = oracle.match_all(q)
    g = snap(s, ctx)
    t = 1 - 1 / g
    a = add[d]
    dated = ~np.isnan(a)
    v = np.where(dated, (t + np.where(dated, a, 0.0)) / 10 ** 9, t)
    if v.size:
        classes = np.unique(np.stack([np.where(dated, a, -1.0), g]), axis=1).shape[1]
        u = np.unique(v)
        assert u.size == classes, "%s two (date, score) classes share a final value" % ctx
        assert u.size < 2 or np.diff(u).min() > 100 * FINAL_TOL, "%s (date, score) classes closer than 100 * FINAL_TOL" % ctx
    order = np.lexsort((d, -v))
    return d[order].astype(np.uint32), v[order]


def assert_final_rows(want, vals, docids, count, total, k, ctx):
    wd, wv = want
    n = wd.size if k is None else min(k, wd.size)
    assert int(total) == wd.size, "%s total %d != %d" % (ctx, int(total), wd.size)
    assert int(count) == n, "%s count %d != %d" % (ctx, int(count), n)
    gd = np.asarray(docids[:n], dtype=np.uint32)
    if not np.array_equal(gd, wd[:n]):
        r = int(np.nonzero(gd != wd[:n])[0][0])
        raise AssertionError("%s rank %d: doc %d, expected doc %d" % (ctx, r, int(gd[r]), int(wd[r])))
    err = np.abs(np.asarray(vals[:n], dtype=np.float64) - wv[:n])
    assert err.size == 0 or err.max() <= FINAL_TOL, "%s final value off by %g" % (ctx, float(err.max()))


@pytest.fixture(scope="module")
def dated(ex):
    ix = whole_day_dates(ex.ix, 5)
    qs = exact_queries(ix, 80, 21, emax=2, max_terms=4)[:-1]       # scores <= 14: classes 6e-13 apart
    out = {}
    for cls in (DescDateBM25F, AscDateBM25F):
        add = cls().doc_final_terms(ix)
        want = [expected_final(ex.oracle, add, q, "%s query %d" % (cls.__name__, i)) for i, q in enumerate(qs)]
        # the formula above is the oracle's
        o = exact_oracle(ix, final_add=add)
        for q, (wd, wv) in zip(qs[:10], want):
            d, v = o.match_all(q)
            ref = dict(zip(d.tolist(), v.tolist()))
            assert all(abs(ref[x] - y) <= FINAL_TOL for x, y in zip(wd.tolist(), wv.tolist()))
        out[cls] = want
    yield ix, qs, out
    ex.close_engines()


@pytest.mark.gpu
@pytest.mark.parametrize("cls", [DescDateBM25F, AscDateBM25F])
def test_final_exact_order(dated, cls):
    ix, qs, wants = dated
    want = wants[cls]
    s = Searcher(ix, weighting=exact_weighting(cls))
    b = s.pack(qs)
    for k in (3, 10, 100, 150, 256):
        vals, docids, counts, totals = s.search_packed(b, k)
        for i, w in enumerate(want):
            assert_final_rows(w, vals[i], docids[i], counts[i], totals[i], k, "%s k=%d query %d:" % (cls.__name__, k, i))
    # limit=None and limits past 256: further passes bounded by the last (final value, docnum) returned
    deep = [i for i, w in enumerate(want) if 256 < w[0].size < 8000][:8] + [i for i, w in enumerate(want) if 0 < w[0].size < 256][:2]
    assert len(deep) >= 6
    for limit in (None, 700):
        res = s.search_batch([qs[i] for i in deep], limit=limit)
        for j, i in enumerate(deep):
            top = res[j].top_n
            assert_final_rows(want[i], [v for v, _ in top], [d for _, d in top], len(top), len(res[j]), limit,
                              "%s limit=%s query %d:" % (cls.__name__, limit, i))
    i = deep[0]
    for p, pagelen in ((30, 10), (2, 150), (3, 100)):
        page = s.search_page(qs[i], p, pagelen)
        lo = (p - 1) * pagelen
        assert page.total == want[i][0].size and page.offset == lo
        assert [h.docnum for h in page] == want[i][0][lo:lo + pagelen].tolist(), "page %d of %d" % (p, pagelen)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 150, 256])
def test_final_shards_merge_exact(dated, k):
    """Three shards' (final value, docnum) lists merged by bm25f_merge_final_lists: the whole index's result, final
    values bit for bit (one float32 score and one date term give one float64 value on every shard)."""
    import torch
    from document_search_engine_b200.distributed import device_view
    ix, qs, wants = dated
    Q, G = len(qs), 3
    w = exact_weighting(DescDateBM25F)
    s = Searcher(ix, weighting=w)
    whole = s.search_packed(s.pack(qs), k)
    vals = torch.empty(G * Q * k, dtype=torch.float64, device="cuda:0")
    docs = torch.empty(G * Q * k, dtype=torch.int32, device="cuda:0")
    totals = np.zeros(Q, dtype=np.uint64)
    searchers = [Searcher(ix.shard(g, G), weighting=w, stats_ix=ix) for g in range(G)]
    for g, s in enumerate(searchers):
        plan = s.engine.prepare(s.pack(qs), k, arena=True)
        plan.execute()
        d_final, d_docids, d_totals = plan.device_final()
        s.engine.synchronize()
        vals[g * Q * k:(g + 1) * Q * k].copy_(device_view(d_final, Q * k, 0, "<f8"))
        docs[g * Q * k:(g + 1) * Q * k].copy_(device_view(d_docids, Q * k, 0, "<i4"))
        totals += device_view(d_totals, Q, 0).cpu().numpy().view(np.uint64)
        plan.close()
    torch.cuda.synchronize()
    out_v = torch.empty(Q * k, dtype=torch.float64, device="cuda:0")
    out_d = torch.empty(Q * k, dtype=torch.int32, device="cuda:0")
    out_c = torch.empty(Q, dtype=torch.int32, device="cuda:0")
    eng = searchers[0].engine
    eng.merge_final_lists(vals.data_ptr(), docs.data_ptr(), G, Q, k, out_v.data_ptr(), out_d.data_ptr(), out_c.data_ptr())
    eng.synchronize()
    v = out_v.cpu().numpy().reshape(Q, k)
    d = out_d.cpu().numpy().view(np.uint32).reshape(Q, k)
    c = out_c.cpu().numpy().view(np.uint32)
    for i, want in enumerate(wants[DescDateBM25F]):
        assert_final_rows(want, v[i], d[i], c[i], totals[i], k, "k=%d query %d:" % (k, i))
        n = int(c[i])
        assert np.array_equal(v[i, :n].view(np.uint64), whole[0][i, :n].view(np.uint64)), "k=%d query %d" % (k, i)
    assert np.array_equal(totals, whole[3]) and np.array_equal(c, whole[2])
    for s in searchers:
        s.engine.close()


# ---- document shards and the exchange kernels on one GPU ----------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3, 8])
def test_emulated_all_gather_equals_whole(ex, G):
    """Every shard's gather span (keys, then match counts) copied into one [G, span] tensor - what
    ``all_gather_into_tensor`` produces - and merged by ``bm25f_merge_gathered``: the whole index's result bit for
    bit, totals included; warp merge for k <= 32, bitonic merge above."""
    import torch
    from document_search_engine_b200.distributed import device_view
    ix = ex.ix
    searchers = [Searcher(ix.shard(g, G), weighting=exact_weighting(), stats_ix=ix) for g in range(G)]
    assert sum(s.ix.n_docs_all for s in searchers) == ix.n_docs_all
    batches = [s.pack(ex.big) for s in searchers]
    Q = len(ex.big)
    eng = searchers[0].engine
    for k in (1, 10, 32, 33, 100, 150, 256, 1024):
        gathered = None
        for g, (s, b) in enumerate(zip(searchers, batches)):
            plan = s.engine.prepare(b, k, arena=True)
            plan.execute()
            base, span, tot_off = plan.gather_span()
            assert tot_off >= Q * k and span == tot_off + Q
            s.engine.synchronize()
            if gathered is None:
                gathered = torch.empty((G, span), dtype=torch.int64, device="cuda:0")
                span0 = span
            assert span == span0
            gathered[g].copy_(device_view(base, span, 0))
            plan.close()
        torch.cuda.synchronize()
        keys = torch.empty(Q * k, dtype=torch.int64, device="cuda:0")
        scores = torch.empty(Q * k, dtype=torch.float32, device="cuda:0")
        docids = torch.empty(Q * k, dtype=torch.int32, device="cuda:0")
        counts = torch.empty(Q, dtype=torch.int32, device="cuda:0")
        totals = torch.empty(Q, dtype=torch.int64, device="cuda:0")
        eng.merge_gathered(gathered.data_ptr(), G, span0, tot_off, Q, k, keys.data_ptr(), scores.data_ptr(),
                           docids.data_ptr(), counts.data_ptr(), totals.data_ptr())
        eng.synchronize()
        out = (scores.cpu().numpy().reshape(Q, k), docids.cpu().numpy().view(np.uint32).reshape(Q, k),
               counts.cpu().numpy(), totals.cpu().numpy())
        assert_exact(ex.want_big, out, k, "G=%d k=%d" % (G, k))
        hk, ht = merge_gathered_host(gathered.cpu().numpy().view(np.uint64), Q, k, tot_off)
        assert np.array_equal(keys.cpu().numpy().view(np.uint64).reshape(Q, k), hk)
        assert np.array_equal(totals.cpu().numpy().view(np.uint64), ht)
    for s in searchers:
        s.engine.close()


@pytest.mark.gpu
def test_sharded_searcher_world_one(ex):
    """``ShardedSearcher.run_plan`` with one rank: the decode-only branch (``bm25f_decode_keys``)."""
    from document_search_engine_b200.distributed import ShardedSearcher
    ss = ShardedSearcher(ex.ix, rank=0, world=1, device=0, weighting=exact_weighting())
    try:
        b = ss.pack(ex.big)
        for k in (1, 10, 33, 150, 1024):
            assert_exact(ex.want_big, ss.search_packed(b, k), k, "world=1 k=%d" % k)
    finally:
        ss.engine.set_stream(None)
        ex.close_engines()


def synthetic_lists(rng, G, Q, k, empty_frac=0.1):
    """``[G, Q, k]`` uint64 key lists: each sorted descending with a random length < k and zero-padded, some queries
    empty on every list; scores from a small set with exact ties and negative values, docnums unique per query."""
    s = rng.choice(np.array([-3.5, -0.125, 0.0, 0.5, 0.75, 1.0, 7.875, 1e30], np.float32), size=(G, Q, k))
    i = np.arange(k, dtype=np.uint64)[None, None, :]
    g = np.arange(G, dtype=np.uint64)[:, None, None]
    with np.errstate(over="ignore"):
        d = ((i * np.uint64(G) + g) * np.uint64(2654435761)) & np.uint64(0xFFFFFFFF)    # a bijection on 32 bits
    d = np.broadcast_to(d, (G, Q, k))
    keys = make_keys(s.reshape(-1), d.reshape(-1)).reshape(G, Q, k)
    keys = np.sort(keys, axis=2)[:, :, ::-1]
    length = rng.integers(0, k, size=(G, Q))
    length[:, rng.random(Q) < empty_frac] = 0
    keys = np.where(np.arange(k)[None, None, :] < length[:, :, None], keys, np.uint64(0))
    return np.ascontiguousarray(keys)


@pytest.mark.gpu
def test_exchange_kernels_on_synthetic_keys():
    """``bm25f_merge_gathered``, ``bm25f_merge_keys`` and ``bm25f_decode_keys`` bit for bit against their host
    restatements: lists of random lengths < k, all-empty lists, negative scores, exact ties, k that are not powers
    of two, garbage between the keys and the counts, shard counts that add up past 2^32."""
    import torch
    from document_search_engine_b200._ffi import EngineError
    ix = exact_corpus(2000, 50, 1)
    s = Searcher(ix, weighting=exact_weighting())
    eng = s.engine
    rng = np.random.default_rng(7)
    dev = "cuda:0"

    def t(a, dtype=torch.int64):
        return torch.from_numpy(np.ascontiguousarray(a).view(np.int64 if dtype == torch.int64 else np.int32)).to(dev)

    ks = [1, 5, 31, 32, 33, 100, 257, 1024]
    covered, n = set(), 0
    for G in (1, 2, 3, 8, 17):
        for Q in (1, 7, 9, 1000):
            n += 1
            for k in ks[n % len(ks)::3][:2 if Q == 1000 else 3]:
                covered.add(k)
                keys = synthetic_lists(rng, G, Q, k)
                pad = int(rng.integers(1, 9))
                tot_off = Q * k + pad
                span = tot_off + Q + int(rng.integers(0, 3))
                gathered = rng.integers(0, 1 << 63, size=(G, span), dtype=np.int64).view(np.uint64)
                gathered[:, :Q * k] = keys.reshape(G, Q * k)
                # every shard's count fits 32 bits, two of them add up past 2^32
                gathered[:, tot_off:tot_off + Q] = rng.integers(1 << 31, 1 << 32, size=(G, Q), dtype=np.uint64)
                want_keys, want_tot = merge_gathered_host(gathered, Q, k, tot_off)
                ws, wd, wc = decode_keys_host(want_keys)
                ctx = "G=%d Q=%d k=%d" % (G, Q, k)

                g_dev = t(gathered)
                out_k = torch.empty(Q * k, dtype=torch.int64, device=dev)
                out_s = torch.empty(Q * k, dtype=torch.float32, device=dev)
                out_d = torch.empty(Q * k, dtype=torch.int32, device=dev)
                out_c = torch.empty(Q, dtype=torch.int32, device=dev)
                out_t = torch.empty(Q, dtype=torch.int64, device=dev)
                eng.merge_gathered(g_dev.data_ptr(), G, span, tot_off, Q, k, out_k.data_ptr(), out_s.data_ptr(),
                                   out_d.data_ptr(), out_c.data_ptr(), out_t.data_ptr())
                eng.synchronize()
                assert np.array_equal(out_k.cpu().numpy().view(np.uint64).reshape(Q, k), want_keys), ctx
                assert np.array_equal(out_s.cpu().numpy().view(np.uint32).reshape(Q, k), ws.view(np.uint32)), ctx
                assert np.array_equal(out_d.cpu().numpy().view(np.uint32).reshape(Q, k), wd), ctx
                assert np.array_equal(out_c.cpu().numpy().view(np.uint32), wc), ctx
                assert np.array_equal(out_t.cpu().numpy().view(np.uint64), want_tot), ctx
                if G > 1:
                    assert want_tot.min() >= 1 << 32, ctx

                # the same lists without the counts: bm25f_merge_keys, then bm25f_decode_keys (counts only, too)
                k_dev = t(keys)
                eng.merge_keys(k_dev.data_ptr(), G, Q, k, out_k.data_ptr())
                eng.synchronize()
                assert np.array_equal(out_k.cpu().numpy().view(np.uint64).reshape(Q, k), merge_keys_host(keys, k)), ctx
                out_c.fill_(-1)
                eng.decode_keys(out_k.data_ptr(), Q, k, 0, 0, out_c.data_ptr())
                eng.synchronize()
                assert np.array_equal(out_c.cpu().numpy().view(np.uint32), wc), ctx
                out_s.zero_()
                out_d.zero_()
                eng.decode_keys(out_k.data_ptr(), Q, k, out_s.data_ptr(), out_d.data_ptr(), out_c.data_ptr())
                eng.synchronize()
                assert np.array_equal(out_s.cpu().numpy().view(np.uint32).reshape(Q, k), ws.view(np.uint32)), ctx
                assert np.array_equal(out_d.cpu().numpy().view(np.uint32).reshape(Q, k), wd), ctx
    assert covered == set(ks)
    # refused: a span that cannot hold the keys, k = 0
    buf = torch.zeros(4096, dtype=torch.int64, device=dev)
    p = buf.data_ptr()
    with pytest.raises(EngineError):
        eng.merge_gathered(p, 2, 9 * 10 - 1, 9 * 10 - 1, 9, 10, p, p, p, p, p)
    with pytest.raises(EngineError):
        eng.merge_gathered(p, 2, 100, 90, 9, 0, p, p, p, p, p)
    with pytest.raises(EngineError):
        eng.merge_keys(p, 2, 9, 0, p)
    eng.close()
    ix._engine_cache.clear()


@pytest.mark.gpu
def test_merge_final_lists_on_synthetic_ties():
    """``bm25f_merge_final_lists`` against ``merge_final_host`` with final values that tie exactly across lists."""
    import torch
    ix = exact_corpus(2000, 50, 1)
    s = Searcher(ix, weighting=exact_weighting())
    eng = s.engine
    rng = np.random.default_rng(9)
    dev = "cuda:0"
    for G, Q, k in ((1, 7, 10), (2, 9, 33), (3, 1000, 100), (8, 7, 256), (17, 9, 150), (5, 1, 1)):
        v = rng.choice(np.array([5.51, 5.5, 0.75, 0.5, -1.0]), size=(G, Q, k))
        i = np.arange(k, dtype=np.uint64)[None, None, :]
        g = np.arange(G, dtype=np.uint64)[:, None, None]
        d = np.broadcast_to(((i * np.uint64(G) + g) * np.uint64(2654435761)) % np.uint64(0xFFFFFFFF), (G, Q, k)).astype(np.uint32)
        order = np.lexsort((d, -v), axis=2)
        v = np.take_along_axis(v, order, 2)
        d = np.take_along_axis(d, order, 2)
        length = rng.integers(0, k + 1, size=(G, Q))
        empty = np.arange(k)[None, None, :] >= length[:, :, None]
        d = np.where(empty, np.uint32(0xFFFFFFFF), d)
        v = np.where(empty, rng.random((G, Q, k)), v)                    # garbage values in empty slots
        wv, wd, wc = merge_final_host(v, d, k)
        out_v = torch.empty(Q * k, dtype=torch.float64, device=dev)
        out_d = torch.empty(Q * k, dtype=torch.int32, device=dev)
        out_c = torch.empty(Q, dtype=torch.int32, device=dev)
        vd = torch.from_numpy(np.ascontiguousarray(v)).to(dev)
        dd = torch.from_numpy(np.ascontiguousarray(d).view(np.int32)).to(dev)
        eng.merge_final_lists(vd.data_ptr(), dd.data_ptr(), G, Q, k, out_v.data_ptr(), out_d.data_ptr(), out_c.data_ptr())
        eng.synchronize()
        ctx = "G=%d Q=%d k=%d" % (G, Q, k)
        assert np.array_equal(out_v.cpu().numpy().reshape(Q, k), wv), ctx
        assert np.array_equal(out_d.cpu().numpy().view(np.uint32).reshape(Q, k), wd), ctx
        assert np.array_equal(out_c.cpu().numpy().view(np.uint32), wc), ctx
    eng.close()
    ix._engine_cache.clear()
