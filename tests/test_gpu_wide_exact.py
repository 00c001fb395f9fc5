"""Bit-exact results for wide and many-group queries on every kernel that serves them.

``tests/test_gpu_score_exact.py`` checks scores bit for bit against an exact host model (``Model``), but only on
narrow queries: at most 13 leaves, about 3 AND-groups, positive boosts.  The reference UI's filters reach the engine
as much wider queries - ``book:tes?`` / ``Prefix`` expand into up to 256 OR leaves, ``date:[oct 1965 to dec 8 1967]``
into a cover of dozens of year, month and day tokens, and ``And`` of those and words gives many leaves in many
groups - and those shapes are served by code paths the narrow queries never reach:

* 9-32 leaves: ``k_score_isect`` (one lane per leaf at 32 leaves, the full group mask at 32 groups) or the CTA kernels;
* 33-256 leaves: ``k_score_pipe`` / ``k_score_topk`` (per-tile leaf walks, ``u8`` group counters up to 32 groups, the
  per-query boundary table of ``n_leaves x (T + 1)`` rows, the 256-entry shared leaf and bound tables);
* a zero, negative or <= 1e-30 leaf weight: the whole batch on ``k_score_topk``, scores <= 0, exact cancellation,
  negative keys and paging through a negative tail;
* 2-32 AND-groups, ``Not`` with 30 groups, and the refusals just past every limit;
* batches whose boundary table is too large for one call (split by ``Searcher._run_packed``).

Every GPU assertion compares float32 scores (as uint32), docnums, counts and totals with the model, without
tolerance.  Which kernel served a batch is asserted from the engine's ``postings_*`` statistics.  The CPU part checks
that every ladder has its exact live leaf and group counts after the planner's dropping rules, that the model is BM25F
on these shapes, that the corpora discriminate (reversed leaf order and largest-first groups change scores), and that
``fma_exact`` - a vectorised ``fmaf`` emulation that keeps the model fast on 30k-posting lists - equals the
rational-arithmetic ``fma_f32``.
"""
from datetime import date, datetime, timedelta
from fractions import Fraction

import numpy as np
import pytest

from document_search_engine_b200 import And, BM25F, DateRange, DescDateBM25F, FlatIndex, Not, Or, Prefix, Term, Wildcard
from document_search_engine_b200 import searching
from document_search_engine_b200._ffi import EngineError, PackedBatch
from document_search_engine_b200.query import UnsupportedQuery, expand_multiterms
from document_search_engine_b200.searching import Searcher
from oracle.numpy_oracle import NumpyOracle
from tests.test_gpu_score_exact import (K_ALL, TERM_UNKNOWN, VOCAB, WEIGHTING, Model, ScoreCorpus, assert_exact,
                                        assert_results, engineless_searcher, fma_f32, round_f32)

BAR = np.float32(1e-30)            # the planner's "positive weight" bar (bm25f_prepare: w > 1e-30f)


# ---- a vectorised exact fmaf -------------------------------------------------------------------------------------

def fma_exact(w, u, acc) -> np.ndarray:
    """``fmaf(w, u, acc)`` elementwise, vectorised.  ``p = w * u`` is exact in float64 and ``s = p + acc`` is
    ``RN64(x)`` of the exact sum ``x`` with two-sum error ``err = x - s``.  Every boundary between two float32 (a
    float32 midpoint) is a float64 number, and rounding is monotone, so ``RN32(s) != RN32(x)`` only when ``s`` is
    itself a float32 midpoint and ``err != 0``: then ``x`` lies on the side of the midpoint that ``err`` points to."""
    w, u, acc = (np.atleast_1d(np.asarray(x, dtype=np.float32)) for x in (w, u, acc))
    w, u, acc = np.broadcast_arrays(w, u, acc)
    p = w.astype(np.float64) * u.astype(np.float64)
    a = acc.astype(np.float64)
    s = p + a
    bv = s - p
    err = (p - (s - bv)) + (a - bv)
    f = s.astype(np.float32)
    f64 = f.astype(np.float64)
    # the float32 neighbour of f on the side of s; s is a midpoint when it is halfway between the two
    other = np.nextafter(f, np.where(s > f64, np.float32(np.inf), np.float32(-np.inf)))
    mid = (err != 0) & (f64 != s) & ((f64 + other.astype(np.float64)) * 0.5 == s)
    # x is beyond the midpoint (towards `other`) when err points the way s lies from f
    flip = mid & ((err > 0) == (s > f64))
    f[flip] = other[flip]
    return f


# ---- WideCorpus ----------------------------------------------------------------------------------------------------

N_WIDE = 30_000
N_COMMON = 40
DATE0 = datetime(1960, 1, 1)
N_DAYS = 3653                       # 1960-01-01 .. 1969-12-31
#: pattern families in the body field: prefix -> (words in the lexicon, words whose every posting is deleted)
FAMILIES = {"qa": (32, 0), "qb": (34, 1), "qc": (256, 1), "qd": (256, 0), "qe": (257, 0)}


def cw(i):
    return "c%02d" % i


class WideCorpus:
    """30k documents: title and body (scorable, different B), a non-scorable ``book`` and a ``date`` field; 20 %
    deleted; 40 common body words in ~95 % of documents (tf 1..5) so that ANDs of 32 single-word groups match
    thousands; pattern families whose expansions give 32, 33, 255, 256 and 257 terms; dates over a decade."""

    def __init__(self, seed=20261022):
        rng = np.random.default_rng(seed)
        n = N_WIDE
        body = [[] for _ in range(n)]
        title = [[] for _ in range(n)]
        for i in range(N_COMMON):
            has = np.nonzero(rng.random(n) < 0.95)[0]
            tf = rng.integers(1, 6, has.size)
            for d, t in zip(has.tolist(), tf.tolist()):
                body[d] += [cw(i)] * t
            for d in np.nonzero(rng.random(n) < 0.12)[0].tolist():
                title[d].append(cw(i))
        filler = rng.zipf(1.3, (n, 12)) % 3000
        for d in range(n):
            body[d] += ["w%d" % x for x in filler[d]]
            title[d] += ["w%d" % x for x in filler[d, :3]]
        deleted = rng.random(n) < 0.2
        self.pattern_words = {}
        for pre, (nw, ndead) in FAMILIES.items():
            width = 2 if nw <= 100 else 3
            words = ["%s%0*d" % (pre, width, j) for j in range(nw)]
            self.pattern_words[pre] = words
            for j, word in enumerate(words):
                docs = rng.choice(n, int(rng.integers(5, 60)), replace=False)
                if j >= nw - ndead:
                    deleted[docs] = True          # every posting of this word is deleted: dropped by the planner
                for d, t in zip(docs.tolist(), rng.integers(1, 4, docs.size).tolist()):
                    body[d] += [word] * t
        books = rng.integers(0, 12, n)
        days = rng.integers(0, N_DAYS, n)
        docs = [{"title": title[d], "body": body[d], "book": "b%d" % books[d],
                 "date": DATE0 + timedelta(days=int(days[d]))} for d in range(n)]
        self.ix = ix = FlatIndex.from_documents(docs, ["title", "body"], id_fields=["book"], date_fields=["date"], stored=["date"],
                                                deleted=np.nonzero(deleted)[0].tolist())
        # length bytes 0, 1, 254 and 255 in both scorable fields, on live documents
        live = np.nonzero(~deleted)[0]
        for f in (0, 1):
            for b, ds in zip((0, 1, 254, 255), rng.choice(live, (4, 40), replace=False)):
                ix.len_bytes[f, ds] = b
        self.deleted = deleted

    def date_cover(self, lo, hi):
        """``DateRange`` over the days lo .. hi and the number of tokens its cover has in this index."""
        q = DateRange("date", lo, hi)
        e = q.expand(self.ix.lexicon("date"))
        return q, len(e.subqueries) if isinstance(e, Or) else 1


# ---- query ladders -------------------------------------------------------------------------------------------------

LEAF_RUNGS = (8, 9, 31, 32, 33, 64, 65, 128, 200, 255, 256)
GROUP_RUNGS = (2, 8, 9, 16, 30, 31, 32)


def score_pool(c, m):
    """Posting lists of ScoreCorpus with live postings, both scorable fields, plus dense and book lists."""
    V = VOCAB
    pool = [t for t in list(range(3, 700)) + list(range(V + 3, V + 900)) if m.live_df[t] > 0]
    return pool


def leaf_ladder(c, m, seed=1):
    """Flat ORs with live leaf counts LEAF_RUNGS (mixed fields, a dense and a book list in each), 250 live leaves +
    6 dropped ones, ``And(word, Or(200))`` and ``And`` of 4 groups of 64 leaves."""
    rng = np.random.default_rng(seed)
    pool = score_pool(c, m)

    def leaves(n):
        ts = [c.dense[int(rng.integers(0, 4))], c.books[int(rng.integers(0, 12))]]
        ts += [int(t) for t in rng.choice([t for t in pool if t not in ts], n - 2, replace=False)]
        return [c.term(t, float(rng.uniform(0.25, 3.0))) for t in rng.permutation(ts)]
    qs = [Or(leaves(n)) for n in LEAF_RUNGS]
    dropped = [Term("body", "no-such-term-%d" % i) for i in range(4)] + [c.term(t) for t in c.all_deleted]
    mixed = leaves(250) + dropped
    qs.append(Or([mixed[int(i)] for i in rng.permutation(len(mixed))]))
    qs.append(And([c.term(c.dense[1], 1.3), Or(leaves(200))]))
    qs.append(And([Or(leaves(64)) for _ in range(4)]))
    return qs


LEAF_WANT = [(n, 1) for n in LEAF_RUNGS] + [(250, 1), (201, 2), (256, 4)]


def group_ladder(wc, multi):
    """ANDs with G groups: single body words (G leaves), or with ``multi`` three leaves a group (title and body of one
    common word and another body word)."""
    rng = np.random.default_rng(7 + multi)
    qs = []
    for G in GROUP_RUNGS:
        words = rng.permutation(N_COMMON)[:G]
        if multi:
            qs.append(And([Or([Term("title", cw(i), boost=1.5), Term("body", cw(i)),
                               Term("body", cw((i + 7) % N_COMMON), boost=float(rng.uniform(0.25, 3)))])
                           for i in words]))
        else:
            qs.append(And([Term("body", cw(i), boost=float(rng.uniform(0.25, 3))) for i in words]))
    return qs


def not_queries(wc):
    """``Not`` with 30 positive groups (31 leaves) and ``Not(DateRange)`` inside the 32-leaf limit."""
    rng = np.random.default_rng(9)
    words = rng.permutation(N_COMMON)
    nd, k = wc.date_cover(date(1962, 3, 12), date(1962, 6, 2))
    assert 20 <= k <= 30
    return [And([Term("body", cw(i), boost=float(rng.uniform(0.25, 3))) for i in words[:30]] + [Not(Term("body", "w7"))]),
            And([Term("body", cw(i)) for i in words[:20]] + [Not(Term("title", cw(3)))]),
            And([Term("body", cw(words[0])), Term("body", cw(words[1])), Not(nd)])]


def weight_queries(c, m):
    """Zero, negative, cancelling, all-negative and sub-bar weights, on narrow and wide shapes."""
    rng = np.random.default_rng(5)
    pool = score_pool(c, m)

    def mids(n):
        return [int(t) for t in rng.choice(pool, n, replace=False)]
    d0, d1, d2, d3 = c.dense
    bk = c.books[4]
    a, b = mids(2)
    return [
        c.term(d2, 0.0),                                                         # every match scores +0.0
        Or([c.term(d0, 0.0)] + [c.term(t, 1.0) for t in mids(3)]),               # zero among positives
        Or([c.term(t, 0.0 if i % 7 == 0 else 1.0) for i, t in enumerate(mids(60))]),
        Or([c.term(a, -1.5), c.term(b, 0.7), c.term(d1, 0.2)]),                  # a negative boost
        Or([c.term(t, float(rng.uniform(-2, 2))) for t in mids(120)]),
        Or([c.term(bk, 1.25), c.term(bk, -1.25), c.term(d3, 0.5)]),              # weight-only list: products cancel
        Or([c.term(d0, -1.0), c.term(d1, -0.5)]),                                # every match scores < 0
        Or([c.term(d2, 1e-31), c.term(a)]),                                      # 0 < w <= 1e-30: below the bar
        And([c.term(d0, -0.3), Or([c.term(t, float(rng.uniform(-1, 3))) for t in mids(40)])]),
    ]


def expansion_queries(wc):
    """Prefix / Wildcard at 32, 33, 255 and 256 live terms; DateRange covers of 40-90 tokens, alone and with words."""
    d1, n1 = wc.date_cover(date(1962, 5, 3), date(1968, 11, 28))
    d2, n2 = wc.date_cover(date(1961, 2, 9), date(1963, 3, 20))
    assert 40 <= n1 <= 90 and 40 <= n2 <= 90, (n1, n2)
    return [Prefix("body", "qa"), Wildcard("body", "qb?[0-9]", boost=2.0), Prefix("body", "qc", boost=0.5),
            Wildcard("body", "qd*"), Wildcard("body", "qc?[0-4]?"), d1, d2,
            And([Term("body", cw(3)), d1]), And([Term("body", cw(5)), Term("title", cw(6)), d2]),
            And([Prefix("body", "qa"), Term("body", cw(1))]), Or([Term("body", "w3"), Prefix("body", "qb", boost=0.75)])]


# ---- fixtures ------------------------------------------------------------------------------------------------------

class Setup:
    def __init__(self):
        self.c = c = ScoreCorpus()
        self.wc = wc = WideCorpus()
        w = BM25F(**WEIGHTING)
        self.m = Model(c.ix, w, fma=fma_exact)
        self.wm = Model(wc.ix, w, fma=fma_exact)
        self.leaf = leaf_ladder(c, self.m)
        self.weights = weight_queries(c, self.m)
        self.groups1 = group_ladder(wc, False)
        self.groupsm = group_ladder(wc, True)
        self.nots = not_queries(wc)
        self.exp = expansion_queries(wc)
        self._want = {}

    def want(self, name, b):
        """Model results of packed batch ``b``, cached by ``name``."""
        if name not in self._want:
            m = self.m if name.startswith("s:") else self.wm
            self._want[name] = m.batch(b)
        return self._want[name]

    def close(self):
        for ix in (self.c.ix, self.wc.ix):
            for eng in ix._engine_cache.values():
                eng.close()
            ix._engine_cache.clear()


@pytest.fixture(scope="module")
def su():
    s = Setup()
    yield s
    s.close()


def live_shape(m, b, q):
    """``(live positive leaves, groups)`` of query ``q`` of packed batch ``b`` after the planner's dropping rules."""
    o = b.query_leaf_offsets
    plan, _ = m.plan(b.leaf_term[o[q]:o[q + 1]], b.leaf_group[o[q]:o[q + 1]], int(b.query_n_groups[q]))
    return (-1 if plan is None else len(plan)), int(b.query_n_groups[q])


def cta_items(n_docs, tile_docs, split, m, b):
    """Work items per query the host planner cuts for the CTA kernels (``bm25f_prepare``) and the tile count T."""
    T = -(-n_docs // tile_docs)
    out = []
    for q in range(b.n_queries):
        o = b.query_leaf_offsets
        P = sum(int(m.live_df[t]) for t in b.leaf_term[o[q]:o[q + 1]] if t != TERM_UNKNOWN)   # lists hold live postings
        out.append(min(T, max(1, (P + split // 2) // split)))
    return T, out


DEFAULT_SPLIT = 1 << 16                 # bm25f_options.split_postings default (h->split)


# ---- CPU -------------------------------------------------------------------------------------------------------------

def test_fma_exact_equals_fma_f32():
    """``fma_exact`` is ``fma_f32`` (one rounding of the rational value) on the crafted double-rounding cases, on
    subnormals, and on 10^5 random triples of which most land on a float32 midpoint in float64."""
    e23 = np.float32(2.0 ** -23)
    one_up = np.float32(1) + e23
    u = np.float32(2.0 ** -24) * (np.float32(1) - e23)
    assert fma_exact(one_up, u, one_up)[0] == one_up
    assert fma_exact(-one_up, u, one_up)[0] == one_up
    assert fma_exact(3.0, 0.5, 1.0)[0] == np.float32(2.5)
    tiny = np.float32(2.0 ** -149)
    assert fma_exact(tiny, 0.5, tiny)[0] == np.float32(2.0 ** -148)
    assert fma_exact(2.0, 0.5, -1.0)[0] == 0.0 and not np.signbit(fma_exact(2.0, 0.5, -1.0)[0])
    rng = np.random.default_rng(11)
    n = 100_000
    # acc: normal and subnormal float32 of both signs; w * u = h * (1 +- i^2 2^-46) with h half an ulp of acc (times
    # a random power of two near 1), so that the float64 sum often is a float32 midpoint with a tiny nonzero error
    acc = (rng.uniform(1, 2, n) * 2.0 ** rng.integers(-140, 30, n)).astype(np.float32)
    acc[::3] = -acc[::3]
    acc[::11] = (rng.integers(1, 1 << 20, acc[::11].size) * 2.0 ** -149).astype(np.float32)     # subnormal
    ulp = np.abs(np.spacing(acc)).astype(np.float64)
    i = rng.integers(1, 33, n).astype(np.float64)
    wv = ((1 + i * 2.0 ** -23) * (ulp / 2) * 2.0 ** rng.integers(-1, 2, n)).astype(np.float32)
    uv = np.where(rng.random(n) < 0.5, 1 - i * 2.0 ** -23, 1 + i * 2.0 ** -23).astype(np.float32)
    wv[rng.random(n) < 0.5] *= -1
    plain = rng.random(n) < 0.2                   # and plain random products
    wv[plain] = rng.uniform(-40, 40, plain.sum()).astype(np.float32)
    uv[plain] = rng.uniform(0, 1, plain.sum()).astype(np.float32)
    got = fma_exact(wv, uv, acc)
    ref = fma_f32(wv, uv, acc)
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    p, a = wv.astype(np.float64) * uv.astype(np.float64), acc.astype(np.float64)
    s = p + a
    s32 = s.astype(np.float32)
    assert np.count_nonzero(s32 != got) > 2000          # a single float64 rounding would be wrong this often
    sub = np.abs(got) < np.finfo(np.float32).tiny
    assert np.count_nonzero(sub & (got != 0)) > 1000
    # a sample against the rational value directly
    for j in rng.choice(n, 300, replace=False):
        assert got[j] == round_f32(Fraction(float(wv[j])) * Fraction(float(uv[j])) + Fraction(float(acc[j])))


@pytest.fixture(scope="module")
def cpu():
    return Setup()


def test_ladders_hit_their_counts(cpu):
    """Every rung has its exact live leaf and group count after the planner drops unknown terms and empty lists;
    the group-count queries match more than 1024 documents; the expansion families give 32, 33, 255, 256 and 257
    terms (the last is refused by ``pack``)."""
    m, wm = cpu.m, cpu.wm
    s = engineless_searcher(cpu.c.ix, BM25F(**WEIGHTING))
    b = s.pack(cpu.leaf)
    assert [live_shape(m, b, q) for q in range(b.n_queries)] == LEAF_WANT
    o = b.query_leaf_offsets
    assert int(o[len(LEAF_RUNGS) + 1] - o[len(LEAF_RUNGS)]) == 256          # 250 live + 6 dropped inputs
    ws = engineless_searcher(cpu.wc.ix, BM25F(**WEIGHTING))
    for multi, qs in ((False, cpu.groups1), (True, cpu.groupsm)):
        b = ws.pack(qs)
        want = [(3 * G if multi else G, G) for G in GROUP_RUNGS]
        assert [live_shape(wm, b, q) for q in range(b.n_queries)] == want
        for q, (d, _) in enumerate(wm.batch(b)):
            assert d.size > 1024, "G=%d: %d matches" % (GROUP_RUNGS[q], d.size)
    b = ws.pack(cpu.nots)
    assert live_shape(wm, b, 0) == (30, 30) and int(b.query_leaf_offsets[1]) == 31
    assert all(int(b.query_leaf_offsets[q + 1] - b.query_leaf_offsets[q]) <= 32 for q in range(b.n_queries))
    assert all(wm.batch(b)[q][0].size > 256 for q in range(b.n_queries))
    lex = cpu.wc.ix.lexicon("body")
    sizes = {pre: len(expand_multiterms(Prefix("body", pre), lambda f: lex).subqueries) for pre in FAMILIES}
    assert sizes == {pre: nw for pre, (nw, _) in FAMILIES.items()}
    b = ws.pack(cpu.exp[:4])
    assert [live_shape(wm, b, q)[0] for q in range(4)] == [32, 33, 255, 256]
    assert b.query_leaf_offsets[2] - b.query_leaf_offsets[1] == 34            # lexicon count != live count
    with pytest.raises(UnsupportedQuery):
        ws.pack([Prefix("body", "qe")])


def test_weights_have_every_edge(cpu):
    """Zero weights, negative weights, a weight in (0, 1e-30], scores < 0, exact zeros and cancelling documents."""
    m = cpu.m
    s = engineless_searcher(cpu.c.ix, BM25F(**WEIGHTING))
    b = s.pack(cpu.weights)
    w = b.leaf_weight
    assert (w == 0).any() and (w < 0).any()
    sub = w[(w > 0) & (w <= BAR)]
    assert sub.size == 1 and 0 < sub[0] <= BAR
    want = m.batch(b)
    d, sc = want[0]
    assert d.size > 1000 and (sc.view(np.uint32) == 0).all() and np.array_equal(d, np.sort(d))
    assert (want[3][1] < 0).any() and (want[3][1] > 0).any()
    assert (want[6][1] < 0).all() and want[6][0].size > 1200
    # the cancelling pair: documents of the book that are not in the dense list score exactly +0.0
    d5, s5 = want[5]
    assert np.count_nonzero(s5.view(np.uint32) == 0) > 100 and (s5 > 0).any()
    for q in (4, 8):
        assert (want[q][1] < 0).any() and (want[q][1] > 0).any()


def test_multi_tile_geometry(cpu):
    """Under tile_docs 1024 and 256 (with small items) every CTA item of the wide ladders spans at least 3 tiles."""
    c, m = cpu.c, cpu.m
    b = engineless_searcher(c.ix, BM25F(**WEIGHTING)).pack(cpu.leaf)
    for tile, split in ((1024, DEFAULT_SPLIT), (256, 16384)):
        T, items = cta_items(c.ix.n_docs_all, tile, split, m, b)
        assert T // max(items) >= 3, (tile, split, T, items)
    T, items = cta_items(c.ix.n_docs_all, 256, 16384, m, b)
    assert max(items) >= 8                            # the small split cuts a wide query into many items


def test_model_is_bm25f_on_wide_shapes(cpu):
    """The model's matches are the oracle's; scores within 1e-5 relative or 1e-6 absolute (cancelling sums)."""
    w = BM25F(**WEIGHTING)
    for ix, m, qs in ((cpu.c.ix, cpu.m, cpu.leaf + cpu.weights),
                      (cpu.wc.ix, cpu.wm, cpu.groups1 + cpu.groupsm + cpu.nots + cpu.exp)):
        o = NumpyOracle(ix, B=0.75, K1=1.2, field_B={"title": 0.5})
        b = engineless_searcher(ix, w).pack(qs)
        for i, (q, (d, s)) in enumerate(zip(qs, m.batch(b))):
            od, osc = o.match_all(q)
            order = np.argsort(d, kind="stable")
            assert np.array_equal(d[order], od.astype(np.uint32)), "query %d" % i
            assert np.allclose(s[order], osc, rtol=1e-5, atol=1e-6), "query %d" % i


class LargestFirst(Model):
    """The model with the AND-groups in the opposite order (largest first), the caller's order inside a group."""

    def plan(self, terms, groups, n_groups):
        plan, neg = Model.plan(self, terms, groups, n_groups)
        if plan is None:
            return plan, neg
        order = list(dict.fromkeys(int(groups[i]) for i in plan))[::-1]
        return [i for g in order for i in plan if groups[i] == g], neg


def _changed(a, b):
    n = 0
    for (d1, s1), (d2, s2) in zip(a, b):
        assert np.array_equal(np.sort(d1), np.sort(d2))
        n += int(np.count_nonzero(s1[np.argsort(d1)] != s2[np.argsort(d2)]))
    return n


def test_corpora_discriminate(cpu):
    """Reversing the leaf order changes scores on many documents of the wide and many-group ladders, and so does
    ordering the groups largest-first: a kernel that walks leaves or groups in another order cannot pass."""
    w = BM25F(**WEIGHTING)
    b = engineless_searcher(cpu.c.ix, w).pack(cpu.leaf)
    assert _changed(cpu.m.batch(b), cpu.m.batch(b, reverse=True)) > 1000
    wb = engineless_searcher(cpu.wc.ix, w).pack(cpu.groups1 + cpu.groupsm)
    fwd = cpu.wm.batch(wb)
    assert _changed(fwd, cpu.wm.batch(wb, reverse=True)) > 1000
    assert _changed(fwd, LargestFirst(cpu.wc.ix, w, fma=fma_exact).batch(wb)) > 1000


# ---- GPU -----------------------------------------------------------------------------------------------------------

FAMS = [("auto", {}), ("host_plan", dict(host_plan=1)), ("pipe", dict(variant=1)), ("topk", dict(variant=2)),
        ("isect", dict(variant=5))]


def _run(s, b, k):
    out = s.search_packed(b, k)
    return out, s.engine.stats()


def same_rows(a, b, ctx):
    """The first ``len(a[2])`` queries of result tuples ``a`` and ``b`` are identical, scores bit for bit."""
    for i in range(len(a[2])):
        n = int(a[2][i])
        assert int(b[2][i]) == n and int(a[3][i]) == int(b[3][i]), "%s query %d" % (ctx, i)
        assert np.array_equal(a[0][i, :n].view(np.uint32), b[0][i, :n].view(np.uint32)), "%s query %d" % (ctx, i)
        assert np.array_equal(a[1][i, :n], b[1][i, :n]), "%s query %d" % (ctx, i)


def _served(st, cls):
    """Assert that the last batch's postings all went to kernel class ``cls``."""
    total = st["postings_touched"]
    got = {"cta": st["postings_cta"], "topk": st["postings_topk"], "lookup": st["postings_lookup"],
           "stream": st["postings_stream"], "team": st["postings_team"]}
    want = {"cta": total, "topk": total if cls == "topk" else 0}
    if cls in ("lookup", "stream", "team"):
        want = {"cta": 0, "topk": 0, cls: total}
    for n, v in want.items():
        assert got[n] == v, "%s: %s = %d, expected %d (%r)" % (cls, n, got[n], v, st)
    assert total > 0


@pytest.mark.gpu
@pytest.mark.parametrize("fam,opts", FAMS, ids=[f[0] for f in FAMS])
def test_leaf_ladder_exact(su, fam, opts):
    """Flat ORs of 8..256 live leaves, 250 live + 6 dropped, And(word, Or(200)), And of 4 x 64: every k and
    ``limit=None``; the rungs over 32 leaves on the CTA kernels (pipe, or topk when forced), the rest where the family
    routes them (isect when forced)."""
    c = su.c
    s = Searcher(c.ix, weighting=BM25F(**WEIGHTING), **opts)
    wide = s.pack(su.leaf[4:])                      # 33 leaves and more
    narrow = s.pack(su.leaf[1:4])                   # 9, 31 and 32 leaves
    ww, wn = su.want("s:wide", wide), su.want("s:narrow", narrow)
    for k in (1,) + K_ALL:
        out, st = _run(s, wide, k)
        assert_exact(ww, out, k, "%s wide k=%d" % (fam, k))
        _served(st, "topk" if fam == "topk" else "cta")
        out, st = _run(s, narrow, k)
        assert_exact(wn, out, k, "%s narrow k=%d" % (fam, k))
        if fam == "isect" and k <= 256:
            _served(st, "lookup")
        elif k > 256 or fam in ("pipe", "topk"):
            _served(st, "topk" if fam == "topk" else "cta")
    assert_results(ww, s.search_batch(su.leaf[4:], limit=None), None, "%s wide limit=None" % fam)
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam,opts", [("stream", dict(variant=3)), ("team", dict(variant=4))], ids=["stream", "team"])
def test_eight_leaf_rung_on_warp_kernels(su, fam, opts):
    """The 8-leaf OR and the 2- and 8-group ANDs on the warp stream / team kernels."""
    s = Searcher(su.c.ix, weighting=BM25F(**WEIGHTING), **opts)
    b = s.pack(su.leaf[:1])
    ws = Searcher(su.wc.ix, weighting=BM25F(**WEIGHTING), **opts)
    g = ws.pack(su.groups1[:2])
    for k in ((1, 10, 32) if fam == "team" else (1, 10, 32, 33, 256)):
        out, st = _run(s, b, k)
        assert_exact(su.want("s:eight", b), out, k, "%s or k=%d" % (fam, k))
        _served(st, fam)
        out, st = _run(ws, g, k)
        assert_exact(su.want("w:and8", g), out, k, "%s and k=%d" % (fam, k))
        _served(st, fam)
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam,opts", FAMS, ids=[f[0] for f in FAMS])
def test_group_ladder_exact(su, fam, opts):
    """ANDs of 2..32 groups: single words (32 groups = 32 leaves: k_score_isect under auto / variant 5 up to k = 256)
    and three-leaf groups (more than 32 leaves from 16 groups on: the CTA kernels), every k and ``limit=None``;
    ``Not`` with 30 groups and ``Not(DateRange)`` up to k = 256."""
    s = Searcher(su.wc.ix, weighting=BM25F(**WEIGHTING), **opts)
    one, multi, nots = s.pack(su.groups1), s.pack(su.groupsm), s.pack(su.nots)
    w1, wm_, wn = su.want("w:g1", one), su.want("w:gm", multi), su.want("w:not", nots)
    big = s.pack(su.groupsm[3:])                    # 48 leaves and more
    wb = su.want("w:gbig", big)
    for k in (1,) + K_ALL:
        out, st = _run(s, one, k)
        assert_exact(w1, out, k, "%s single-word groups k=%d" % (fam, k))
        if fam == "isect" and k <= 256:
            _served(st, "lookup")
        out, _ = _run(s, multi, k)
        assert_exact(wm_, out, k, "%s multi-leaf groups k=%d" % (fam, k))
        out, st = _run(s, big, k)
        assert_exact(wb, out, k, "%s > 32 leaves k=%d" % (fam, k))
        _served(st, "topk" if fam == "topk" else "cta")
        if k <= 256:
            out, st = _run(s, nots, k)
            assert_exact(wn, out, k, "%s not k=%d" % (fam, k))
            _served(st, "lookup")
    assert_results(w1 + wm_, s.search_batch(su.groups1 + su.groupsm, limit=None), None, "%s limit=None" % fam)
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam,opts", FAMS[:4], ids=[f[0] for f in FAMS[:4]])
def test_weights_exact(su, fam, opts):
    """Zero, negative, cancelling, all-negative and sub-bar weights: the batch runs on k_score_topk whatever the
    family; and the wide positive ladder gives the same bits alone (pipe) and next to one negative-weight query."""
    c = su.c
    s = Searcher(c.ix, weighting=BM25F(**WEIGHTING), **opts)
    b = s.pack(su.weights)
    want = su.want("s:weights", b)
    for k in (1,) + K_ALL:
        out, st = _run(s, b, k)
        assert_exact(want, out, k, "%s weights k=%d" % (fam, k))
        assert st["postings_topk"] == st["postings_cta"] > 0
    assert_results(want, s.search_batch(su.weights, limit=None), None, "%s weights limit=None" % fam)
    alone = s.pack(su.leaf[4:])
    mixed = s.pack(su.leaf[4:] + su.weights[3:4])
    ww = su.want("s:wide", alone)
    for k in (10, 256, 1024):
        a, st_a = _run(s, alone, k)
        _served(st_a, "topk" if fam == "topk" else "cta")
        m, st_m = _run(s, mixed, k)
        assert st_m["postings_topk"] == st_m["postings_cta"] > 0
        assert_exact(ww, a, k, "%s alone k=%d" % (fam, k))
        assert_exact(ww + su.want("s:neg1", s.pack(su.weights[3:4])), m, k, "%s mixed k=%d" % (fam, k))
        same_rows(a, m, "%s alone / mixed k=%d" % (fam, k))
    su.close()


@pytest.mark.gpu
def test_expansions_end_to_end(su):
    """Prefix / Wildcard at 32, 33, 255 and 256 terms and DateRange covers of 40-90 tokens, alone and in ``And``, through
    ``search_batch`` and ``search_page``, against the model on the same queries' packed batch."""
    s = Searcher(su.wc.ix, weighting=BM25F(**WEIGHTING))
    qs = su.exp
    want = su.want("w:exp", s.pack(qs))
    for limit in (1, 10, 33, 256, 257, 1024, None):
        assert_results(want, s.search_batch(qs, limit=limit), limit, "expansions limit=%s" % limit)
    nw = su.want("w:not", s.pack(su.nots))
    assert_results(nw, s.search_batch(su.nots, limit=256), 256, "not limit=256")
    for j in (2, 3, 5, 7):
        assert want[j][0].size > 1200
        hits = []
        for p in range(1, 9):
            hits += [(h.score, h.docnum) for h in s.search_page(qs[j], p, 150)]
        assert hits == s.search(qs[j], limit=1200).top_n, "query %d" % j
        assert_results([want[j]], [s.search(qs[j], limit=1200)], 1200, "query %d" % j)
    su.close()


GEOMETRY = [("tile1024", dict(tile_docs=1024)), ("tile256_split16384", dict(tile_docs=256, split_postings=16384)),
            ("pipe_chunk64", dict(tile_docs=1024, variant=1, chunk_postings=64, stages=2)),
            ("topk_tile256", dict(tile_docs=256, split_postings=16384, variant=2))]


@pytest.mark.gpu
@pytest.mark.parametrize("name,opts", GEOMETRY, ids=[g[0] for g in GEOMETRY])
def test_multi_tile_items_exact(su, name, opts):
    """Small tiles (every CTA item spans at least 3 tiles), small items, a shallow pipe ring: the wide ladder, the
    many-group ladder and the weights batch stay exact; the item count is the one the CPU part reasons about."""
    c = su.c
    s = Searcher(c.ix, weighting=BM25F(**WEIGHTING), **opts)
    wide = s.pack(su.leaf[4:])
    T, items = cta_items(c.ix.n_docs_all, opts["tile_docs"], opts.get("split_postings", DEFAULT_SPLIT), su.m, wide)
    assert T // max(items) >= 3
    for k in (10, 256, 1024):
        out, st = _run(s, wide, k)
        assert_exact(su.want("s:wide", wide), out, k, "%s wide k=%d" % (name, k))
        assert st["n_items"] == sum(items) and st["tile_docs"] == opts["tile_docs"]
        _served(st, "topk" if opts.get("variant") == 2 else "cta")
        b = s.pack(su.weights)
        out, st = _run(s, b, k)
        assert_exact(su.want("s:weights", b), out, k, "%s weights k=%d" % (name, k))
        assert st["postings_topk"] == st["postings_cta"] > 0
    ws = Searcher(su.wc.ix, weighting=BM25F(**WEIGHTING), **opts)
    big = ws.pack(su.groupsm[3:])
    for k in (33, 1024):
        out, _ = _run(ws, big, k)
        assert_exact(su.want("w:gbig", big), out, k, "%s groups k=%d" % (name, k))
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", [1, 2], ids=["pipe", "topk"])
@pytest.mark.parametrize("threads", [64, 96, 256, 512])
def test_threads_below_and_above_leaf_count(su, variant, threads):
    """CTAs of 64..512 threads on queries of more leaves than threads (65 and 256 leaves at 64 threads), on items that
    span many tiles: every leaf's boundary row is loaded on every tile (k_score_topk once loaded only the first
    ``threads`` leaves' rows past an item's second tile)."""
    c = su.c
    s = Searcher(c.ix, weighting=BM25F(**WEIGHTING), tile_docs=1024, threads=threads, variant=variant)
    wide = s.pack(su.leaf[4:])
    for k in (10, 1024):
        out, st = _run(s, wide, k)
        assert st["threads"] == threads
        assert_exact(su.want("s:wide", wide), out, k, "threads=%d k=%d" % (threads, k))
        _served(st, "topk" if variant == 2 else "cta")
    ws = Searcher(su.wc.ix, weighting=BM25F(**WEIGHTING), tile_docs=1024, threads=threads, variant=variant)
    big = ws.pack(su.groupsm[3:] + su.exp[2:4])
    out, _ = _run(ws, big, 1024)
    assert_exact(su.want("w:threads", big), out, 1024, "threads=%d groups" % threads)
    su.close()


@pytest.mark.gpu
def test_pages_across_hits_256_and_1024(su):
    """Pages of 10 and 150 across hits 256 and 1024 for a wide OR, a 32-group AND and an all-negative query (its
    paging bounds are keys of negative scores): concatenated pages equal ``search(q, limit=P * n)`` and the model."""
    s = Searcher(su.c.ix, weighting=BM25F(**WEIGHTING))
    ws = Searcher(su.wc.ix, weighting=BM25F(**WEIGHTING))
    cases = [(s, su.m, su.leaf[9]), (ws, su.wm, su.groups1[-1]), (s, su.m, su.weights[6])]
    for j, (srch, m, q) in enumerate(cases):
        wd, wsc = m.batch(srch.pack([q]))[0]
        assert wd.size > 1200
        for pagelen, P in ((10, 105), (150, 8)):
            hits = []
            for p in range(1, P + 1):
                page = srch.search_page(q, p, pagelen)
                assert page.total == wd.size and page.offset == (p - 1) * pagelen
                hits += [(h.score, h.docnum) for h in page]
            full = srch.search(q, limit=P * pagelen)
            assert hits == full.top_n, "query %d pagelen %d" % (j, pagelen)
            assert_results([(wd, wsc)], [full], P * pagelen, "query %d pagelen %d" % (j, pagelen))
    su.close()


@pytest.mark.gpu
def test_batches_split_for_the_boundary_table(su, monkeypatch):
    """With the per-call boundary table bounded so that 256 leaves fit one call, a 300-query batch of 40-256 leaves
    runs as several engine calls, through ``search_packed`` and between pipelined small batches in
    ``search_packed_stream``; the results equal the model and the unsplit run."""
    c, m = su.c, su.m
    rng = np.random.default_rng(17)
    pool = score_pool(c, m)
    qs = [Or([c.term(int(t), float(rng.uniform(0.25, 3))) for t in rng.choice(pool, int(rng.integers(40, 257)), replace=False)])
          for _ in range(300)]
    small = su.leaf[:2]
    s = Searcher(c.ix, weighting=BM25F(**WEIGHTING))
    b, sb = s.pack(qs), s.pack(small)
    want, wsmall = m.batch(b), su.want("s:small", sb)
    unsplit = s.search_packed(b, 100)
    assert_exact(want, unsplit, 100, "unsplit")
    calls, submits = [], []
    eng = s.engine
    real_search, real_submit = eng.search_batch, eng.submit
    monkeypatch.setattr(eng, "search_batch", lambda batch, k: calls.append(batch.n_queries) or real_search(batch, k))
    monkeypatch.setattr(eng, "submit", lambda batch, k: submits.append(batch.n_queries) or real_submit(batch, k))
    monkeypatch.setattr(searching, "BOUNDS_BYTES_PER_CALL", 1)
    split = s.search_packed(b, 100)
    assert len(calls) >= 100 and sum(calls) == 300 and max(calls) < 300
    assert_exact(want, split, 100, "split")
    same_rows(unsplit, split, "unsplit / split")
    calls.clear()
    outs = list(s.search_packed_stream([sb, b, sb, sb, b, sb], 100))
    assert submits == [2, 2, 2, 2] and sum(calls) == 600
    for i, o in enumerate(outs):
        assert_exact(want if i in (1, 4) else wsmall, o, 100, "stream batch %d" % i)
    su.close()


@pytest.mark.gpu
def test_device_planner_boundary(su):
    """300 queries of exactly 8 leaves in 8 groups are planned on the device (three more launches than the host
    planner); one 9-leaf query among them sends the batch to the host planner.  All bit-exact."""
    wc, wm = su.wc, su.wm
    rng = np.random.default_rng(23)
    qs = [And([Term("body", cw(int(i)), boost=float(rng.uniform(0.25, 3))) for i in rng.permutation(N_COMMON)[:8]])
          for _ in range(300)]
    nine = qs[:150] + [Or([Term("body", cw(i)) for i in range(9)])] + qs[150:]
    runs = {}
    for name, batch_qs in (("eight", qs), ("nine", nine)):
        for plan in ("device", "host"):
            s = Searcher(wc.ix, weighting=BM25F(**WEIGHTING), **({} if plan == "device" else dict(host_plan=1)))
            b = s.pack(batch_qs)
            assert max(live_shape(wm, b, q)[0] for q in range(b.n_queries)) == (8 if name == "eight" else 9)
            out, st = _run(s, b, 10)
            assert_exact(su.want("w:" + name, b), out, 10, "%s %s" % (name, plan))
            runs[name, plan] = st["n_launches"]
    assert runs["eight", "device"] >= runs["eight", "host"] + 3
    assert runs["nine", "device"] == runs["nine", "host"]
    su.close()


@pytest.mark.gpu
def test_refusals_then_exact(su):
    """257 leaves and 33 groups are refused by ``pack`` and, hand-built, by the engine; Not with 31 groups or beyond 32
    live leaves, a wide query under a final() weighting and a 33-leaf query on ``compact_store`` are refused with the
    library's messages.  After each refusal the engine serves an exact batch."""
    c, wc = su.c, su.wc
    w = BM25F(**WEIGHTING)
    s = Searcher(wc.ix, weighting=w)
    good = s.pack(su.groupsm)
    wgood = su.want("w:gm", good)

    def still_exact(ctx, srch=s, b=good, want=wgood, k=300):
        assert_exact(want, srch.search_packed(b, k), k, "after " + ctx)
    words = [Term("body", cw(i)) for i in range(33)]
    with pytest.raises(UnsupportedQuery):
        s.pack([And(words)])
    with pytest.raises(UnsupportedQuery):
        s.pack([Prefix("body", "qe")])
    with pytest.raises(UnsupportedQuery):
        s.pack([Or([Term("body", x) for x in wc.pattern_words["qe"]])])
    still_exact("pack refusals")
    terms = np.array([wc.ix.term_id("body", x) for x in wc.pattern_words["qe"]], np.uint32)
    hand = [PackedBatch([0, 257], [1], terms, np.ones(257), np.zeros(257)),
            PackedBatch([0, 33], [33], terms[:33], np.ones(33), np.arange(33))]
    for hb, msg in zip(hand, ("257 leaves", "33 groups")):
        with pytest.raises(EngineError, match=msg):
            s.search_packed(hb, 10)
        still_exact("hand-built " + msg)
    not31 = And(words[:31] + [Not(Term("body", "w7"))])
    not33 = And([Or(words[:32]), Term("body", cw(33 % N_COMMON)), Not(Term("body", "w7"))])
    for q in (not31, not33):
        with pytest.raises(EngineError, match="NOT clauses are served"):
            s.search_packed(s.pack([q]), 10)
        still_exact("not refusal")
    fs = Searcher(wc.ix, weighting=DescDateBM25F(**WEIGHTING))
    with pytest.raises(EngineError, match="at most 32 leaves"):
        fs.search_packed(fs.pack([Or(words)]), 10)
    still_exact("final() refusal")
    cs = Searcher(wc.ix, weighting=w, compact_store=1)
    small = cs.pack(su.groups1)
    wsmall = su.want("w:g1", small)
    still_exact("compact", cs, small, wsmall, 256)
    with pytest.raises(EngineError, match="compact_store"):
        cs.search_packed(cs.pack([Or(words)]), 10)
    still_exact("compact refusal", cs, small, wsmall, 256)
    su.close()
