"""Bit-exact scores on a length-normalised corpus: one float32 score per document, whichever kernel serves the query.

``tests/test_gpu_exact_order.py`` makes result order exact on a corpus where ``B = 0`` makes every impact a small
dyadic fraction, so every kernel's arithmetic lands on the same float32 by construction.  Here the corpus has what
makes BM25F BM25F - length bytes from 0 to 255, a different ``B`` per field, ``K1 = 1.2``, a non-scorable field, term
counts up to the packing limit - and the expected result is a host model of the engine's documented arithmetic,
evaluated without tolerance:

* impact ``u = fl32(tf / (tf + fl64(norm32[field][length byte])))`` in float64 (``k_impacts``), with the float32 norm
  tables of ``weighting.norm_tables(ix)``; ``u = fl32(tf)`` for a field that is not scorable (W15);
* leaf weight ``w``: the float32 the packed batch carries (``Searcher.pack``);
* score: ``acc = fmaf(w, u, acc)`` from 0, over the leaves that hold the document, in the plan's leaf order - NOT
  leaves first (they add nothing), then the AND groups by live size, smallest first (stable), the caller's order
  inside a group, leaves of empty lists dropped (``bm25f_prepare``, ``plan.cuh``).

Scores, docnums, match counts and totals must be equal bit for bit for every kernel family, limit, page, weighting
switch, store layout and shard count.  The CPU part checks that the corpus has every edge it is built for, that the
``fmaf`` emulation is exact, and that the corpus discriminates: on it, the two-rounding ``w * tf / (tf + norm)`` and a
reversed leaf order both change scores, so none of the GPU assertions can hold by accident.
"""
from fractions import Fraction

import numpy as np
import pytest

from document_search_engine_b200 import And, BM25F, FlatIndex, Not, Or, Term
from document_search_engine_b200.corpus import BODY, TITLE, make_corpus
from document_search_engine_b200.query import GROUP_NOT
from document_search_engine_b200.searching import Searcher
from oracle.numpy_oracle import NumpyOracle

TERM_UNKNOWN = 0xFFFFFFFF
TF_MAX = float(2 ** 24 - 1)           # the largest term count the packed payload holds
N_DOCS, VOCAB, N_BOOKS = 40_000, 20_000, 12
FIELDS = ("title", "body", "book")     # two scorable fields and one ID-like field (W15)
WEIGHTING = dict(K1=1.2, title_B=0.5)  # body keeps B = 0.75
LENGTH_BYTES = (0, 1, 254, 255)
#: top-k sizes on both sides of the one-key (32), four-key (128), warp-kernel (256) and CTA-kernel (1024) limits
K_ALL = (10, 32, 33, 128, 129, 256, 257, 1024)


# ---- exact float32 arithmetic on the host ------------------------------------------------------------------------

def round_f32(x: Fraction) -> np.float32:
    """The rational ``x`` rounded once to float32 (nearest, ties to even, subnormals included)."""
    if x == 0:
        return np.float32(0.0)
    sign, x = (-1, -x) if x < 0 else (1, x)
    e = x.numerator.bit_length() - x.denominator.bit_length()
    if x < Fraction(2) ** e:
        e -= 1                                               # now 2**e <= x < 2**(e + 1)
    q = max(e - 23, -149)                                    # exponent of the last significant bit
    m = round(x / Fraction(2) ** q)                          # Fraction.__round__: half to even
    return np.float32(sign * float(m) * 2.0 ** q)


def fma_f32(w, u, acc) -> np.ndarray:
    """Elementwise ``fmaf(w, u, acc)`` on float32 inputs: ``w * u + acc`` rounded once.  The product is exact in
    float64; where the float64 sum is not (two-sum error term != 0), rounding it again to float32 could differ from
    one rounding, so those elements are rounded from the exact rational value."""
    w, u, acc = (np.atleast_1d(np.asarray(x, dtype=np.float32)) for x in (w, u, acc))
    w, u, acc = np.broadcast_arrays(w, u, acc)
    p = w.astype(np.float64) * u.astype(np.float64)
    a = acc.astype(np.float64)
    s = p + a
    bv = s - p
    err = (p - (s - bv)) + (a - bv)
    out = s.astype(np.float32)
    for i in np.nonzero(err != 0)[0]:
        out[i] = round_f32(Fraction(float(p[i])) + Fraction(float(a[i])))
    return out


# ---- the corpus ---------------------------------------------------------------------------------------------------

def _with_book_field(base, rng):
    """``base`` (title, body) plus a non-scorable ``book`` field: every document in one of N_BOOKS books, weight 1
    (a few 2), no length."""
    n, V = base.n_docs_all, base.vocab_size
    book = rng.integers(0, N_BOOKS, n)
    order = np.argsort(book, kind="stable").astype(np.uint32)
    counts = np.bincount(book, minlength=V)
    offs = np.concatenate([base.term_offsets, base.term_offsets[-1] + np.cumsum(counts).astype(np.uint64)])
    tfs = np.ones(n, np.float32)
    tfs[rng.choice(n, 50, replace=False)] = 2.0
    return FlatIndex(field_names=list(FIELDS), n_docs_all=n, term_offsets=offs,
                     docids=np.concatenate([base.docids, order]), tfs=np.concatenate([base.tfs, tfs]),
                     term_field=np.concatenate([base.term_field, np.full(V, 2, np.uint8)]),
                     len_bytes=np.vstack([base.len_bytes, np.zeros((1, n), np.uint8)]),
                     field_length_total=np.concatenate([base.field_length_total, np.zeros(1, np.uint64)]),
                     vocab_size=V, scorable=[True, True, False])


class ScoreCorpus:
    """The corpus, its deliberately placed edges, and the term lists the queries are drawn from."""

    def __init__(self, seed=20261021):
        rng = np.random.default_rng(seed)
        self.ix = ix = _with_book_field(make_corpus(N_DOCS, VOCAB, seed, fields=(TITLE, BODY), device="cpu"), rng)
        V = VOCAB
        df = np.diff(ix.term_offsets).astype(np.int64)
        post = lambda t: ix.docids[int(ix.term_offsets[t]):int(ix.term_offsets[t + 1])]
        deleted = (rng.random(N_DOCS) < 0.2).astype(np.uint8)

        # -- lists whose live length is 31, 32 or 33, that lose their first or last posting, or every posting: title
        # lists with disjoint documents, so that placing one does not move another
        used = np.zeros(N_DOCS, bool)

        def pick(lo, hi, n):
            out = []
            for t in rng.permutation(np.nonzero((df[:V] >= lo) & (df[:V] <= hi))[0]):
                d = post(t)
                if not used[d].any():
                    used[d] = True
                    out.append(int(t))
                    if len(out) == n:
                        return out
            raise AssertionError("not enough disjoint title lists with %d..%d postings" % (lo, hi))

        self.live_target = {}
        for L, t in zip((31, 32, 33), pick(45, 120, 3)):
            d = post(t)
            keep = rng.choice(d.size, L, replace=False)
            deleted[d] = 1
            deleted[d[keep]] = 0
            self.live_target[t] = L
        self.lose_first, self.lose_last = pick(20, 200, 2)
        d = post(self.lose_first)
        deleted[d[0]], deleted[d[1]] = 1, 0
        d = post(self.lose_last)
        deleted[d[-1]], deleted[d[-2]] = 1, 0
        self.all_deleted = pick(2, 12, 2)
        for t in self.all_deleted:
            deleted[post(t)] = 1
        ix.deleted = deleted
        live = deleted == 0

        # -- short lists for single-term queries (df <= 256: limit 256 returns all of them), per scorable field
        self.short = {0: list(self.live_target) + [self.lose_first, self.lose_last]}
        self.short[0] += [int(t) for t in rng.choice(np.nonzero((df[:V] >= 40) & (df[:V] <= 250))[0], 8, replace=False)
                          if int(t) not in self.short[0]]
        self.short[1] = [V + int(t) for t in rng.choice(np.nonzero((df[V:2 * V] >= 40) & (df[V:2 * V] <= 250))[0], 10,
                                                        replace=False)]
        # length bytes 0, 1, 254 and 255 on live documents of those lists, in both scorable fields
        for f in (0, 1):
            docs = np.unique(np.concatenate([post(t) for t in self.short[f]]))
            docs = docs[live[docs]]
            chosen = rng.choice(docs, 4 * len(LENGTH_BYTES), replace=False).reshape(len(LENGTH_BYTES), -1)
            for b, ds in zip(LENGTH_BYTES, chosen):
                ix.len_bytes[f, ds] = b
        # term counts at the packing limit: in short lists and in long ones
        self.dense = [V + 0, V + 1, V + 2, 0]                 # body ranks 0-2, title rank 0: thousands of postings
        for t in self.short[0][3:7] + self.short[1][:4] + self.dense:
            a = int(ix.term_offsets[t])
            i = a + np.nonzero(live[post(t)])[0]
            ix.tfs[rng.choice(i, 1 if t not in self.dense else 5, replace=False)] = TF_MAX
        self.books = [2 * V + b for b in range(N_BOOKS)]

    def text(self, t):
        """``(field name, term text)`` of posting list ``t``."""
        return FIELDS[t // VOCAB], t % VOCAB

    def term(self, t, boost=1.0):
        f, x = self.text(t)
        return Term(f, x, boost=boost)


def unpacked_copy(ix, seed=3):
    """The same corpus with non-integral term counts and one above 2**24: the payload cannot be packed."""
    rng = np.random.default_rng(seed)
    tfs = ix.tfs.copy()
    i = rng.choice(tfs.size, tfs.size // 3, replace=False)
    tfs[i] = tfs[i] * np.float32(1.25) + np.float32(0.1)
    tfs[int(np.argmax(tfs))] = np.float32(2 ** 24 + 2)
    return FlatIndex(field_names=ix.field_names, n_docs_all=ix.n_docs_all, term_offsets=ix.term_offsets,
                     docids=ix.docids, tfs=tfs, term_field=ix.term_field, len_bytes=ix.len_bytes,
                     field_length_total=ix.field_length_total, vocab_size=ix.vocab_size, deleted=ix.deleted,
                     scorable=ix.scorable)


def multi_queries(c, n, seed, with_not=False, wide=False):
    """ORs (mixed fields, the non-scorable field, unknown terms), ANDs, AND-of-OR, single terms; with ``with_not``
    ``Not`` clauses; with ``wide`` ORs of 9..13 leaves (more than the warp kernels take).  Otherwise at most 8
    leaves a query, so that a batch of >= 256 of them is planned on the device."""
    rng = np.random.default_rng(seed)
    V = VOCAB
    mid = [int(t) for t in rng.integers(3, 400, 200)] + [V + int(t) for t in rng.integers(3, 600, 300)]
    short = c.short[0] + c.short[1] + c.all_deleted

    def b():
        return float(rng.uniform(0.25, 3.0))

    def leaves(pool, m):
        return [c.term(int(t), b()) for t in rng.choice(pool, m, replace=False)]

    out = []
    for i in range(n):
        kind = i % (9 if with_not else 7)
        if wide:
            q = Or(leaves(mid, int(rng.integers(6, 10))) + leaves(c.dense, 2) + leaves(short, int(rng.integers(1, 3))))
        elif kind == 0:
            q = Or(leaves(mid, int(rng.integers(1, 4))) + leaves(c.dense + c.books, 1) + leaves(short, int(rng.integers(0, 3))))
        elif kind == 1:                                      # one word in both fields, title boosted (config 5)
            r = int(rng.integers(0, 60))
            q = Or([Term("title", r, boost=2.0), Term("body", r)] + [Term("body", int(rng.integers(0, 60)), boost=b())])
        elif kind == 2:
            q = And(leaves(c.dense, 1) + leaves(mid, int(rng.integers(1, 3))))
        elif kind == 3:                                      # AND of OR groups
            q = And([Or(leaves(c.dense + mid[:20], 2)), Or(leaves(mid, int(rng.integers(2, 4)))),
                     c.term(int(rng.choice(c.books)), b())])
        elif kind == 4:
            q = c.term(int(rng.choice(mid + c.dense)), b())
        elif kind == 5:
            q = Or(leaves(short + mid, 3) + [Term("body", "no-such-term")])
        elif kind == 6:
            q = And(leaves(c.dense, 2) + leaves(short + mid, 1))
        elif kind == 7:
            q = And(leaves(c.dense, 2) + [Not(c.term(int(rng.choice(mid))))])
        else:
            q = Or(leaves(mid, 2) + leaves(c.dense, 1) + [Not(Or([c.term(int(t)) for t in rng.choice(mid, 2, replace=False)]))])
        out.append(q)
    return out


# ---- the host model ---------------------------------------------------------------------------------------------

def impacts(ix, norm):
    """float32 impact of every posting of ``ix`` under the float32 norm tables ``norm``, as ``k_impacts`` computes it."""
    field = np.repeat(ix.term_field, np.diff(ix.term_offsets).astype(np.int64))
    tf = ix.tfs.astype(np.float64)
    nv = norm[field, ix.len_bytes[field, ix.docids]].astype(np.float64)
    with np.errstate(divide="ignore"):                    # tf / (tf - 1) in the rows of weight-only fields
        u = (tf / (tf + nv)).astype(np.float32)
    weight_only = (norm == -1.0).all(axis=1)[field]
    u[weight_only] = ix.tfs[weight_only]
    return u


class Model:
    """Expected results of packed batches on ``ix`` under ``weighting``.  ``fma``: the ``fmaf`` emulation to use
    (``fma_f32``, or an equal one that is faster on long lists)."""

    def __init__(self, ix, weighting, fma=None):
        self.ix = ix
        self.fma = fma or fma_f32
        self.norm = weighting.norm_tables(ix)
        self.u = impacts(ix, self.norm)
        self.live = np.ones(ix.docids.size, bool) if ix.deleted is None else ix.deleted[ix.docids] == 0
        cs = np.concatenate([[0], np.cumsum(self.live, dtype=np.int64)])
        offs = ix.term_offsets.astype(np.int64)
        self.live_df = cs[offs[1:]] - cs[offs[:-1]]

    def postings(self, t):
        a, b = int(self.ix.term_offsets[t]), int(self.ix.term_offsets[t + 1])
        m = self.live[a:b]
        return self.ix.docids[a:b][m], self.u[a:b][m]

    def plan(self, terms, groups, n_groups):
        """Leaf indices in the plan's order (NOT leaves excluded) and the NOT leaves; None when a group is empty."""
        pos = [i for i in range(terms.size) if groups[i] != GROUP_NOT]
        gsize = np.zeros(n_groups, np.int64)
        for i in pos:
            if terms[i] != TERM_UNKNOWN:
                gsize[groups[i]] += self.live_df[terms[i]]
        if n_groups == 0 or (gsize == 0).any():
            return None, []
        order = np.argsort(gsize, kind="stable")
        plan = [i for g in order for i in pos if groups[i] == g and terms[i] != TERM_UNKNOWN and self.live_df[terms[i]] > 0]
        neg = [i for i in range(terms.size) if groups[i] == GROUP_NOT and terms[i] != TERM_UNKNOWN]
        return plan, neg

    def query(self, terms, weights, groups, n_groups, reverse=False):
        """``(docnums u32, scores f32)`` of every match in (score descending, docnum ascending) order."""
        plan, neg = self.plan(terms, groups, n_groups)
        if plan is None:
            return np.zeros(0, np.uint32), np.zeros(0, np.float32)
        n = self.ix.n_docs_all
        acc = np.zeros(n, np.float32)
        cnt = np.zeros(n, np.int32)
        last = np.full(n, -1, np.int32)
        for i in (plan[::-1] if reverse else plan):
            d, u = self.postings(terms[i])
            acc[d] = self.fma(weights[i], u, acc[d])
            first = last[d] != groups[i]                    # the document's first leaf of this group (a group's
            cnt[d[first]] += 1                              # leaves are contiguous in the plan)
            last[d] = groups[i]
        for i in neg:
            cnt[self.postings(terms[i])[0]] = -1
        docs = np.nonzero(cnt == n_groups)[0]
        sc = acc[docs]
        order = np.lexsort((docs, -sc.astype(np.float64)))
        return docs[order].astype(np.uint32), sc[order]

    def batch(self, b, reverse=False):
        o = b.query_leaf_offsets
        return [self.query(b.leaf_term[o[q]:o[q + 1]], b.leaf_weight[o[q]:o[q + 1]], b.leaf_group[o[q]:o[q + 1]],
                           int(b.query_n_groups[q]), reverse) for q in range(b.n_queries)]


def engineless_searcher(ix, weighting):
    """A ``Searcher`` without an engine: enough for ``pack`` on the CPU (the lowering and the leaf weights)."""
    s = Searcher.__new__(Searcher)
    s.ix = s.stats_ix = ix
    s.weighting = weighting
    s._term_w = None
    return s


# ---- comparison ----------------------------------------------------------------------------------------------------

def assert_rows(want, scores, docids, count, total, k, ctx):
    wd, ws = want
    n = wd.size if k is None else min(k, wd.size)
    assert int(total) == wd.size, "%s total %d != %d" % (ctx, int(total), wd.size)
    assert int(count) == n, "%s count %d != %d" % (ctx, int(count), n)
    gd = np.asarray(docids[:n], dtype=np.uint32)
    gs = np.asarray(scores[:n], dtype=np.float32)
    bad = np.nonzero((gd != wd[:n]) | (gs.view(np.uint32) != ws[:n].view(np.uint32)))[0]
    if bad.size:
        r = int(bad[0])
        raise AssertionError("%s rank %d of %d (%d ranks differ): doc %d score %r, expected doc %d score %r" % (
            ctx, r, n, bad.size, int(gd[r]), float(gs[r]), int(wd[r]), float(ws[r])))


def assert_exact(wants, out, k, ctx):
    scores, docids, counts, totals = out
    for i, w in enumerate(wants):
        assert_rows(w, scores[i], docids[i], counts[i], totals[i], k, "%s query %d:" % (ctx, i))


def assert_results(wants, results, k, ctx):
    for i, (w, r) in enumerate(zip(wants, results)):
        top = r.top_n
        assert_rows(w, [s for s, _ in top], [d for _, d in top], len(top), len(r), k, "%s query %d:" % (ctx, i))


# ---- CPU -------------------------------------------------------------------------------------------------------------

def test_fma_emulation_is_one_rounding():
    """Crafted cases where rounding the float64 sum to float32 is a double rounding that misses the true ``fmaf``,
    and random inputs against the exact rational rounding."""
    e23 = np.float32(2.0 ** -23)
    one_up = np.float32(1) + e23                               # odd last bit
    u = np.float32(2.0 ** -24) * (np.float32(1) - e23)        # one_up * u = 2**-24 - 2**-70: just below half an ulp
    # 1 + 2**-23 + (2**-24 - 2**-70): float64 rounds to the float32 midpoint, ties-to-even would round up
    assert np.float32(np.float64(one_up) + np.float64(one_up) * np.float64(u)) == np.float32(1 + 2.0 ** -22)
    assert fma_f32(one_up, u, one_up)[0] == one_up
    # the same from above: 1 + 2**-23 - (2**-24 - 2**-70) is just above the midpoint between 1 and 1 + 2**-23
    assert np.float32(np.float64(one_up) - np.float64(one_up) * np.float64(u)) == np.float32(1.0)
    assert fma_f32(-one_up, u, one_up)[0] == one_up
    # exact sums, subnormal results, cancellation to zero
    assert fma_f32(3.0, 0.5, 1.0)[0] == np.float32(2.5)
    tiny = np.float32(2.0 ** -149)
    assert fma_f32(tiny, 0.5, tiny)[0] == np.float32(2.0 ** -148)    # 1.5 * 2**-149: tie, to even
    assert fma_f32(2.0, 0.5, -1.0)[0] == 0.0
    rng = np.random.default_rng(1)
    n = 4000
    w = rng.uniform(0.1, 40, n).astype(np.float32)
    u = rng.uniform(0, 1, n).astype(np.float32)
    acc = (rng.uniform(0, 1, n) * 10.0 ** rng.integers(-3, 9, n)).astype(np.float32)
    acc[::7] = -acc[::7]
    got = fma_f32(w, u, acc)
    ref = np.array([round_f32(Fraction(float(a)) * Fraction(float(b)) + Fraction(float(c))) for a, b, c in zip(w, u, acc)])
    assert np.array_equal(got.view(np.uint32), ref.astype(np.float32).view(np.uint32))
    # the inputs reach the exact path (the float64 sum is inexact) often enough to mean something
    p, a = w.astype(np.float64) * u.astype(np.float64), acc.astype(np.float64)
    s = p + a
    assert np.count_nonzero((p - (s - (s - p))) + (a - (s - p)) != 0) > 100


@pytest.fixture(scope="module")
def corpus():
    return ScoreCorpus()


def test_round_f32_matches_numpy_on_float64():
    rng = np.random.default_rng(2)
    x = np.concatenate([rng.standard_normal(2000) * 10.0 ** rng.integers(-40, 37, 2000), [1e-45, 3e-45, 0.0]])
    assert np.array_equal(np.array([round_f32(Fraction(float(v))) for v in x], np.float32), x.astype(np.float32))


def test_corpus_has_every_edge(corpus):
    c = corpus
    ix = c.ix
    m = Model(ix, BM25F(**WEIGHTING))
    assert ix.scorable == [True, True, False] and (m.norm[2] == -1).all() and not (m.norm[:2] < 0).any()
    assert not np.array_equal(m.norm[0], m.norm[1])                    # a different B per scorable field
    assert 0.15 < ix.deleted.mean() < 0.25
    live_df = m.live_df
    assert sorted(live_df[list(c.live_target)].tolist()) == [31, 32, 33]
    assert all(live_df[t] == 0 and ix.df[t] > 0 for t in c.all_deleted)
    for t, i in ((c.lose_first, 0), (c.lose_last, -1)):
        a, b = int(ix.term_offsets[t]), int(ix.term_offsets[t + 1])
        assert not m.live[a:b][i] and m.live[a:b].sum() > 1
    for f in (0, 1):
        lbs, tfs = set(), set()
        for t in c.short[f]:
            assert 0 < live_df[t] <= 256 and ix.term_field[t] == f
            d, _ = m.postings(t)
            lbs |= set(ix.len_bytes[f, d].tolist())
            a, b = int(ix.term_offsets[t]), int(ix.term_offsets[t + 1])
            tfs |= set(ix.tfs[a:b][m.live[a:b]].tolist())
        assert set(LENGTH_BYTES) <= lbs, "field %d" % f
        assert {1.0, TF_MAX} <= tfs, "field %d" % f
    for t in c.dense:
        a, b = int(ix.term_offsets[t]), int(ix.term_offsets[t + 1])
        assert live_df[t] > 5000 and TF_MAX in ix.tfs[a:b][m.live[a:b]]
    assert all(ix.tfs == np.floor(ix.tfs)) and ix.tfs.min() >= 1 and ix.tfs.max() <= TF_MAX   # packable
    u = unpacked_copy(ix)
    assert (u.tfs != np.floor(u.tfs)).any() and u.tfs.max() >= 2 ** 24


def test_model_is_bm25f(corpus):
    """The model's matches are the oracle's, its scores within 1e-5 of the float64 BM25F."""
    c = corpus
    w = BM25F(**WEIGHTING)
    qs = multi_queries(c, 90, 5, with_not=True) + [c.term(t) for t in c.short[0] + c.short[1] + c.books[:2]]
    b = engineless_searcher(c.ix, w).pack(qs)
    o = NumpyOracle(c.ix, B=0.75, K1=1.2, field_B={"title": 0.5})
    for i, (q, (d, s)) in enumerate(zip(qs, Model(c.ix, w).batch(b))):
        od, osc = o.match_all(q)
        order = np.argsort(d, kind="stable")
        assert np.array_equal(d[order], od.astype(np.uint32)), "query %d" % i
        assert np.allclose(s[order], osc, rtol=1e-5, atol=0), "query %d" % i


def test_corpus_discriminates(corpus):
    """On this corpus the CTA kernels' former arithmetic (``fl32(w * tf) / fl32(tf + norm)``, no FMA) and a
    reversed leaf order both give other float32 scores than the model, so the bit-exact GPU checks mean something."""
    c = corpus
    ix = c.ix
    w = BM25F(**WEIGHTING)
    m = Model(ix, w)
    qs = multi_queries(c, 120, 6)
    b = engineless_searcher(ix, w).pack(qs)
    two_roundings = 0
    for t, wt in zip(b.leaf_term, b.leaf_weight):
        if t == TERM_UNKNOWN or ix.term_field[t] == 2:
            continue
        a, e = int(ix.term_offsets[t]), int(ix.term_offsets[t + 1])
        tf = ix.tfs[a:e]
        nv = m.norm[ix.term_field[t], ix.len_bytes[ix.term_field[t], ix.docids[a:e]]]
        old = (np.float32(wt) * tf) / (tf + nv)                  # float32 throughout: one rounding per operation
        new = (np.float64(wt) * m.u[a:e].astype(np.float64)).astype(np.float32)
        two_roundings += int(np.count_nonzero(old != new))
    assert two_roundings > 1000
    fwd, rev = m.batch(b), m.batch(b, reverse=True)
    reordered = 0
    for (d1, s1), (d2, s2) in zip(fwd, rev):
        assert np.array_equal(np.sort(d1), np.sort(d2))
        o1, o2 = np.argsort(d1), np.argsort(d2)
        reordered += int(np.count_nonzero(s1[o1] != s2[o2]))
    assert reordered > 100


# ---- GPU -----------------------------------------------------------------------------------------------------------

class Setup:
    def __init__(self):
        self.c = c = ScoreCorpus()
        self.ixs = {"packed": c.ix, "unpacked": unpacked_copy(c.ix)}
        self.models = {}
        self.big = multi_queries(c, 300, 11)                 # >= 256 queries of <= 8 leaves, no Not: device-planned
        self.wide = multi_queries(c, 24, 12, wide=True)
        self.nots = multi_queries(c, 45, 13, with_not=True)
        self.singles = [c.term(t, 1.5) for t in c.short[0] + c.short[1] + c.all_deleted]
        self.long = [c.term(t, 0.75) for t in c.dense + c.books[:2]]

    def model(self, name, weighting):
        key = (name,) + weighting.norm_key()
        if key not in self.models:
            self.models[key] = Model(self.ixs[name], weighting)
        return self.models[key]

    def close(self):
        for ix in self.ixs.values():
            for eng in ix._engine_cache.values():
                eng.close()
            ix._engine_cache.clear()


@pytest.fixture(scope="module")
def su():
    s = Setup()
    yield s
    s.close()


def _searcher(su, name, weighting=None, **opts):
    return Searcher(su.ixs[name], weighting=weighting or BM25F(**WEIGHTING), **opts)


FAMILIES = [("auto", {}), ("host_plan", dict(host_plan=1)), ("pipe", dict(variant=1)), ("cta", dict(variant=2)),
            ("stream", dict(variant=3)), ("team", dict(variant=4)), ("isect", dict(variant=5))]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["packed", "unpacked"])
@pytest.mark.parametrize("fam,opts", [FAMILIES[0], FAMILIES[2], FAMILIES[3]], ids=["auto", "pipe", "cta"])
def test_single_terms_exact(su, name, fam, opts):
    """(a) Every live posting of short lists (all length bytes, both scorable fields, live lengths 31-33, lists that
    lost their first, last or every posting) at limit 256; long lists at limits 10 to 1024 and ``limit=None``."""
    s = _searcher(su, name, **opts)
    assert s.engine.stats()["packed_payload"] == (1 if name == "packed" else 0)
    m = su.model(name, s.weighting)
    b = s.pack(su.singles)
    want = m.batch(b)
    assert_exact(want, s.search_packed(b, 256), 256, "%s %s short" % (name, fam))
    b = s.pack(su.long)
    want = m.batch(b)
    for k in (10, 33, 256, 300, 1024):
        assert_exact(want, s.search_packed(b, k), k, "%s %s long k=%d" % (name, fam, k))
    assert_results(want, s.search_batch(su.long, limit=None), None, "%s %s long limit=None" % (name, fam))
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fam,opts", FAMILIES, ids=[f[0] for f in FAMILIES])
def test_multi_leaf_every_family_exact(su, fam, opts):
    """(b) ORs, ANDs, AND-of-OR and NOT, every kernel family forced, for k around every kernel limit; the batch of
    >= 256 queries is device-planned under ``auto`` and host-planned under ``host_plan``."""
    s = _searcher(su, "packed", **opts)
    m = su.model("packed", s.weighting)
    big, wide, nots = s.pack(su.big), s.pack(su.wide), s.pack(su.nots)
    wb, ww, wn = m.batch(big), m.batch(wide), m.batch(nots)
    for k in K_ALL:
        assert_exact(wb, s.search_packed(big, k), k, "%s big k=%d" % (fam, k))
        assert_exact(ww, s.search_packed(wide, k), k, "%s wide k=%d" % (fam, k))
        if k <= 256:                                     # NOT clauses are served up to k = 256
            assert_exact(wn, s.search_packed(nots, k), k, "%s not k=%d" % (fam, k))
    su.close()


@pytest.mark.gpu
def test_multi_leaf_unpacked_exact(su):
    s = _searcher(su, "unpacked")
    m = su.model("unpacked", s.weighting)
    big = s.pack(su.big)
    want = m.batch(big)
    for k in (10, 129, 1024):
        assert_exact(want, s.search_packed(big, k), k, "unpacked big k=%d" % k)
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("pagelen", [10, 150])
def test_pages_split_one_ranking(su, pagelen):
    """(c) ``search_page`` pages 1..P, across hits 32, 256 and 1024, concatenated: ``search(q, limit=P * n)``, which
    is a prefix of ``limit=None`` (scores included) and the model's ranking."""
    c = su.c
    s = _searcher(su, "packed")
    m = su.model("packed", s.weighting)
    qs = [Or([c.term(c.dense[0], 0.7), c.term(c.dense[3], 1.3), c.term(VOCAB + 40, 2.0)]),
          And([c.term(c.dense[1]), Or([c.term(c.dense[2], 0.5), c.term(c.books[3], 0.9)])])]
    P = 105 if pagelen == 10 else 8
    for j, q in enumerate(qs):
        wd, ws = m.batch(s.pack([q]))[0]
        assert wd.size > 3000
        hits = []
        for p in range(1, P + 1):
            page = s.search_page(q, p, pagelen)
            assert page.total == wd.size and page.offset == (p - 1) * pagelen
            hits += [(h.score, h.docnum) for h in page]
        full = s.search(q, limit=P * pagelen)
        assert hits == full.top_n, "query %d" % j
        every = s.search(q, limit=None)
        assert every.top_n[:P * pagelen] == full.top_n, "query %d" % j
        assert_results([(wd, ws)], [every], None, "query %d limit=None" % j)
    su.close()


@pytest.mark.gpu
def test_reweighting_and_compact_store(su):
    """(d) One engine scores with BM25F(), BM25F(B=0.3, K1=2, title_B=0.9), BM25F() again: each equals its model,
    the third equals the first bit for bit.  ``compact_store=1`` under the same weighting equals the default store."""
    ix = su.ixs["packed"]
    runs = []
    engine = None
    for w in (BM25F(), BM25F(B=0.3, K1=2, title_B=0.9), BM25F()):
        s = Searcher(ix, weighting=w)
        assert engine is None or s.engine is engine
        engine = s.engine
        m = Model(ix, w)
        b = s.pack(su.big)
        want = m.batch(b)
        out = {}
        for k in (10, 256, 300):
            out[k] = s.search_packed(b, k)
            assert_exact(want, out[k], k, "%r k=%d" % (w.norm_key(), k))
        runs.append(out)
    for k in runs[0]:
        for a, b in zip(runs[0][k], runs[2][k]):
            assert np.array_equal(a, b)
    cs = Searcher(ix, weighting=BM25F(), compact_store=1)
    assert cs.engine is not engine
    b = cs.pack(su.big)
    for k in (10, 256):
        for a, b2 in zip(runs[0][k], cs.search_packed(b, k)):
            assert np.array_equal(a, b2)
    su.close()


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3, 8])
def test_shards_one_group_bit_equal(su, G):
    """(e) Terms and flat ORs (one group: the leaf order does not depend on the shard) on 2, 3 and 8 shards, merged by
    ``bm25f_merge_gathered``: the whole index's result bit for bit.  An AND's groups are ordered by their size on each
    shard, which may differ between shards, so multi-group queries keep the tolerance of the parity tests."""
    import torch
    from document_search_engine_b200.distributed import device_view
    ix = su.ixs["packed"]
    w = BM25F(**WEIGHTING)
    whole = Searcher(ix, weighting=w)
    qs = [q for q in su.big + su.singles + su.long if type(q).__name__ == "Term" or
          (type(q).__name__ == "Or" and all(type(x).__name__ == "Term" for x in q.subqueries))]
    assert len(qs) > 100
    want = su.model("packed", w).batch(whole.pack(qs))
    searchers = [Searcher(ix.shard(g, G), weighting=w, stats_ix=ix) for g in range(G)]
    batches = [s.pack(qs) for s in searchers]
    Q = len(qs)
    for k in (10, 33, 256, 1024):
        ref = whole.search_packed(whole.pack(qs), k)
        gathered = None
        for g, (s, b) in enumerate(zip(searchers, batches)):
            plan = s.engine.prepare(b, k, arena=True)
            plan.execute()
            base, span, tot_off = plan.gather_span()
            s.engine.synchronize()
            if gathered is None:
                gathered = torch.empty((G, span), dtype=torch.int64, device="cuda:0")
            gathered[g].copy_(device_view(base, span, 0))
            plan.close()
        torch.cuda.synchronize()
        keys = torch.empty(Q * k, dtype=torch.int64, device="cuda:0")
        scores = torch.empty(Q * k, dtype=torch.float32, device="cuda:0")
        docids = torch.empty(Q * k, dtype=torch.int32, device="cuda:0")
        counts = torch.empty(Q, dtype=torch.int32, device="cuda:0")
        totals = torch.empty(Q, dtype=torch.int64, device="cuda:0")
        searchers[0].engine.merge_gathered(gathered.data_ptr(), G, span, tot_off, Q, k, keys.data_ptr(),
                                           scores.data_ptr(), docids.data_ptr(), counts.data_ptr(), totals.data_ptr())
        searchers[0].engine.synchronize()
        out = (scores.cpu().numpy().reshape(Q, k), docids.cpu().numpy().view(np.uint32).reshape(Q, k),
               counts.cpu().numpy().view(np.uint32), totals.cpu().numpy().view(np.uint64))
        assert_exact(want, out, k, "G=%d k=%d" % (G, k))
        for i in range(Q):
            n = int(ref[2][i])
            assert np.array_equal(out[0][i, :n].view(np.uint32), ref[0][i, :n].view(np.uint32))
            assert np.array_equal(out[1][i, :n], ref[1][i, :n])
        assert np.array_equal(out[2], ref[2]) and np.array_equal(out[3], ref[3])
    for s in searchers:
        s.engine.close()
    su.close()
