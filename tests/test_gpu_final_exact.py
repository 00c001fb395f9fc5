"""Bit-exact date-ordered weightings: one float64 final value per match, ties inside a date, and the stream kernel's
date-block skip.

``DescDateBM25F`` / ``AscDateBM25F`` rank a match by its final value, computed on the device in float64
(``final_value`` in ``csrc/final.cuh``)::

    t = 1 - 1 / s               (s: the float32 score)
    v = t                       (no date)
    v = (t + add) / 1e9         (add = date seconds + 1.0, about 5.5e9 for a 20th-century date)

then by docnum.  Next to 5.5e9 the float64 spacing is 2**-20, so documents of one date whose float32 scores are
close get the identical ``v`` and their order is decided by docnum alone; computing ``t`` in float32, or multiplying
by ``1e-9`` instead of dividing, moves many of those values by a step.  The expected result here is a host model of
that arithmetic, compared without tolerance: the float32 scores of ``tests/test_gpu_score_exact.py`` (exact), then
the three float64 operations above in numpy, which performs the same IEEE operations (the library is built without
fast-math, float64 division is correctly rounded and ``final_value`` has no multiply-add to fuse), then the order of
the engine's 96-bit keys: ``orderable_f64(v)`` descending, docnum ascending.  (Whoosh computes the score itself in
float64; that separate deviation is what the parity tests' tolerance covers.)

The stored dates are laid out along the docnums for the stream kernel's skip of 32-document blocks whose largest date
term cannot reach the k-th best (``stream.cuh``, sub-range epilogue): session dates newest first, so the k-th best
fills early in a document range and later blocks are older; blocks without a date; a lone newer date at offset 0 or
31 of a block inside a run of older ones; dates near 1800 and 2200, whose values lie in [0, 1) and below 0 and so
mix with the values of undated documents.
"""
from datetime import datetime, timedelta

import numpy as np
import pytest

from document_search_engine_b200 import And, AscDateBM25F, BM25F, DescDateBM25F, Or, Phrase, Term
from document_search_engine_b200.searching import Searcher, orderable_f64
from oracle.numpy_oracle import NumpyOracle
from tests.test_date_final import FINAL_TOL
from tests.test_gpu_score_exact import (WEIGHTING, Model, ScoreCorpus, assert_exact, engineless_searcher,
                                        multi_queries)

CLASSES = (DescDateBM25F, AscDateBM25F)
#: top-k sizes on both sides of one, four and eight keys a lane, and of the k_merge_final<4> / <8> switch (k = 128)
K_FINAL = (1, 31, 32, 33, 128, 129, 256)

# ---- stored dates --------------------------------------------------------------------------------------------------

N_EARLY = 320                  # docnums [0, 320): 1810, then 1790 (Desc values in [0, 1), then below 0)
N_LATE = 320                   # [320, 640): 2190, then 2210 (Asc values in [0, 1), then below 0)
N_SESSIONS = 40                # [640, n): session dates, newest first, ~980 documents each:
SESSION_0 = datetime(1978, 6, 1, 14)   # 35 from 1978 down to 1965, 137 days apart,
#: then five from 1934 down to 1933: there (t + add) / 1e9 and (t + add) * 1e-9 can round two different sums to one
#: value or one sum to two, so the order differs (the quotient's binade is coarser than the spacing of t + add there,
#: in both orders)
SESSION_30S = datetime(1934, 6, 1, 9)
CHAPTERED, N_CHAPTERS = 0.25, 8   # share of headings with a chapter number, and its range 1 .. N_CHAPTERS
LONE_EVERY = 25                # every 25th block of the session part holds one newer date, at offset 0 or 31
UNDATED_BLOCK_EVERY = 37       # every 37th block of the session part has no dated document at all


def final_dates(ix, seed=17):
    """Attach stored fields (``date``, ``heading`` with an optional chapter number, which adds that many seconds) to
    ``ix`` as described in the module docstring; one document in eight without a date besides the undated blocks.
    Returns the docnums of the lone newer dates."""
    rng = np.random.default_rng(seed)
    n = ix.n_docs_all
    chapter = np.where(rng.random(n) < CHAPTERED, rng.integers(1, N_CHAPTERS + 1, n), 0)
    undated = rng.random(n) < 0.12
    lo_sess = N_LATE + N_EARLY
    per_session = -(-(n - lo_sess) // N_SESSIONS)
    when, session = [None] * n, np.zeros(n, np.int64)
    for i in range(n):
        if i < lo_sess:
            chapter[i] = 0
            when[i] = datetime((1810, 1790, 2190, 2210)[2 * i // N_EARLY], 1, 1)
        else:
            session[i] = (i - lo_sess) // per_session
            j = int(session[i])
            first = SESSION_0 if j < N_SESSIONS - 5 else SESSION_30S
            when[i] = first - timedelta(days=137 * (j % (N_SESSIONS - 5)), hours=j % 5)
    b_sess = lo_sess // 32
    for b in range(b_sess, n // 32):
        if b % UNDATED_BLOCK_EVERY == 5:
            undated[32 * b:32 * b + 32] = True
    lone = []
    for b in range(b_sess + 80, n // 32 - 1, LONE_EVERY):        # from session 2 on
        d = 32 * b + (0 if (b // LONE_EVERY) % 2 else 31)
        undated[d] = False
        when[d] = SESSION_0
        chapter[d] = N_CHAPTERS + 1 + (b // LONE_EVERY) % 9      # newer than every other document of session 0
        lone.append(d)
    stored = []
    for i in range(n):
        h = "Session %d%s" % (session[i], ", Chapter %d" % chapter[i] if chapter[i] else "")
        stored.append({"heading": h} if undated[i] else {"heading": h, "date": when[i]})
    ix.stored = stored
    return np.asarray(lone, dtype=np.int64)


def block_max(add):
    """The largest date term of every aligned block of 32 documents, -inf where it has none (``d_final_blk``), with
    the library's two trailing entries."""
    n = add.size
    blk = np.full(n // 32 + 2, -np.inf)
    a = np.where(np.isnan(add), -np.inf, add)
    m = (n // 32) * 32
    blk[:n // 32] = a[:m].reshape(-1, 32).max(axis=1)
    if n > m:
        blk[n // 32] = a[m:].max()
    return blk


# ---- the host model ------------------------------------------------------------------------------------------------

def final_values(s, add, f32_t=False, times=False):
    """float64 final values of float32 scores ``s`` with date terms ``add`` (NaN: no date).  ``f32_t``: ``1 - 1/s``
    in float32; ``times``: ``* 1e-9`` instead of ``/ 1e9`` (the two faults the corpus must expose)."""
    s = np.asarray(s, dtype=np.float32)
    if f32_t:
        t = (np.float32(1) - np.float32(1) / s).astype(np.float64)
    else:
        t = 1.0 - 1.0 / s.astype(np.float64)
    dated = ~np.isnan(add)
    v = t.copy()
    v[dated] = (t[dated] + add[dated]) * 1e-9 if times else (t[dated] + add[dated]) / 1e9
    return v


def ranked(d, v):
    """``(docnums u32, values f64)`` in the engine's order: orderable value descending, docnum ascending."""
    order = np.lexsort((d, ~orderable_f64(v)))
    return d[order].astype(np.uint32), v[order]


class FinalModel:
    """Expected results of packed batches under a date-ordered weighting."""

    def __init__(self, ix, weighting):
        self.scores = Model(ix, weighting)
        self.add = weighting.doc_final_terms(ix)

    def batch(self, b):
        """Per query ``(docnums, values, float32 scores)`` of every match, in ranking order."""
        out = []
        for d, s in self.scores.batch(b):
            rd, rv = ranked(d, final_values(s, self.add[d]))
            out.append((rd, rv, dict(zip(d.tolist(), s.tolist()))))
        return out


def assert_final_rows(want, vals, docids, count, total, k, ctx):
    wd, wv = want[0], want[1]
    n = wd.size if k is None else min(k, wd.size)
    assert int(total) == wd.size, "%s total %d != %d" % (ctx, int(total), wd.size)
    assert int(count) == n, "%s count %d != %d" % (ctx, int(count), n)
    gd = np.asarray(docids[:n], dtype=np.uint32)
    gv = np.asarray(vals[:n], dtype=np.float64)
    bad = np.nonzero((gd != wd[:n]) | (gv.view(np.uint64) != wv[:n].view(np.uint64)))[0]
    if bad.size:
        r = int(bad[0])
        raise AssertionError("%s rank %d of %d (%d ranks differ): doc %d value %r, expected doc %d value %r" % (
            ctx, r, n, bad.size, int(gd[r]), float(gv[r]), int(wd[r]), float(wv[r])))


def assert_final(wants, out, k, ctx):
    vals, docids, counts, totals = out
    for i, w in enumerate(wants):
        assert_final_rows(w, vals[i], docids[i], counts[i], totals[i], k, "%s query %d:" % (ctx, i))


def assert_final_results(wants, results, k, ctx):
    for i, (w, r) in enumerate(zip(wants, results)):
        top = r.top_n
        assert_final_rows(w, [v for v, _ in top], [d for _, d in top], len(top), len(r), k, "%s query %d:" % (ctx, i))


# ---- the emulated skip rule ----------------------------------------------------------------------------------------

def keys96(v, d):
    """The engine's 96-bit keys of values ``v`` and docnums ``d`` as Python ints (orderable value, ~docnum)."""
    return [(h << 32) | (0xFFFFFFFF - x) for h, x in zip(orderable_f64(np.asarray(v, np.float64)).tolist(),
                                                         np.asarray(d).tolist())]


def sweep_item(docs, vals, add, blk, lo, hi, sw, k, after=None, fault=None):
    """The keys ``k_score_stream<KR, true>`` keeps for the item ``[lo, hi)`` of one query whose matches are ``docs``
    (ascending) with final values ``vals``: sub-ranges of ``sw`` documents from ``lo``; in each one with a match,
    32-document chunks from the sub-range start, a chunk looked at when the k-th best is below 1, or when the largest
    date term of its block - or of the next block, for a chunk that does not start a block - reaches
    ``add_min = thr_v * 1e9 - 2``; a match of a chunk looked at gets a key when it has no date and the k-th best is
    below 1, or when its own date term reaches ``add_min``; the keys above the k-th best (and below the paging bound
    ``after``) are inserted in lane order.

    ``fault``: ``"margin"`` (``+ 2.0``), ``"second"`` (no check of the next block), ``"undated"`` (undated documents
    only while the k-th best is below 0)."""
    top = []                                                  # the item's keys, descending
    thr_key, thr_v, add_min = 0, -np.inf, -np.inf
    m = (docs >= lo) & (docs < hi)
    docs, vals = docs[m].tolist(), vals[m].tolist()
    adds = [float(add[d]) for d in docs]
    p = 0
    for sub_lo in range(lo, hi, sw):
        sub_hi = min(sub_lo + sw, hi)
        q = p
        while q < len(docs) and docs[q] < sub_hi:
            q += 1
        if q == p:
            continue
        n_it = (sub_hi - sub_lo + 31) // 32
        for c0 in range(0, n_it, 32):
            passing = []
            for it in range(c0, min(c0 + 32, n_it)):
                d0 = sub_lo + 32 * it
                ok = thr_v < 1.0 or blk[d0 >> 5] >= add_min
                if fault != "second":
                    ok = ok or ((d0 & 31) != 0 and blk[(d0 >> 5) + 1] >= add_min)
                if ok:
                    passing.append(d0)
            for d0 in passing:
                keys = []
                for i in range(p, q):
                    if d0 <= docs[i] < min(d0 + 32, sub_hi):
                        a = adds[i]
                        if np.isnan(a) and thr_v < (0.0 if fault == "undated" else 1.0) or not np.isnan(a) and a >= add_min:
                            keys.append(i)
                keys = [kk for kk, x in zip(keys96([vals[i] for i in keys], [docs[i] for i in keys]), keys)]
                for key in [x for x in keys if x > thr_key and (after is None or x < after)]:
                    if key > thr_key:
                        top.append(key)
                        top.sort(reverse=True)
                        del top[k:]
                        if len(top) == k:
                            thr_key = top[-1]
                            thr_v = _orderable_value(thr_key >> 32)
                            add_min = thr_v * 1e9 + (2.0 if fault == "margin" else -2.0)
        p = q
    return top


def _orderable_value(u):
    u = np.uint64(u)
    u = (u & np.uint64(0x7FFFFFFFFFFFFFFF)) if (u >> np.uint64(63)) else ~u
    return float(np.array([u], dtype=np.uint64).view(np.float64)[0])


def boosted(c, n, seed):
    """Flat ORs of two dense and two mid-frequency lists with boosts in the tens to hundreds: scores near 1000, where
    ``t`` moves by less than one step of the final value over hundreds of float32 steps of the score."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        b = (20.0, 100.0, 400.0)[i % 3]
        out.append(Or([c.term(int(t), b * float(rng.uniform(0.5, 1.5))) for t in rng.choice(c.dense, 2, replace=False)] +
                      [c.term(int(t), b * float(rng.uniform(0.5, 1.5))) for t in rng.integers(3, 400, 2)]))
    return out


# ---- the corpus ----------------------------------------------------------------------------------------------------

class FinalCorpus:
    def __init__(self):
        self.c = c = ScoreCorpus()
        self.ix = c.ix
        self.lone = final_dates(self.ix)
        self.qs = multi_queries(c, 70, 31) + [c.term(t, 1.5) for t in c.short[0][:6] + c.short[1][:6]] + boosted(c, 12, 34)
        self.nots = multi_queries(c, 36, 32, with_not=True)[7::9] + multi_queries(c, 36, 33, with_not=True)[8::9]
        self.one_group = [q for q in self.qs if type(q) is Term or
                          (type(q) is Or and all(type(x) is Term for x in q.subqueries))]
        self.models = {}

    def model(self, cls):
        if cls not in self.models:
            w = cls(**WEIGHTING)
            m = FinalModel(self.ix, w)
            b = engineless_searcher(self.ix, w)
            self.models[cls] = (m, m.batch(b.pack(self.qs)), m.batch(b.pack(self.nots)))
        return self.models[cls]

    def close(self):
        for eng in self.ix._engine_cache.values():
            eng.close()
        self.ix._engine_cache.clear()


@pytest.fixture(scope="module")
def fc():
    f = FinalCorpus()
    yield f
    f.close()


# ---- CPU -------------------------------------------------------------------------------------------------------------

def test_corpus_has_every_edge(fc):
    ix = fc.ix
    n = ix.n_docs_all
    desc, asc = DescDateBM25F().doc_final_terms(ix), AscDateBM25F().doc_final_terms(ix)
    undated = np.isnan(desc)
    assert 0.10 <= undated.mean() <= 0.20
    assert 0.15 < ix.deleted.mean() < 0.25
    # values in [0, 1) and below 0 for either order, next to undated documents
    for add, a, b in ((desc, 0, N_EARLY), (asc, N_EARLY, N_EARLY + N_LATE)):
        v = (1.0 - 1.0 / 3.0 + add[a:b]) / 1e9
        assert ((v >= 0) & (v < 1)).sum() > 100 and (v < 0).sum() > 100 and undated[a:b].mean() > 0.08
    # session dates shared by hundreds of documents, with chapter seconds
    sess = N_LATE + N_EARLY
    days = np.floor((desc[sess:] - 1.0) / 86400)
    _, cnt = np.unique(days[~np.isnan(days)], return_counts=True)
    assert cnt.size >= N_SESSIONS and np.sort(cnt)[-N_SESSIONS:].min() > 500
    sec = (desc[sess:] - 1.0) % 86400
    assert np.unique(sec[~np.isnan(sec)] % 3600).size > N_CHAPTERS
    # newest first along the docnums of the session part, apart from the lone newer dates
    a = desc[sess:].copy()
    a[fc.lone - sess] = np.nan
    days = np.floor((a - 1.0) / 86400)
    days = days[~np.isnan(days)]
    assert (np.diff(days) <= 0).all()
    # blocks without a dated document; a lone newer date at offset 0 or 31 after a long run of older blocks
    blk = block_max(desc)
    b_sess = sess // 32
    assert np.isinf(blk[b_sess:n // 32]).sum() >= 25
    offs = set()
    for d in fc.lone:
        b = d // 32
        assert blk[b] == desc[d] and np.max(np.where(np.isnan(desc[32 * b:32 * b + 32]), -np.inf,
                                                      desc[32 * b:32 * b + 32])) == desc[d]
        assert (blk[b - 20:b] < desc[d] - 86400).all() and blk[b + 1] < desc[d] - 86400
        offs.add(int(d % 32))
    assert offs == {0, 31} and fc.lone.size >= 40


def test_model_is_the_oracle(fc):
    """The model's matches are ``NumpyOracle(final_add=...)``'s and its values the oracle's up to the float32 score:
    that deviates from the float64 one by a relative 1e-5 at most (``test_gpu_score_exact.py``), which moves
    ``1 - 1/s`` by up to 1e-5 / s - the whole difference for an undated document, a billionth of it (plus
    ``FINAL_TOL``, a few steps of the final value) for a dated one."""
    for cls in CLASSES:
        add = cls().doc_final_terms(fc.ix)
        o = NumpyOracle(fc.ix, B=0.75, K1=1.2, field_B={"title": 0.5}, final_add=add)
        _, want, want_not = fc.model(cls)
        for i, (q, w) in enumerate(zip(fc.qs + fc.nots, want + want_not)):
            od, ov = o.match_all(q)
            order = np.argsort(w[0], kind="stable")
            assert np.array_equal(w[0][order], od.astype(np.uint32)), "%s query %d" % (cls.__name__, i)
            wd, wv = w[0][order], w[1][order]
            dated = ~np.isnan(add[wd])
            s = np.array([w[2][x] for x in wd.tolist()], dtype=np.float64)
            tol = np.where(dated, FINAL_TOL + 1e-14 / s, 1e-5 / s + 1e-12)
            assert (np.abs(wv - ov) <= tol).all(), "%s query %d" % (cls.__name__, i)


def collisions(want, top=256):
    """Pairs of neighbouring ranks among the first ``top`` with the identical final value and different float32
    scores."""
    d, v, sc = want
    d, v = d[:top], v[:top]
    same = np.nonzero(v[1:] == v[:-1])[0]
    return sum(1 for r in same if sc[int(d[r])] != sc[int(d[r + 1])])


def test_corpus_discriminates(fc):
    """On the expected results, ties of the final value among different scores are common, and both a float32
    ``1 - 1/s`` and ``* 1e-9`` change values and the order; dates one and two seconds apart sit on either side of
    the k-th best."""
    for cls in CLASSES:
        m, want, _ = fc.model(cls)
        assert sum(collisions(w) for w in want) >= 200, cls.__name__
        for fault in ("f32_t", "times"):
            moved = reordered = 0
            for d, v, sc in want:
                s = np.array([sc[x] for x in d.tolist()], dtype=np.float32)
                v2 = final_values(s, m.add[d], **{fault: True})
                moved += int(np.count_nonzero(v2[:256] != v[:256]))
                reordered += int(not np.array_equal(ranked(d, v2)[0], d))
            assert moved >= 500 and reordered >= 1, (cls.__name__, fault, moved, reordered)
    _, want, _ = fc.model(DescDateBM25F)
    add = fc.models[DescDateBM25F][0].add
    gaps = set()
    for d, v, _ in want:
        for k in K_FINAL:
            if d.size > k and not np.isnan(add[d[k - 1]]) and not np.isnan(add[d[k]]):
                gaps.add(float(add[d[k - 1]] - add[d[k]]))
    assert {0.0, 1.0, 2.0} <= gaps


#: document ranges as the planner cuts a query into stream-kernel items: [n * s / S, n * (s + 1) / S)
EMULATED_SPLITS = (1, 7, 39)


def test_skip_rule_emulation_is_decisive(fc):
    """An emulation of the stream kernel's sweep (``sweep_item``) over items of this corpus's queries under
    ``DescDateBM25F``, at k = 1, 33 and 256 and for the passes of a ``limit=None`` listing (k = 256 below the last key
    of the previous pass): the correct rule keeps each item's top-k, and each of three faults of the skip - margin
    ``+ 2.0``, no check of the next block for a chunk that does not start a block, undated documents only while the
    k-th best is below 0 - drops a document of the query's expected result.  Without a GPU this is the only evidence
    that the GPU tests reach the skip: they run these queries and passes on the stream kernel with 128-document
    sub-ranges (flat ORs; 64 for ANDs) and items this small."""
    m, want, _ = fc.model(DescDateBM25F)
    add = m.add
    blk = block_max(add)
    n = fc.ix.n_docs_all
    b = engineless_searcher(fc.ix, DescDateBM25F(**WEIGHTING)).pack(fc.qs)
    found = {f: None for f in ("margin", "second", "undated")}
    checked = 0
    for i, (d, v, _) in enumerate(want):
        if d.size == 0:
            continue
        sw = 128 if int(b.query_n_groups[i]) == 1 else 64
        order = np.argsort(d, kind="stable")
        da, va = d[order], v[order]
        keys_da = np.array(keys96(va, da), dtype=object)
        keys_all = sorted(keys_da.tolist(), reverse=True)
        cases = [(k, None, set(keys_all[:k])) for k in (1, 33, 256)]
        cases += [(256, keys_all[p - 1], set(keys_all[p:p + 256])) for p in range(256, len(keys_all), 256)][:6]
        for k, after, expected in cases:
            for S in EMULATED_SPLITS:
                for s in range(S):
                    lo, hi = n * s // S, n * (s + 1) // S
                    mine = [x for x in keys_da[(da >= lo) & (da < hi)].tolist() if after is None or x < after]
                    if not mine:
                        continue
                    true_top = sorted(mine, reverse=True)[:k]
                    if checked < 60 and S > 1:
                        assert sweep_item(da, va, add, blk, lo, hi, sw, k, after) == true_top, (i, k, S, s)
                        checked += 1
                    for f in found:
                        if found[f] is None and set(true_top) & expected:
                            got = set(sweep_item(da, va, add, blk, lo, hi, sw, k, after, fault=f))
                            if (set(true_top) & expected) - got:
                                found[f] = (i, k, after is not None, S, s)
        if checked >= 60 and all(found.values()):
            break
    assert checked >= 60
    assert all(found.values()), found


# ---- GPU -----------------------------------------------------------------------------------------------------------

#: the kernels a final() step runs on: auto, the stream kernel, the team kernel (which hands a final() query to the
#: stream kernel), the candidate-driven kernel; then the same with small items: 128-document sub-ranges, stream items
#: of ~1k postings and candidate-driven items of 128 candidates, cut at docnums n * s / S that are not multiples of 32
ROUTES = [("auto", {}), ("stream", dict(variant=3)), ("team", dict(variant=4)), ("isect", dict(variant=5)),
          ("stream_small", dict(variant=3, subtile_docs=128, warp_split=1024)),
          ("isect_small", dict(variant=5, isect_split=128)),
          ("auto_small", dict(subtile_docs=128, warp_split=1024, isect_split=128))]


@pytest.mark.gpu
@pytest.mark.parametrize("cls", CLASSES, ids=lambda c: c.__name__)
@pytest.mark.parametrize("route,opts", ROUTES, ids=[r[0] for r in ROUTES])
def test_final_values_bit_exact(fc, route, opts, cls):
    """ORs, ANDs, AND-of-OR, single terms, boosted ORs and ``Not`` clauses at every k: final values, docnums, counts
    and totals equal the model's bit for bit."""
    _, want, want_not = fc.model(cls)
    s = Searcher(fc.ix, weighting=cls(**WEIGHTING), **opts)
    b, bn = s.pack(fc.qs), s.pack(fc.nots)
    for k in K_FINAL:
        assert_final(want, s.search_packed(b, k), k, "%s %s k=%d" % (route, cls.__name__, k))
        assert_final(want_not, s.search_packed(bn, k), k, "%s %s not k=%d" % (route, cls.__name__, k))
    fc.close()


def deep_queries(fc, cls):
    """Indices of queries whose listing has more than 700 matches, a final value shared by different float32 scores
    across a boundary of pages of 10 or 150, and negative final values."""
    _, want, _ = fc.model(cls)
    out = []
    for i, (d, v, sc) in enumerate(want):
        if d.size < 700 or not (v < 0).any():
            continue
        tie = [r for r in range(10, d.size, 10) if v[r - 1] == v[r] and sc[int(d[r - 1])] != sc[int(d[r])]]
        if tie:
            out.append((i, tie))
    return sorted(out, key=lambda x: want[x[0]][0].size)


@pytest.mark.gpu
@pytest.mark.parametrize("cls", CLASSES, ids=lambda c: c.__name__)
@pytest.mark.parametrize("route,opts", [ROUTES[0], ROUTES[4]], ids=["auto", "stream_small"])
def test_final_limits_and_pages(fc, route, opts, cls):
    """``limit`` 257, 700 and ``None`` take further passes below the last key returned; ``search_page`` pages of 10
    and 150 hits with boundaries inside classes of one final value and among negative values."""
    _, want, _ = fc.model(cls)
    deep = deep_queries(fc, cls)
    assert len(deep) >= 4
    s = Searcher(fc.ix, weighting=cls(**WEIGHTING), **opts)
    idx = [i for i, _ in deep[:8]] + [i for i, w in enumerate(want) if 0 < w[0].size < 300][:4]
    qs = [fc.qs[i] for i in idx]
    for limit in (257, 700, None):
        assert_final_results([want[i] for i in idx], s.search_batch(qs, limit=limit), limit,
                             "%s %s limit=%s" % (route, cls.__name__, limit))
    for i, ties in deep[:4]:
        d, v, _ = want[i]
        neg = int(np.argmax(v < 0))
        for pagelen in (10, 150):
            pages = {ties[0] // pagelen, ties[-1] // pagelen, neg // pagelen + 1, d.size // pagelen}
            for p in sorted(pages):
                page = s.search_page(fc.qs[i], p, pagelen)
                lo = (p - 1) * pagelen
                assert page.total == d.size and page.offset == lo
                got = [h.score for h in page], [h.docnum for h in page]
                assert_final_rows((d[lo:lo + pagelen], v[lo:lo + pagelen]), got[0], got[1], len(got[1]),
                                  d[lo:lo + pagelen].size, None, "%s query %d page %d of %d" % (cls.__name__, i, p, pagelen))
    fc.close()


@pytest.mark.gpu
def test_weighting_switches_and_compact_store(fc):
    """One engine: BM25F, DescDateBM25F, AscDateBM25F, BM25F again - each equals its model bit for bit; then the same
    under ``compact_store=1``."""
    ix = fc.ix
    for opts in ({}, dict(compact_store=1)):
        engine = None
        for cls in (BM25F, DescDateBM25F, AscDateBM25F, BM25F):
            s = Searcher(ix, weighting=cls(**WEIGHTING), **opts)
            assert engine is None or s.engine is engine
            engine = s.engine
            b = s.pack(fc.qs)
            for k in (1, 33, 256):
                out = s.search_packed(b, k)
                if cls is BM25F:
                    assert_exact(Model(ix, s.weighting).batch(b), out, k, "%r BM25F k=%d" % (opts, k))
                else:
                    assert_final(fc.model(cls)[1], out, k, "%r %s k=%d" % (opts, cls.__name__, k))
    fc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3, 8])
def test_shards_merge_final_lists(fc, G):
    """Terms and flat ORs (one group: one leaf order on every shard) on 2, 3 and 8 document shards, each shard's
    (final value, docnum) lists merged by ``bm25f_merge_final_lists``: the whole index's result bit for bit."""
    import torch
    from document_search_engine_b200.distributed import device_view
    idx = [i for i, q in enumerate(fc.qs) if any(q is x for x in fc.one_group)]
    qs = [fc.qs[i] for i in idx]
    Q = len(qs)
    for cls in CLASSES:
        want = [fc.model(cls)[1][i] for i in idx]
        w = cls(**WEIGHTING)
        searchers = [Searcher(fc.ix.shard(g, G), weighting=w, stats_ix=fc.ix) for g in range(G)]
        for k in (1, 33, 129, 256):
            vals = torch.empty(G * Q * k, dtype=torch.float64, device="cuda:0")
            docs = torch.empty(G * Q * k, dtype=torch.int32, device="cuda:0")
            totals = np.zeros(Q, dtype=np.uint64)
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
            eng.merge_final_lists(vals.data_ptr(), docs.data_ptr(), G, Q, k, out_v.data_ptr(), out_d.data_ptr(),
                                  out_c.data_ptr())
            eng.synchronize()
            out = (out_v.cpu().numpy().reshape(Q, k), out_d.cpu().numpy().view(np.uint32).reshape(Q, k),
                   out_c.cpu().numpy().view(np.uint32), totals)
            assert_final(want, out, k, "G=%d %s k=%d" % (G, cls.__name__, k))
        for s in searchers:
            s.engine.close()


@pytest.mark.gpu
def test_refusals_leave_the_engine_serving(fc):
    """Under a final() step the device refuses more than 32 leaves, a zero or negative boost and k > 256 (and
    ``search_packed`` refuses limit > 256); after each refusal the engine serves the next batch exactly."""
    c = fc.c
    _, want, _ = fc.model(DescDateBM25F)
    s = Searcher(fc.ix, weighting=DescDateBM25F(**WEIGHTING))
    good = s.pack(fc.qs[:20])
    mids = [int(t) for t in np.random.default_rng(3).choice(np.arange(3, 400), 33, replace=False)]
    bad = [[Or([c.term(t) for t in mids])], [Or([c.term(mids[0]), c.term(mids[1], 0.0)])],
           [And([c.term(mids[0]), c.term(mids[1], -1.0)])]]
    for qs in bad:
        with pytest.raises(Exception):
            s.search_packed(s.pack(fc.qs[:3] + qs), 10)
        assert_final(want[:20], s.search_packed(good, 33), 33, "after %r" % (qs,))
    with pytest.raises(NotImplementedError):
        s.search_packed(good, 257)
    with s.engine.lock:
        with pytest.raises(Exception):
            s.engine.search_batch_final(good, 257)
    assert_final(want[:20], s.search_packed(good, 256), 256, "after k=257")
    fc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("cls", CLASSES, ids=lambda c: c.__name__)
def test_phrase_final(cls):
    """A phrase query and an AND with a phrase (a per-batch document list with a tiny weight among the leaves): the
    date-ordered listing is the final step applied, in numpy, to the engine's own BM25F scores of the same queries."""
    from tests.test_gpu_phrases import mc_corpus
    ix = mc_corpus()
    final_dates(ix, seed=5)
    qs = [Phrase("body", [5, 6], slop=40), And([Term("title", 4), Phrase("body", [7, 5], slop=20)]),
          Phrase("body", [3, 8, 3], slop=5)]
    plain = Searcher(ix, weighting=BM25F())
    ref = plain.search_batch(qs, limit=None)
    add = cls().doc_final_terms(ix)
    s = Searcher(ix, weighting=cls())
    for limit in (33, None):
        got = s.search_batch(qs, limit=limit)
        for i, r in enumerate(ref):
            d = np.array([x for _, x in r.top_n], dtype=np.int64)
            sc = np.array([x for x, _ in r.top_n], dtype=np.float32)
            assert d.size > 50, "query %d" % i
            wd, wv = ranked(d, final_values(sc, add[d]))
            top = got[i].top_n
            assert_final_rows((wd, wv), [v for v, _ in top], [x for _, x in top], len(top), len(got[i]), limit,
                              "%s phrase query %d limit=%s" % (cls.__name__, i, limit))
    for eng in ix._engine_cache.values():
        eng.close()
    ix._engine_cache.clear()
