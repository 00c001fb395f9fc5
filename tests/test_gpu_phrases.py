"""Phrase queries with the positional filter on the device (bm25f_put_positions / bm25f_phrase_lists; reference
search-form.html:20-40, Whoosh query.Phrase).

Every document set and match count must equal ``FlatIndex.phrase_docs`` (the CPU reference) minus the deleted
documents, exactly; scores are the oracle's within the parity tolerance, and bit for bit the same whichever kernel,
limit or page serves the query (the filter leaf's fmaf(1e-29, 1, acc) is part of the same leaf-order chain in every
kernel).  The CPU part restates the kernel's chunked scan in Python and checks it against the reference on crafted
word sequences, and checks the word order ``make_corpus(positions=True)`` keeps."""
import random

import numpy as np
import pytest

from document_search_engine_b200 import And, BM25F, DescDateBM25F, FlatIndex, Not, Phrase, Prefix, Term
from document_search_engine_b200 import _ffi
from document_search_engine_b200.corpus import BODY, TITLE, make_corpus, make_queries
from oracle.numpy_oracle import NumpyOracle
from tests.parity import assert_batch_parity, assert_query_parity

WORDS = ["w%d" % i for i in range(12)]
FILL = "fill"


def crafted_docs():
    """Bodies of 0, 1, 31, 32, 33, 64 and 4096 tokens, with phrases at the first and last position, across 32-token
    boundaries, repeated words, and words further apart than the chunk."""
    f = lambda n: [FILL] * n
    big = f(4096)
    big[4094:4096] = ["w1", "w2"]
    big[1000:1008] = ["w%d" % i for i in range(1, 9)]                            # the 8-word phrase, adjacent
    big[2000:2015] = ["w1", FILL, "w2", FILL, FILL, "w3", FILL, "w4", FILL, FILL, "w5", "w6", "w7", FILL, "w8"]
    big[100], big[135] = "w4", "w5"                                                  # 35 apart: slop 40 only
    big[3000], big[3001] = "w3", "w3"
    return [
        [], ["w1"], f(29) + ["w1", "w2"], ["w1", "w2"] + f(30), f(31) + ["w1", "w2"],
        f(31) + ["w3", "w3"] + f(29) + ["w1", "w2"],                                  # 64: straddle, and at the end
        big,
        f(30) + ["w4"] + f(2) + ["w5"],                                               # w4 at 30, w5 at 33: a carry
        f(31) + ["w1", "w1", "w1"] + f(3),
        ["w4", FILL, "w5"],                                                           # slop 40 > the document
        ["w3"] + f(40), f(63) + ["w3"],                                               # one w3: no "w3 w3"
    ]


def small_corpus(n=20000, seed=11):
    """A 12-word vocabulary: adjacent pairs are frequent ("w1 w2" matches thousands of documents)."""
    rng = random.Random(seed)
    docs = []
    for i in range(n):
        docs.append({"body": [rng.choice(WORDS) for _ in range(rng.randrange(0, 70))],
                     "title": [rng.choice(WORDS + ["solo"]) for _ in range(rng.randrange(0, 5))],
                     "tags": ["t%02d" % rng.randrange(60) for _ in range(rng.randrange(0, 3))],
                     "book": "b%d" % (i % 7)})
    docs += [{"body": b, "title": ["w1"], "book": "b0"} for b in crafted_docs()]
    deleted = sorted(rng.sample(range(n), n // 10))
    return FlatIndex.from_documents(docs, ["body", "title", "tags", "book"], id_fields=["book"], deleted=deleted)


def small_phrases():
    P = Phrase
    eight = ["w%d" % i for i in range(1, 9)]
    return [P("body", ["w1", "w2"]), P("body", ["w3", "w3"]), P("body", ["w1", "w1", "w1"]), P("body", ["w1", "w2", "w3"]),
            P("body", ["w4", "w5"], slop=2), P("body", ["w4", "w5"], slop=5), P("body", ["w4", "w5"], slop=40),
            P("body", ["w6", "w7", "w8"], slop=2, boost=2.0), P("body", eight), P("body", eight, slop=5),
            P("body", ["w2", "w1"], slop=0), P("body", ["w1", "nope"]), P("body", ["w1", "solo"]),
            P("title", ["w1", "w2"]), P("nofield", ["a", "b"]), P("body", ["w5", FILL, "w4"], slop=3)]


def live(ix, docs):
    docs = np.asarray(docs, dtype=np.int64)
    return docs if ix.deleted is None else docs[ix.deleted[docs] == 0]


def want_docs(ix, p):
    """The CPU reference: global docnums that pass the positional test, deleted documents removed."""
    return (live(ix, ix.phrase_docs(p.fieldname, p.words, p.slop)) + ix.doc_base).tolist()


def bits(top):
    """(score bits, docnum) pairs: equality is bit equality."""
    return [(np.float32(s).view(np.uint32).item(), d) for s, d in top]


@pytest.fixture(scope="module")
def small():
    return small_corpus()


def mc_corpus(n=6000, vocab=400, seed=20261107):
    ix = make_corpus(n, vocab, seed, (TITLE, BODY), device="cpu", positions=True)
    ix.deleted = (np.random.default_rng(seed).random(n) < 0.2).astype(np.uint8)
    return ix


@pytest.fixture(scope="module")
def mc():
    return mc_corpus()


def cut_phrases(ix, n, seed, field="body", skip_top=5):
    """Phrases cut from real adjacent tokens (2 or 3 words, slop 1, 2, 5 or 40), some at a document's first or last
    position."""
    rng = np.random.default_rng(seed)
    f = ix.field_index(field)
    offs, ids = ix.positions[f]
    V = ix.vocab_size
    out = []
    while len(out) < n:
        d = int(rng.integers(ix.n_docs_all))
        a, b = int(offs[d]), int(offs[d + 1])
        w = int(rng.integers(2, 4))
        if b - a < w:
            continue
        kind = len(out) % 3
        p = a if kind == 0 else (b - w if kind == 1 else int(rng.integers(a, b - w + 1)))
        ranks = (ids[p:p + w] - f * V).tolist()
        if min(ranks) < skip_top:
            continue
        out.append(Phrase(field, ranks, slop=(1, 2, 5, 40)[len(out) % 4]))
    return out


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def chunked_scan(seq, words, slop, chunk=32):
    """The kernel's scan (csrc/phrase.cuh), restated: chunks of `chunk` tokens; per word an exclusive max-scan of the
    previous word's kept positions in the chunk, else its carry from the earlier chunks."""
    n = len(words)
    carry = [-1] * n
    for c0 in range(0, len(seq), chunk):
        toks = seq[c0:c0 + chunk]
        kept = [c0 + i for i, t in enumerate(toks) if t == words[0]]
        for j in range(1, n):
            cprev = carry[j - 1]
            nxt = []
            if kept or (cprev >= 0 and c0 - cprev <= slop):
                for i, t in enumerate(toks):
                    p = c0 + i
                    lower = [e for e in kept if e < p]
                    prev = max(lower) if lower else cprev
                    if t == words[j] and prev >= 0 and p - prev <= slop:
                        nxt.append(p)
            if kept:
                carry[j - 1] = max(kept)
            kept = nxt
        if kept:
            return True
    return False


def test_chunked_scan_equals_the_reference():
    rng = random.Random(3)
    docs = crafted_docs() + [[rng.choice(WORDS[:4]) for _ in range(rng.randrange(0, 90))] for _ in range(300)]
    ix = FlatIndex.from_documents([{"body": d} for d in docs], ["body"])
    cases = [(p.words, p.slop) for p in small_phrases() if p.fieldname == "body" and "nope" not in p.words and "solo" not in p.words]
    cases += [(["w0", "w1"], s) for s in (0, 1, 2, 3, 33, 10 ** 6)] + [(["w2", "w2", "w2"], s) for s in (1, 2, 31)]
    cases += [(["w0", "w1", "w0", "w3"], 4), (["w3", "w3"], 1)]
    matched = 0
    for words, slop in cases:
        want = set(ix.phrase_docs("body", words, slop).tolist())
        for chunk in (32, 4, 1):
            got = {d for d, seq in enumerate(docs) if chunked_scan(seq, words, slop, chunk)}
            assert got == want, (words, slop, chunk)
        matched += len(want)
    assert matched > 300
    # the crafted documents are where the edges are: every one of these matches only there
    for words, slop, doc in [(["w1", "w2"], 1, 2), (["w1", "w2"], 1, 3), (["w1", "w2"], 1, 4), (["w3", "w3"], 1, 5),
                             (["w4", "w5"], 3, 7), (["w1", "w1", "w1"], 1, 8), (["w4", "w5"], 40, 9)]:
        assert doc in ix.phrase_docs("body", words, slop).tolist()
    assert 10 not in ix.phrase_docs("body", ["w3", "w3"], 1).tolist() and 11 not in ix.phrase_docs("body", ["w3", "w3"], 100).tolist()


def test_make_corpus_keeps_the_word_order():
    plain = make_corpus(3000, 300, 77, (TITLE, BODY), device="cpu")
    ix = make_corpus(3000, 300, 77, (TITLE, BODY), device="cpu", positions=True)
    assert plain.positions == {}
    for name in ("term_offsets", "docids", "tfs", "term_field", "len_bytes", "field_length_total", "df"):
        assert getattr(plain, name).tobytes() == getattr(ix, name).tobytes(), name
    from document_search_engine_b200.numeric import lengths_to_bytes
    V = ix.vocab_size
    for f in range(2):
        offs, ids = ix.positions[f]
        lengths = np.diff(offs)
        assert offs[0] == 0 and int(offs[-1]) == ids.size == int(ix.field_length_total[f])
        assert np.array_equal(lengths_to_bytes(lengths), ix.len_bytes[f])
        assert ids.min() >= f * V and ids.max() < (f + 1) * V
        # every document's word multiset is its postings: (term, doc) -> tf
        doc_of = np.repeat(np.arange(ix.n_docs_all), lengths)
        key = ids.astype(np.int64) * ix.n_docs_all + doc_of
        uk, cnt = np.unique(key, return_counts=True)
        a, b = int(ix.term_offsets[f * V]), int(ix.term_offsets[(f + 1) * V])
        tids = np.repeat(np.arange(f * V, (f + 1) * V), np.diff(ix.term_offsets[f * V:(f + 1) * V + 1].astype(np.int64)))
        pk = tids * ix.n_docs_all + ix.docids[a:b].astype(np.int64)
        assert np.array_equal(uk, pk) and np.array_equal(cnt.astype(np.float32), ix.tfs[a:b])


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def check_sets(ix, s, phrases):
    """search(limit=None) and one batch: the document sets and totals are the reference's exactly."""
    o = NumpyOracle(ix)
    batch = s.search_batch(phrases, limit=None)
    for p, rb in zip(phrases, batch):
        want = want_docs(ix, p) if ix.field_index(p.fieldname) >= 0 else []
        r = s.search(p, limit=None)
        assert len(r) == len(want) and sorted(d for _, d in r.top_n) == want, p
        assert bits(rb.top_n) == bits(r.top_n) and len(rb) == len(r), p
        assert_query_parity(o, p, r.top_n, len(r), None, ctx=repr(p))
    return [len(r) for r in batch]


@pytest.mark.gpu
def test_filter_equals_the_reference(small, mc):
    with small.searcher() as s:
        sizes = check_sets(small, s, small_phrases())
    assert max(sizes) > 2000 and sizes.count(0) >= 4
    assert all(n > 0 for n, p in zip(sizes, small_phrases()) if p.words[0] in ("w4", "w6") or len(p.words) == 8)
    with mc.searcher() as s:
        sizes = check_sets(mc, s, cut_phrases(mc, 60, 1) + cut_phrases(mc, 12, 2, field="title", skip_top=0))
    assert sum(n > 0 for n in sizes) > 60                             # (a phrase cut from a deleted document may be gone)


@pytest.mark.gpu
def test_every_limit_and_page(small):
    o = NumpyOracle(small)
    qs = [Phrase("body", ["w1", "w2"]), And([Term("body", "w0"), Phrase("body", ["w3", "w4"], slop=2)]),
          Phrase("body", ["w4", "w5"], slop=40), Phrase("body", ["w2", "w3", "w2"], slop=5)]
    with small.searcher() as s:
        for q in qs:
            full = s.search(q, limit=None)
            assert len(full) > 300, q
            assert_query_parity(o, q, full.top_n, len(full), None, ctx=repr(q))
            for limit in (10, 150, 256, 257, 300, 1024, 2000):
                r = s.search(q, limit=limit)
                assert len(r) == len(full) and bits(r.top_n) == bits(full.top_n[:limit]), (q, limit)
            pages = []
            for p in (1, 2, 3):
                pg = s.search_page(q, p, 150)
                assert pg.total == len(full)
                pages += [(h.score, h.docnum) for h in pg]
            assert bits(pages) == bits(s.search(q, limit=450).top_n)
            pages = []
            for p in range(24, 29):                                          # hits 231 .. 280: across hit 256
                pages += [(h.score, h.docnum) for h in s.search_page(q, p, 10)]
            assert bits(pages) == bits(s.search(q, limit=280).top_n[230:])


@pytest.mark.gpu
def test_every_kernel_variant_agrees(small):
    qs = small_phrases() + [And([Term("body", "w0"), Phrase("body", ["w1", "w2"])]),
                            And([Phrase("body", ["w1", "w2"]), Phrase("body", ["w2", "w1"], boost=3.0)])]
    ref = None
    for variant in range(6):
        with small.searcher(variant=variant) as s:
            got = [[bits(r.top_n) + [len(r)] for r in s.search_batch(qs, limit=limit)] for limit in (10, 300, None)]
        if ref is None:
            ref = got
        assert got == ref, variant
    small._engine_cache.clear()


@pytest.mark.gpu
def test_more_than_32_leaves(small):
    o = NumpyOracle(small)
    qs = [And([Phrase("body", ["w1", "w2"]), Prefix("tags", "t")]), And([Prefix("tags", "t0"), Phrase("body", ["w3", "w3"])])]
    with small.searcher() as s:
        for limit in (10, 300, None):
            res = s.search_batch(qs, limit=limit)
            assert_batch_parity(o, qs, res, limit)
        assert len(res[0]) > 100


@pytest.mark.gpu
def test_date_ordered_weighting():
    from tests.test_date_final import FINAL_TOL, dated_corpus
    ix = dated_corpus(mc_corpus(seed=7))
    w = DescDateBM25F()
    o = NumpyOracle(ix, final_add=w.doc_final_terms(ix))
    qs = cut_phrases(ix, 20, 3)
    big = Phrase("body", [0, 1], slop=40)
    qs.append(big)
    with ix.searcher(weighting=DescDateBM25F) as s:
        for limit in (10, 256, 300, None):
            res = s.search_batch(qs, limit=limit)
            assert_batch_parity(o, qs, res, limit, abs_tol=FINAL_TOL)
            if limit is None:
                for q, r in zip(qs, res):
                    assert sorted(d for _, d in r.top_n) == want_docs(ix, q), q
        assert len(s.search(big, limit=None)) > 300
        pages = []
        for p in range(25, 29):
            pages += [(h.score, h.docnum) for h in s.search_page(big, p, 10)]
        assert pages == s.search(big, limit=280).top_n[240:]


@pytest.mark.gpu
def test_batches_and_limits(mc, small):
    o = NumpyOracle(mc)
    phrases = cut_phrases(mc, 320, 4)
    qs = phrases + make_queries(100, mc.vocab_size, 5, 2, 3, "mixed", skip_top=5).queries
    with mc.searcher(filter_postings=1 << 22) as s:
        res = s.search_batch(qs, limit=10)
        assert_batch_parity(o, qs, res, 10)
        for p, r in zip(phrases, res):
            assert len(r) == len(want_docs(mc, p))
    # a filter_postings overflow is refused loudly, and the engine serves the next batch
    with small.searcher(filter_postings=64) as s:
        with pytest.raises(RuntimeError, match="filter_postings"):
            s.search(Phrase("body", ["w1", "w2"]))
        few = [p for p in small_phrases() if 0 < len(want_docs(small, p)) <= 16][:3]       # one batch: <= 48 postings
        assert few
        check_sets(small, s, few)
    # more than BM25F_MAX_FILTER_LISTS distinct phrases in one batch are refused, as before
    many = [Phrase("body", [a, b], slop=sl) for a in WORDS for b in WORDS for sl in range(1, 30)][:4097]
    with small.searcher() as s:
        with pytest.raises(RuntimeError, match="4096"):
            s.search_batch(many, limit=10)
        adjacent = [p for p in many if p.slop == 1][:100]
        assert_batch_parity(NumpyOracle(small), adjacent, s.search_batch(adjacent, limit=10), 10)
    small._engine_cache.clear()


@pytest.mark.gpu
def test_compact_store_serves_phrases(small):
    qs = small_phrases()
    with small.searcher() as s:
        want = [[bits(r.top_n) + [len(r)] for r in s.search_batch(qs, limit=limit)] for limit in (10, 256)]
    with small.searcher(compact_store=1) as s:
        got = [[bits(r.top_n) + [len(r)] for r in s.search_batch(qs, limit=limit)] for limit in (10, 256)]
    assert got == want
    small._engine_cache.clear()


@pytest.mark.gpu
def test_positions_upload_once(small):
    small._engine_cache.clear()
    with small.searcher() as s:
        b0 = s.engine.stats()["device_bytes"]
        s.search(And([Term("body", "w1"), Term("body", "w2")]))
        assert s.engine.stats()["device_bytes"] == b0
        s.search(Phrase("body", ["w1", "w2"]))
        offs, ids = small.positions[0]
        b1 = b0 + offs.nbytes + ids.nbytes
        assert s.engine.stats()["device_bytes"] == b1
        s.search_batch([Phrase("body", ["w3", "w4"]), Phrase("body", ["w5", "w6"], slop=3)], limit=300)
        assert s.engine.stats()["device_bytes"] == b1
        s.search(Phrase("title", ["w1", "w2"]))
        offs, ids = small.positions[1]
        assert s.engine.stats()["device_bytes"] == b1 + offs.nbytes + ids.nbytes
        # a field flattened without word order (the ID field) keeps refusing phrases
        with pytest.raises(NotImplementedError, match="without positions"):
            s.search(Phrase("book", ["b1", "b2"]))
        # the C ABI refuses what it cannot serve
        eng = s.engine
        t = lambda f, w: small.term_id(f, w)
        with pytest.raises(_ffi.EngineError, match="different fields"):
            eng.phrase_lists([[t("body", "w1"), t("title", "w2")]], [1])
        with pytest.raises(_ffi.EngineError, match="no word order"):
            eng.phrase_lists([[t("tags", "t01"), t("tags", "t02")]], [1])
        with pytest.raises(_ffi.EngineError, match="at most 32"):
            eng.phrase_lists([[t("body", "w1")] * 33], [1])
        assert eng.phrase_lists([[t("body", "w1")] * 32, [_ffi.TERM_UNKNOWN, t("body", "w1")]], [1, 1]) > 0
        o = np.zeros(small.n_docs_all + 1, dtype=np.uint64)
        assert eng.lib.bm25f_put_positions(eng._h, 99, _ffi._ptr(o), None) == -1
        o[0] = 1
        assert eng.lib.bm25f_put_positions(eng._h, 0, _ffi._ptr(o), None) == -1
        o[0], o[5] = 0, 7
        assert eng.lib.bm25f_put_positions(eng._h, 0, _ffi._ptr(o), None) == -1
        assert s.engine.stats()["device_bytes"] == b1 + offs.nbytes + ids.nbytes
        check_sets(small, s, small_phrases()[:4])                            # the refusals left the engine as it was
    small._engine_cache.clear()


@pytest.mark.gpu
@pytest.mark.parametrize("n_shards", [2, 3])
def test_shards_cover_the_whole_index(small, n_shards):
    from document_search_engine_b200.searching import Searcher
    qs = small_phrases()[:10]
    got = [[] for _ in qs]
    for g in range(n_shards):
        sh = small.shard(g, n_shards)
        s = Searcher(sh, weighting=BM25F, stats_ix=small)
        for i, r in enumerate(s.search_batch(qs, limit=None)):
            assert len(r) == len(r.top_n)
            assert all(sh.doc_base <= d < sh.doc_base + sh.n_docs_all for _, d in r.top_n)
            got[i] += [d for _, d in r.top_n]
    for q, docs in zip(qs, got):
        assert sorted(docs) == want_docs(small, q), q
