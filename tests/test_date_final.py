"""Date-ordered weightings (SURVEY.md §8 a10 / f1; reference my_whoosh.py:127-154, selected at
my_flask.py:183): ``final`` is applied to every match before the top-k (W14).  CPU: the scalar restatement
against hand-worked values, and the two oracles against each other.  GPU: the device path against the
oracle, whose scores are float64 where the engine's are float32: final values of documents that share a date
differ only in their last few ulps, so parity here is an absolute tolerance of a few ulps of the final value, and
rank by rank the document is the oracle's or one that ties with it inside that tolerance.  The date orders are
checked bit for bit, ties inside one final value included, by ``tests/test_gpu_final_exact.py``."""
from datetime import datetime, timedelta

import numpy as np
import pytest

from document_search_engine_b200 import And, AscDateBM25F, BM25F, DescDateBM25F, FlatIndex, Not, Or, Term
from document_search_engine_b200.corpus import config_corpus, make_queries
from oracle.numpy_oracle import NumpyOracle
from oracle.whoosh_port import OracleSearcher
from tests.parity import assert_batch_parity

#: a few ulps of a final value (~5.5): one rounding step of (1 - 1/s) next to ~5.5e9 seconds is 2^-20, i.e.
#: ~1e-15 after the division by 10**9, and the fp32 score may land on either side of such a step
FINAL_TOL = 3e-15


class _Stored:
    def __init__(self, fields):
        self.fields = fields

    def stored_fields(self, docnum):
        return self.fields[docnum]


def test_final_known_answers():
    """Hand-worked: 1975-03-04 00:00 + chapter 12 s, counted from 1800-01-01 / down to 2200-01-01."""
    s = _Stored([{"date": datetime(1975, 3, 4), "heading": "Session 740 - CHAPTER 12: notes"},
                 {"date": datetime(1975, 3, 4), "heading": "no number here"}, {"heading": "Chapter 3"}])
    days_desc = (datetime(1975, 3, 4) - datetime(1800, 1, 1)).days        # 63979
    assert days_desc == 63979
    want = ((1 - 1 / 3.5) + (63979 * 86400 + 12) + 1.0) / 10 ** 9
    assert DescDateBM25F().final(s, 0, 3.5) == want == 5.527785613714286
    assert DescDateBM25F().final(s, 1, 3.5) == ((1 - 1 / 3.5) + 63979 * 86400 + 1.0) / 10 ** 9
    assert DescDateBM25F().final(s, 2, 3.5) == 1 - 1 / 3.5                 # no date: no date term, no division
    days_asc = (datetime(2200, 1, 1) - datetime(1975, 3, 4)).days
    assert AscDateBM25F().final(s, 0, 0.5) == ((1 - 1 / 0.5) + (days_asc * 86400 - 12) + 1.0) / 10 ** 9
    terms = DescDateBM25F().doc_final_terms(type("Ix", (), {"n_docs_all": 3, "stored": s.fields})())
    assert terms[0] == 63979 * 86400 + 12 + 1.0 and terms[1] == 63979 * 86400 + 1.0 and np.isnan(terms[2])


def dated_corpus(ix, seed=5):
    """Attach stored fields to a synthetic corpus: ~300 session dates shared by many documents, chapters in
    some headings, one document in ten without a date."""
    rng = np.random.default_rng(seed)
    n = ix.n_docs_all
    session = rng.integers(0, 300, n)
    chapter = rng.integers(0, 25, n)
    undated = rng.random(n) < 0.1
    base = datetime(1963, 12, 8)
    stored = []
    for i in range(n):
        f = {"heading": "Session %d%s" % (session[i], ", Chapter %d" % chapter[i] if chapter[i] % 3 == 0 else "")}
        if not undated[i]:
            f["date"] = base + timedelta(days=int(session[i]) * 17, hours=int(session[i]) % 5)
        stored.append(f)
    ix.stored = stored
    return ix


@pytest.fixture(scope="module")
def dated():
    return dated_corpus(config_corpus(1, device="cpu"))


def date_queries(n, seed):
    qs = make_queries(n, 50_000, seed, 2, 4, "mixed", skip_top=0).queries
    out = []
    for i, q in enumerate(qs):
        if i % 5 == 4 and isinstance(q, (And, Or)):
            q = type(q)(list(q.subqueries) + [Not(Term("body", i % 300))])
        out.append(q)
    return out + [Term("body", 3), Term("body", "no-such-term"), And([Term("body", 7), Term("body", "no-such-term")])]


@pytest.mark.parametrize("cls", [DescDateBM25F, AscDateBM25F])
def test_oracles_agree_on_final(dated, cls):
    w = cls()
    o = NumpyOracle(dated, final_add=w.doc_final_terms(dated))
    port = OracleSearcher(dated, final=lambda searcher, docnum, score: w.final(_Stored(dated.stored), docnum, score))
    for q in date_queries(12, 31):
        top, total = o.search(q, limit=10)
        top_p, total_p = port.search(q, limit=10)
        assert total == total_p
        assert [d for _, d in top] == [d for _, d in top_p]
        assert [v for v, _ in top] == pytest.approx([v for v, _ in top_p], rel=0, abs=FINAL_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("cls", [DescDateBM25F, AscDateBM25F])
@pytest.mark.parametrize("k", [10, 3, 100, 150])
def test_final_on_device(dated, cls, k):
    w = cls()
    o = NumpyOracle(dated, final_add=w.doc_final_terms(dated))
    qs = date_queries(150, 77)
    with dated.searcher(weighting=cls) as s:
        res = s.search_batch(qs, limit=k)
    assert_batch_parity(o, qs, res, k, abs_tol=FINAL_TOL)
    # dated documents rank above undated ones (their values are > 1, the others' are < 1)
    for r in res:
        vals = [v for v, _ in r.top_n]
        assert vals == sorted(vals, reverse=True)


@pytest.mark.gpu
def test_final_switches_with_the_weighting(dated):
    """The engine is shared by the searchers of an index: the final() step follows the weighting."""
    qs = date_queries(40, 9)
    o_plain = NumpyOracle(dated)
    o_desc = NumpyOracle(dated, final_add=DescDateBM25F().doc_final_terms(dated))
    with dated.searcher(weighting=BM25F) as s:
        assert_batch_parity(o_plain, qs, s.search_batch(qs, limit=10), 10)
    with dated.searcher(weighting=DescDateBM25F) as s:
        assert_batch_parity(o_desc, qs, s.search_batch(qs, limit=10), 10, abs_tol=FINAL_TOL)
        page = s.search_page(qs[0], 2, pagelen=5)
        assert page.total == len(s.search(qs[0], limit=10))
    with dated.searcher(weighting=BM25F) as s:
        assert_batch_parity(o_plain, qs, s.search_batch(qs, limit=10), 10)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 100, 150])
def test_final_merge_across_shards(dated, k):
    """Document shards under a final() weighting: every shard's (final value, docnum) lists, laid out as an
    all-gather would, merged by bm25f_merge_final_lists, equal the whole corpus (W8 + W14)."""
    import torch
    from document_search_engine_b200.distributed import device_view
    from document_search_engine_b200.searching import Searcher
    qs = date_queries(60, 5)
    Q, G = len(qs), 3
    o = NumpyOracle(dated, final_add=DescDateBM25F().doc_final_terms(dated))
    vals = torch.empty(G * Q * k, dtype=torch.float64, device="cuda:0")
    docs = torch.empty(G * Q * k, dtype=torch.int32, device="cuda:0")
    totals = np.zeros(Q, dtype=np.uint64)
    searchers = [Searcher(dated.shard(g, G), weighting=DescDateBM25F, stats_ix=dated) for g in range(G)]
    for g, s in enumerate(searchers):
        plan = s.engine.prepare(s.pack(qs), k, arena=True)
        plan.execute()
        d_final, d_docids, d_totals = plan.device_final()
        s.engine.synchronize()
        vals[g * Q * k:(g + 1) * Q * k].copy_(device_view(d_final, Q * k, 0, "<f8"))
        docs[g * Q * k:(g + 1) * Q * k].copy_(device_view(d_docids, Q * k, 0, "<i4"))
        totals += device_view(d_totals, Q, 0).cpu().numpy().view(np.uint64)
        plan.close()
    out_v = torch.empty(Q * k, dtype=torch.float64, device="cuda:0")
    out_d = torch.empty(Q * k, dtype=torch.int32, device="cuda:0")
    out_c = torch.empty(Q, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    eng = searchers[0].engine
    eng.merge_final_lists(vals.data_ptr(), docs.data_ptr(), G, Q, k, out_v.data_ptr(), out_d.data_ptr(), out_c.data_ptr())
    eng.synchronize()
    v = out_v.cpu().numpy().reshape(Q, k)
    d = out_d.cpu().numpy().view(np.uint32).reshape(Q, k)
    c = out_c.cpu().numpy()
    from tests.parity import assert_query_parity
    for i, q in enumerate(qs):
        n = int(c[i])
        assert_query_parity(o, q, list(zip(v[i, :n].tolist(), d[i, :n].tolist())), int(totals[i]), k,
                            ctx="query %d" % i, abs_tol=FINAL_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize("cls", [DescDateBM25F, AscDateBM25F])
def test_final_deep_paging(dated, cls):
    """search_page(qp, pagenum=N, pagelen=10) deep into a date-ordered listing (reference my_flask.py:211: limit =
    pagenum * pagelen grows past the 256 keys a warp keeps): further passes collect the hits ordered strictly after
    the last one returned; limit=None returns every match.  Two searchers with different weightings on one index
    (the reference opens one per request, my_flask.py:183-184) keep their own scoring."""
    w = cls()
    o = NumpyOracle(dated, final_add=w.doc_final_terms(dated))
    qs = [q for q in date_queries(60, 5) if len(o.match_all(q)[0]) > 300][:6] + date_queries(4, 6)
    assert len(qs) > 4
    with dated.searcher(weighting=cls) as s, dated.searcher(weighting=BM25F) as plain:
        for limit in (257, 700, None):
            res = s.search_batch(qs, limit=limit)
            assert_batch_parity(o, qs, res, limit, abs_tol=FINAL_TOL)
        assert_batch_parity(NumpyOracle(dated), qs, plain.search_batch(qs, limit=10), 10)
        page = s.search_page(qs[0], 30, pagelen=10)
        want, total = o.search(qs[0], limit=300)
        assert page.total == total and page.offset == 290 and [h.docnum for h in page] == [d for _, d in want[290:300]]
        assert_batch_parity(o, qs[:2], s.search_batch(qs[:2], limit=20), 20, abs_tol=FINAL_TOL)
