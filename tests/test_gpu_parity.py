"""GPU parity tests proper: CUDA path (through the façade -> ctypes -> C ABI) vs the oracle."""
import numpy as np
import pytest

from document_search_engine_b200 import And, BM25F, FlatIndex, Or, Term
from document_search_engine_b200.corpus import (config_corpus, config_queries, make_corpus, make_queries,
                                                 TITLE, BODY)
from oracle.numpy_oracle import NumpyOracle
from tests.parity import assert_batch_parity, assert_query_parity
from tests.test_oracle_kat import kat1_index

pytestmark = pytest.mark.gpu


def test_kat1_gpu():
    ix = kat1_index()
    with ix.searcher(weighting=BM25F) as s:
        r = s.search(Or([Term("f", "a"), Term("f", "b")]), limit=10)
        assert len(r) == 3 and [h.docnum for h in r] == [2, 3, 0]
        want = [3.1036244074953756, 2.1209246397136083, 1.5080645161290325]
        assert [h.score for h in r] == pytest.approx(want, rel=1e-6)
        r = s.search(And([Term("f", "a"), Term("f", "b")]), limit=10)
        assert len(r) == 2 and [h.docnum for h in r] == [2, 3]
        assert s.search(Term("f", "nope")).is_empty()
        assert s.search(And([Term("f", "a"), Term("f", "nope")])).is_empty()
        assert len(s.search(Or([Term("f", "a"), Term("f", "nope")]))) == 3


def test_kat1_deleted_gpu():
    ix = kat1_index(deleted=[2])
    o = NumpyOracle(ix)
    with ix.searcher() as s:
        for q in (Or([Term("f", "a"), Term("f", "b")]), And([Term("f", "a"), Term("f", "b")]), Term("f", "a")):
            r = s.search(q)
            assert_query_parity(o, q, r.top_n, len(r), 10)


@pytest.fixture(scope="module")
def cfg1():
    ix = config_corpus(1, device="cpu")
    return ix, NumpyOracle(ix)


@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("mode", ["and", "or", "mixed"])
def test_config1(cfg1, mode, variant):
    """BASELINE configs[0] (and OR / mixed variations of it), both scoring kernels."""
    ix, o = cfg1
    qs = make_queries(1000, 50_000, 20261001, 2, 2 if mode == "and" else 4, mode)
    with ix.searcher(weighting=BM25F, variant=variant) as s:
        res = s.search_batch(qs.queries, limit=10)
    assert_batch_parity(o, qs.queries, res, 10)


def test_config1_variants_groups(cfg1):
    ix, o = cfg1
    qs = make_queries(300, 50_000, 20261003, 4, 4, "and", variants=True)
    with ix.searcher() as s:
        res = s.search_batch(qs.queries, limit=10)
    assert_batch_parity(o, qs.queries, res, 10)


@pytest.mark.parametrize("variant,chunk,stages", [(1, 64, 2), (1, 256, 8), (1, 2048, 3), (2, 0, 0)])
@pytest.mark.parametrize("tile_docs,split", [(256, 512), (1024, 4096), (4096, 0), (16384, 0), (17408, 1 << 20)])
def test_tiling_and_splitting(cfg1, tile_docs, split, variant, chunk, stages):
    """Tiny tiles, tiny work items, tiny/huge pipeline stages: many tiles per query, chunks that
    split posting sub-ranges, many partial lists to merge."""
    ix, o = cfg1
    qs = make_queries(200, 50_000, 77, 2, 4, "mixed", skip_top=0)       # includes the densest terms
    with ix.searcher(tile_docs=tile_docs, split_postings=split, variant=variant, chunk_postings=chunk,
                     stages=stages) as s:
        res = s.search_batch(qs.queries, limit=10)
    assert_batch_parity(o, qs.queries, res, 10)


@pytest.mark.parametrize("subtile,wsplit,warps,pf", [(128, 2048, 16, 512), (512, 0, 4, 0xFFFFFFFF), (1024, 1 << 14, 8, 0),
                                                      (2816, 1 << 20, 16, 4096), (12288, 1 << 12, 4, 1024)])
@pytest.mark.parametrize("mode", ["mixed", "variants"])
def test_stream_kernel(cfg1, subtile, wsplit, warps, pf, mode):
    """Stream kernel: sub-range sizes, many small items per query (document ranges that start
    inside lists), warps per CTA, prefetch distances, 8-leaf AND-of-OR queries."""
    ix, o = cfg1
    if mode == "variants":
        qs = make_queries(150, 50_000, 31, 4, 4, "and", variants=True, skip_top=0)
    else:
        qs = make_queries(300, 50_000, 78, 1, 4, "mixed", skip_top=0)
    kw = dict(variant=3, subtile_docs=subtile, warp_split=wsplit, stream_warps=warps, prefetch_postings=pf)
    with ix.searcher(**kw) as s:
        res = s.search_batch(qs.queries, limit=10)
        assert s.engine.stats()["n_launches"] <= 4
    assert_batch_parity(o, qs.queries, res, 10)
    with ix.searcher(**kw) as s:
        res = s.search_batch(qs.queries[:60], limit=32)
    assert_batch_parity(o, qs.queries[:60], res, 32)


@pytest.mark.parametrize("subtile,warps,split,pf", [(128, 16, 2048, 2), (512, 4, 0, 0xFFFFFFFF), (1024, 8, 1 << 12, 0),
                                                     (2944, 16, 0, 16), (12288, 3, 1 << 20, 1)])
@pytest.mark.parametrize("mode", ["mixed", "variants"])
def test_team_kernel(cfg1, subtile, warps, split, pf, mode):
    """Warp-team kernel: slice sizes (several table windows per item / one slice per item), warps
    per CTA, item splitting (document ranges that start inside lists), prefetch distances, 8-leaf
    AND-of-OR queries, k = 10 and 32."""
    ix, o = cfg1
    if mode == "variants":
        qs = make_queries(150, 50_000, 31, 4, 4, "and", variants=True, skip_top=0)
    else:
        qs = make_queries(300, 50_000, 78, 1, 4, "mixed", skip_top=0)
    kw = dict(variant=4, cta_slice_docs=subtile, cta_warps=warps, cta_split=split, cta_prefetch=pf)
    with ix.searcher(**kw) as s:
        res = s.search_batch(qs.queries, limit=10)
        assert s.engine.stats()["n_launches"] <= 4
    assert_batch_parity(o, qs.queries, res, 10)
    with ix.searcher(**kw) as s:
        res = s.search_batch(qs.queries[:60], limit=32)
    assert_batch_parity(o, qs.queries[:60], res, 32)


@pytest.mark.parametrize("split,ratio", [(0, 0), (64, 1), (1 << 20, 1000)])
@pytest.mark.parametrize("mode", ["mixed", "variants", "or", "and"])
def test_isect_kernel(cfg1, split, ratio, mode):
    """Candidate-driven kernel forced for every eligible query (variant 5): flat ORs (every leaf is a
    candidate leaf, duplicates dropped), ANDs, AND-of-OR groups; tiny items (document ranges that start
    inside lists); and the auto routing with extreme ratios (everything / nothing goes to it)."""
    ix, o = cfg1
    if mode == "variants":
        qs = make_queries(150, 50_000, 31, 4, 4, "and", variants=True, skip_top=0)
    else:
        qs = make_queries(300, 50_000, 78, 1, 4, mode, skip_top=0)
    for variant in (5, 0):
        with ix.searcher(variant=variant, isect_split=split, isect_ratio=ratio) as s:
            res = s.search_batch(qs.queries, limit=10)
        assert_batch_parity(o, qs.queries, res, 10)
    with ix.searcher(variant=5, isect_split=split) as s:
        res = s.search_batch(qs.queries[:60], limit=32)
    assert_batch_parity(o, qs.queries[:60], res, 32)


@pytest.mark.parametrize("k", [1, 3, 100, 150, 1024])
def test_limits(cfg1, k):
    ix, o = cfg1
    qs = make_queries(60, 50_000, 5, 2, 3, "or", skip_top=0)
    with ix.searcher() as s:
        res = s.search_batch(qs.queries, limit=k)
    assert_batch_parity(o, qs.queries, res, k)


@pytest.mark.parametrize("variant", [0, 3, 5])
@pytest.mark.parametrize("k", [33, 64, 100, 128, 150, 256])
def test_four_keys_per_lane(cfg1, k, variant):
    """32 < k <= 128 on the stream and candidate-driven kernels (four keys per lane): ORs with thousands
    of matches, ANDs with fewer than k, AND-of-OR groups, many partial lists to merge."""
    ix, o = cfg1
    qs = (make_queries(80, 50_000, 5, 2, 3, "mixed", skip_top=0).queries
          + make_queries(40, 50_000, 6, 4, 4, "and", variants=True, skip_top=0).queries)
    with ix.searcher(variant=variant, warp_split=4096, isect_split=128) as s:
        res = s.search_batch(qs, limit=k)
        st = s.engine.stats()
    assert st["postings_cta"] == 0               # nothing fell back to the CTA kernels
    assert_batch_parity(o, qs, res, k)


def test_limit_none_and_paging_past_kernel_k(cfg1):
    ix, o = cfg1
    qs = make_queries(6, 50_000, 9, 2, 3, "or", skip_top=0)            # thousands of matches each
    with ix.searcher() as s:
        res = s.search_batch(qs.queries, limit=None)
        assert_batch_parity(o, qs.queries, res, None)
        res = s.search_batch(qs.queries, limit=2500)
        assert_batch_parity(o, qs.queries, res, 2500)
        page = s.search_page(qs.queries[0], 3, 10)
        top, total = o.search(qs.queries[0], limit=30)
        assert page.total == total and len(page) == total and page.offset == 20 and page.pagelen == 10
        assert [h.docnum for h in page] == [d for _, d in top[20:30]]


def test_two_fields_boosts_per_field_B():
    ix = make_corpus(3000, 2000, 123, (TITLE, BODY), device="cpu")
    qs = make_queries(300, 2000, 321, 1, 3, "mixed", fields=("title", "body"), field_boosts=(2.0, 1.0), skip_top=0)
    w = BM25F(B=0.6, K1=1.5, title_B=0.2)
    o = NumpyOracle(ix, B=0.6, K1=1.5, field_B={"title": 0.2})
    with ix.searcher(weighting=w, tile_docs=512) as s:
        res = s.search_batch(qs.queries, limit=10)
    assert_batch_parity(o, qs.queries, res, 10)


def test_deleted_zero_bytes_and_ties():
    ix = make_corpus(5000, 300, 99, device="cpu")
    rng = np.random.default_rng(0)
    ix.deleted = (rng.random(ix.n_docs_all) < 0.2).astype(np.uint8)
    ix.len_bytes[0, rng.random(ix.n_docs_all) < 0.1] = 0            # W5: scored with fl = 1
    ix.tfs[:] = 1.0                                                  # many exact score ties
    o = NumpyOracle(ix)
    qs = make_queries(200, 300, 11, 1, 4, "mixed", skip_top=0)
    with ix.searcher(tile_docs=1024) as s:
        res = s.search_batch(qs.queries, limit=10)
    assert_batch_parity(o, qs.queries, res, 10)


@pytest.mark.parametrize("variant", [1, 2])
def test_float_weights_use_unpacked_payload(variant):
    ix = make_corpus(2000, 500, 5, device="cpu")
    ix.tfs *= 1.5                                                    # non-integral posting weights (field boost)
    o = NumpyOracle(ix)
    qs = make_queries(100, 500, 3, 1, 3, "mixed", skip_top=0)
    with ix.searcher(variant=variant, tile_docs=512) as s:
        assert s.engine.stats()["packed_payload"] == 0
        res = s.search_batch(qs.queries, limit=10)
    assert_batch_parity(o, qs.queries, res, 10)


def test_leaf_boosts_zero_and_negative(cfg1):
    ix, o = cfg1
    qs = [Or([Term("body", 60, boost=0.0), Term("body", 70)]),
          Or([Term("body", 60, boost=-1.0), Term("body", 70, boost=0.5)]),
          And([Term("body", 55, boost=3.0), Term("body", 60)]),
          Term("body", 52)]
    with ix.searcher() as s:
        res = s.search_batch(qs, limit=10)
    assert_batch_parity(o, qs, res, 10)


def test_sharded_equals_whole(cfg1):
    """W8: shards with global statistics give the same scores; merged lists equal the whole."""
    ix, o = cfg1
    qs = make_queries(100, 50_000, 4, 2, 3, "mixed")
    from document_search_engine_b200.searching import Searcher
    tops = [[] for _ in qs.queries]
    totals = [0] * len(qs.queries)
    for g in range(3):
        sh = ix.shard(g, 3)
        s = Searcher(sh, stats_ix=ix)
        for i, r in enumerate(s.search_batch(qs.queries, limit=10)):
            tops[i].extend(r.top_n)
            totals[i] += len(r)
    with Searcher(ix) as s:
        whole = s.search_batch(qs.queries, limit=10)
    for i, q in enumerate(qs.queries):
        merged = sorted(tops[i], key=lambda t: (-t[0], t[1]))[:10]
        assert_query_parity(o, q, merged, totals[i], 10, ctx="query %d" % i)
        if not qs.is_and[i] or qs.n_terms[i] == 1:
            # one group: the same leaf order on every shard, the whole index's float32 scores bit for bit
            assert merged == whole[i].top_n and totals[i] == len(whole[i]), "query %d" % i


def test_every_field_and_cli_harness():
    """``searcher.search(Every('session'), limit=None)`` is the reference's only harness (cli.py:9): every
    live document that has the field, constant score, docnum order; here with deleted documents, documents
    without the field, a boost, an unknown field, and more matches than one kernel pass returns."""
    from document_search_engine_b200 import Every
    ix = make_corpus(3000, 300, 17, (TITLE, BODY), device="cpu")
    rng = np.random.default_rng(1)
    ix.deleted = (rng.random(ix.n_docs_all) < 0.1).astype(np.uint8)
    ix.len_bytes[0, rng.random(ix.n_docs_all) < 0.3] = 0           # 30 % of the documents have no title
    o = NumpyOracle(ix)
    with ix.searcher() as s:
        for q, limit in ((Every("title"), 10), (Every("body"), None), (Every("title", boost=2.5), 1500), (Every("nope"), 10)):
            r = s.search(q, limit=limit)
            assert_query_parity(o, q, r.top_n, len(r), limit, ctx=str(q))
        r = s.search(Every("title"), limit=None)
        assert [h.docnum for h in r] == sorted(h.docnum for h in r) and all(h.score == 1.0 for h in r)
        live_with_title = int(((ix.len_bytes[0] != 0) & (ix.deleted == 0)).sum())
        assert len(r) == live_with_title == r.scored_length()


def test_pipelined_stream_equals_serial(cfg1):
    """bm25f_submit / bm25f_collect (two batches in flight) return what bm25f_search_batch returns, batch
    by batch and in order; the workspace rules are enforced loudly."""
    from document_search_engine_b200._ffi import EngineError
    ix, o = cfg1
    sets = [make_queries(n, 50_000, 500 + i, 2, 4, "mixed", skip_top=0).queries for i, n in enumerate((300, 7, 1200, 1, 450))]
    with ix.searcher(weighting=BM25F) as s:
        batches = [s.pack(q) for q in sets]
        serial = [s.search_packed(b, 10) for b in batches]
        piped = list(s.search_packed_stream(iter(batches), 10))
        assert len(piped) == len(serial)
        for a, b in zip(serial, piped):
            for x, y in zip(a, b):
                assert np.array_equal(x, y)
        # a consumer that stops early leaves no batch behind
        g = s.search_packed_stream(iter(batches), 10)
        next(g)
        g.close()
        assert np.array_equal(s.search_packed(batches[0], 10)[1], serial[0][1])
        # three in flight: refused; out of order: refused; then both collect fine
        p0 = s.engine.submit(batches[0], 10)
        p1 = s.engine.submit(batches[1], 10)
        with pytest.raises(EngineError, match="in flight"):
            s.engine.submit(batches[2], 10)
        with pytest.raises(EngineError, match="order"):
            p1.collect()
        # a refused collect leaves the batch in flight
        r0, r1 = p0.collect(), p1.collect()
        assert np.array_equal(r0[1], serial[0][1]) and np.array_equal(r0[3], serial[0][3])
        assert np.array_equal(r1[1], serial[1][1]) and np.array_equal(r1[0], serial[1][0])
        with pytest.raises(RuntimeError, match="already collected"):
            p1.collect()
        # and the engine is usable again
        r = s.search_packed(batches[3], 10)
        assert np.array_equal(r[1], serial[3][1])
