"""BASELINE.json full-size checks on the GPU (config 2 / config 3: 1M documents, 200k-term vocabulary).

The oracle cannot score 10k queries over 1M documents in seconds, so at this size the CUDA path is
checked (a) against the oracle on a sample of the batch and (b) through size-independent properties:
inclusion-exclusion of match counts, sharded == whole, every kernel family agrees with every other,
idempotence, W11 order, bounds on totals."""
import numpy as np
import pytest

from document_search_engine_b200 import And, BM25F, Or, Term
from document_search_engine_b200.corpus import config_corpus, config_queries
from document_search_engine_b200.searching import Searcher
from oracle.numpy_oracle import NumpyOracle
from tests.parity import assert_query_parity

pytestmark = pytest.mark.gpu
K = 10


@pytest.fixture(scope="module")
def cfg2():
    ix = config_corpus(2)                      # generated on the GPU: 1M docs, ~1.36e8 postings
    return ix


def _run(ix, queries, **kw):
    s = Searcher(ix, weighting=BM25F, **kw)
    batch = s.pack(queries)
    return s.engine.search_batch(batch, K)


def test_config2_sample_against_oracle(cfg2):
    qs = config_queries(2, 10_000).queries
    scores, docids, counts, totals = _run(cfg2, qs)
    o = NumpyOracle(cfg2)
    for i in range(0, len(qs), 50):            # 200 queries of the real batch
        n = int(counts[i])
        assert_query_parity(o, qs[i], list(zip(scores[i, :n].tolist(), docids[i, :n].tolist())), int(totals[i]), K,
                            ctx="config 2 query %d" % i)


def test_config3_variants_sample_against_oracle(cfg2):
    qs = config_queries(3, 2_000).queries       # AND of four 2-way OR-groups, 8 leaves
    scores, docids, counts, totals = _run(cfg2, qs)
    o = NumpyOracle(cfg2)
    for i in range(0, len(qs), 10):            # 200 queries
        n = int(counts[i])
        assert_query_parity(o, qs[i], list(zip(scores[i, :n].tolist(), docids[i, :n].tolist())), int(totals[i]), K,
                            ctx="config 3 query %d" % i)


def _sample_against_oracle(ix, qs, k, every, ctx, **kw):
    s = Searcher(ix, weighting=BM25F, **kw)
    scores, docids, counts, totals = s.engine.search_batch(s.pack(qs), k)
    o = NumpyOracle(ix)
    checked = 0
    for i in range(0, len(qs), every):
        n = int(counts[i])
        assert_query_parity(o, qs[i], list(zip(scores[i, :n].tolist(), docids[i, :n].tolist())), int(totals[i]), k,
                            ctx="%s query %d" % (ctx, i))
        checked += 1
    s.engine.close()
    ix._engine_cache.clear()
    return checked


def test_config4_shape_top100_sample_against_oracle():
    """BASELINE configs[3] shape at 2M documents (vocabulary 500k, 2-4-term AND/OR, top-100: four keys per lane in the
    warp kernels), 200 sampled queries of a 4000-query batch against the oracle."""
    ix = config_corpus(4, n_docs=2_000_000)
    qs = config_queries(4, 4_000).queries
    assert _sample_against_oracle(ix, qs, 100, 20, "config 4 shape") == 200


def test_config5_shape_two_fields_sample_against_oracle():
    """BASELINE configs[4] shape at 1M documents (vocabulary 1M, two fields, title boost 2: every query term is an OR
    across the fields), 250 sampled queries of a 5000-query batch against the oracle."""
    ix = config_corpus(5, n_docs=1_000_000)
    qs = config_queries(5, 5_000).queries
    assert _sample_against_oracle(ix, qs, 10, 20, "config 5 shape") == 250


def test_kernel_families_agree_and_idempotent(cfg2):
    qs = config_queries(2, 3_000).queries
    ref = _run(cfg2, qs)                        # auto: stream + candidate-driven + teams
    again = _run(cfg2, qs)
    for a, b in zip(ref, again):
        assert np.array_equal(a, b)             # idempotent, bit for bit
    # every family accumulates fmaf(w, impact, acc) in the plan's leaf order: the same float32 score per document,
    # hence the same documents, ranks and scores bit for bit
    for variant in (1, 2, 3, 4, 5):
        cfg2._engine_cache.clear()
        got = _run(cfg2, qs, variant=variant)
        assert np.array_equal(got[3], ref[3]), "totals differ for variant %d" % variant
        assert np.array_equal(got[2], ref[2]), "counts differ for variant %d" % variant
        assert np.array_equal(got[1], ref[1]), "docids differ for variant %d" % variant
        assert np.array_equal(got[0].view(np.uint32), ref[0].view(np.uint32)), "scores differ for variant %d" % variant
    cfg2._engine_cache.clear()


def test_inclusion_exclusion_and_bounds(cfg2):
    rng = np.random.default_rng(5)
    pairs = [(int(a), int(b)) for a, b in zip(rng.integers(51, 5000, 400), rng.integers(51, 50000, 400)) if a != b]
    ors = [Or([Term("body", a), Term("body", b)]) for a, b in pairs]
    ands = [And([Term("body", a), Term("body", b)]) for a, b in pairs]
    singles = [Term("body", t) for ab in pairs for t in ab]
    _, _, _, t_or = _run(cfg2, ors)
    _, _, _, t_and = _run(cfg2, ands)
    sc, dc, cn, t_one = _run(cfg2, singles)
    df = t_one.reshape(-1, 2).astype(np.int64)
    # a single term matches exactly its live postings
    for (a, b), d in zip(pairs, df):
        assert d[0] == cfg2.df[cfg2.term_id("body", a)] and d[1] == cfg2.df[cfg2.term_id("body", b)]
    assert np.array_equal(t_or.astype(np.int64) + t_and.astype(np.int64), df.sum(axis=1))     # |A u B| + |A n B| = |A| + |B|
    assert np.all(t_and.astype(np.int64) <= df.min(axis=1)) and np.all(t_or.astype(np.int64) >= df.max(axis=1))
    # W11 order inside every result list
    for i in range(sc.shape[0]):
        n = int(cn[i])
        s, d = sc[i, :n], dc[i, :n].astype(np.int64)
        assert np.all((s[:-1] > s[1:]) | ((s[:-1] == s[1:]) & (d[:-1] < d[1:])))


def test_sharded_equals_whole_full_size(cfg2):
    qset = config_queries(2, 1_000)
    qs = qset.queries
    whole = _run(cfg2, qs)
    G = 3
    keys, totals = [], np.zeros(len(qs), dtype=np.int64)
    from document_search_engine_b200.searching import make_keys
    for g in range(G):
        sh = cfg2.shard(g, G)
        s = Searcher(sh, weighting=BM25F, stats_ix=cfg2)
        sc, dc, cn, tt = s.engine.search_batch(s.pack(qs), K)
        k = make_keys(sc, dc.astype(np.uint64))
        k[dc == 0xFFFFFFFF] = 0
        keys.append(k)
        totals += tt.astype(np.int64)
        s.engine.close()
        sh._engine_cache.clear()
    merged = np.sort(np.concatenate(keys, axis=1), axis=1)[:, ::-1][:, :K]
    from document_search_engine_b200.distributed import decode_keys_host
    m_sc, m_dc, m_cn = decode_keys_host(np.ascontiguousarray(merged))
    assert np.array_equal(totals, whole[3].astype(np.int64))          # match counts add up exactly
    assert np.array_equal(m_cn, whole[2])
    # Shards use corpus-wide statistics (W8) and every kernel family has the same arithmetic, so a query with one
    # group (a term, a flat OR: its leaf order is the caller's on every shard) scores bit for bit as on the whole
    # index.  An AND orders its groups by their size on each shard, which can differ from the whole index's order
    # (another fmaf order): 1e-6 for those.
    one = ~qset.is_and | (qset.n_terms == 1)
    assert one.sum() > 300
    assert np.array_equal(m_dc[one], whole[1][one])
    assert np.array_equal(m_sc[one].view(np.uint32), whole[0][one].view(np.uint32))
    valid = whole[1] != 0xFFFFFFFF
    with np.errstate(invalid="ignore"):
        assert np.all((np.abs(m_sc - whole[0]) <= 1e-6 * np.abs(whole[0])) | ~valid)
    assert np.mean((m_dc == whole[1]) | ~valid) > 0.999
