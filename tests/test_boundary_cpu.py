"""The C-ABI boundary without a GPU: the library loads, exports every symbol include/bm25f.h declares,
reports its ABI version, and the product path fails loudly when no device is present (no CPU fallback)."""
import ctypes
import os
import re

import numpy as np
import pytest

from document_search_engine_b200 import _ffi
from document_search_engine_b200 import And, FlatIndex, Or, Prefix, Term, Wildcard
from document_search_engine_b200.query import Not, NullQuery, QueryParser, expand_multiterms, lower
from document_search_engine_b200.variants import Variants, expand_with_map
from oracle.numpy_oracle import NumpyOracle
from oracle.whoosh_port import OracleSearcher

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "bm25f.h")


def declared_functions():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(bm25f_[a-z_]+)\s*\(", src)))


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_ffi.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return ctypes.CDLL(_ffi.LIB_PATH)


def test_header_and_binding_agree():
    assert declared_functions() == sorted(_ffi.EXPORTS)
    src = open(HEADER).read()
    assert int(re.search(r"#define BM25F_ABI_VERSION (\d+)", src).group(1)) == _ffi.ABI_VERSION
    assert int(re.search(r"#define BM25F_MAX_K\s+(\d+)", src).group(1)) == _ffi.MAX_K
    assert int(re.search(r"#define BM25F_MAX_LEAVES_PER_QUERY (\d+)", src).group(1)) == _ffi.MAX_LEAVES_PER_QUERY


def test_library_exports_every_declared_symbol(lib):
    missing = [f for f in declared_functions() if not hasattr(lib, f)]
    assert not missing
    lib.bm25f_abi_version.restype = ctypes.c_int
    assert lib.bm25f_abi_version() == _ffi.ABI_VERSION


def test_struct_layouts_match_header():
    # field order / count of the ctypes mirrors vs the header's typedefs
    src = open(HEADER).read()
    bodies = {name: body for body, name in re.findall(r"typedef struct \{([^}]*)\} (\w+);", src)}
    for cname, cls in (("bm25f_index_desc", _ffi.IndexDesc), ("bm25f_options", _ffi.Options),
                       ("bm25f_query_batch", _ffi.QueryBatchDesc), ("bm25f_stats", _ffi.Stats)):
        body = bodies[cname]
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = re.findall(r"(\w+)\s*;", body)
        assert names == [n for n, _ in cls._fields_], cname


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    from document_search_engine_b200.corpus import make_corpus
    ix = make_corpus(50, 40, 1, device="cpu")
    with pytest.raises(_ffi.EngineError):
        ix.searcher()


def test_bad_arguments_do_not_crash(lib):
    lib.bm25f_create.restype = ctypes.c_int
    lib.bm25f_last_error.restype = ctypes.c_char_p
    out = ctypes.c_void_p()
    assert lib.bm25f_create(None, 0, None, ctypes.byref(out)) == -1
    assert b"null" in lib.bm25f_last_error()
    d = _ffi.IndexDesc(_ffi.ABI_VERSION + 7, 1, 0, 0, 0, 0, None, None, None, None, None, None)
    assert lib.bm25f_create(ctypes.byref(d), 0, None, ctypes.byref(out)) == -5       # ABI mismatch
    lib.bm25f_destroy.restype = None
    lib.bm25f_destroy(None)


def test_variants_table(tmp_path):
    p = tmp_path / "uk_us_variations.txt"
    p.write_text("colour color\nhonour honor\n\nanalyse analyze\n", encoding="utf-8")
    v = Variants.load(str(p))
    assert v.uk_variations["colour"] == "color" and v.us_variations["analyze"] == "analyse"
    assert v.uk_us_variations == {"colour", "color", "honour", "honor", "analyse", "analyze"}
    assert v.other("color") == "colour" and v.other("grey") is None
    # the reference's own use: substitute only when the variant occurs in the index (my_flask.py:253-256)
    assert v.substitute("colour", lambda w: 3 if w == "color" else 0) == "color"
    assert v.substitute("colour", lambda w: 0) == "colour"
    # config-3 rewrite: AND of OR-groups
    q = v.expand(And([Term("exact", "colour"), Term("exact", "grey"), Term("exact", "honor", boost=2.0)]))
    assert str(q) == str(And([Or([Term("exact", "colour"), Term("exact", "color")]), Term("exact", "grey"),
                              Or([Term("exact", "honor", boost=2.0), Term("exact", "honour", boost=2.0)])]))
    q = v.expand(Term("exact", "colour"), only_if=lambda f, w: False)
    assert str(q) == str(Term("exact", "colour"))
    q = expand_with_map(And([Term("body", 60), Term("body", 61)]), lambda r: r ^ 1)
    assert str(q) == str(And([Or([Term("body", 60), Term("body", 61)]), Or([Term("body", 61), Term("body", 60)])]))
    # every pair read both ways, and the config-3 rewrite lowers to one group per query word: a 2-way OR group per
    # word that has a variant, a plain leaf for one that has none
    for uk, us in v.uk_variations.items():
        assert v.us_variations[us] == uk and v.other(uk) == us and v.other(us) == uk
    q = v.expand(And([Term("exact", w) for w in ("analyse", "colour", "honour")] + [Term("exact", "zzzz")]))
    assert len(q.subqueries) == 4 and all(isinstance(s, Or) and len(s.subqueries) == 2 for s in q.subqueries[:3])
    assert isinstance(q.subqueries[3], Term)
    leaves, groups, kind = lower(q)
    assert kind == "groups" and groups == 4 and len(leaves) == 7


def test_non_scorable_field_w15():
    """W15: Whoosh's BM25F.scorer() hands a field that is not scorable (the reference's ``book=ID``, my_index.py:152,
    :171; the UI's book filter writes ``book:xyz`` / ``NOT book:xyz`` into the query, static/main.js:5-16) a
    WeightScorer: the score of a posting is its weight (1.0 for an ID field), times the boost - no idf, no length."""
    docs = [{"body": "seth speaks of joy", "book": "ss"}, {"body": "joy and vitality joy", "book": "nopr"},
            {"body": "the nature of joy", "book": "nopr"}, {"body": "dreams", "book": "deavf1"}]
    ix = FlatIndex.from_documents(docs, ["body", "book"], id_fields=["book"])
    assert ix.scorable == [True, False] and ix.len_bytes[1].tolist() == [0, 0, 0, 0]
    assert ix.term_id("book", "nopr") >= 0 and ix.term_id("book", "no") < 0          # the whole value is the term
    for o in (OracleSearcher(ix), NumpyOracle(ix)):
        top, total = o.search(Term("book", "nopr"))
        assert total == 2 and top == [(1.0, 1), (1.0, 2)]
        top, total = o.search(Term("book", "nopr", boost=2.5))
        assert top == [(2.5, 1), (2.5, 2)]
        both, _ = o.search(And([Term("body", "joy"), Term("book", "nopr")]))
        joy = dict((d, s) for s, d in o.search(Term("body", "joy"))[0])
        assert [(d, pytest.approx(joy[d] + 1.0, rel=1e-15)) for s, d in both] == [(d, s) for s, d in both]
        assert sorted(d for _, d in both) == [1, 2]
        top, total = o.search(And([Term("body", "joy"), Not(Term("book", "nopr"))]))
        assert total == 1 and top[0][1] == 0 and top[0][0] == pytest.approx(joy[0], rel=1e-15)
    # the host side hands the engine boost-only leaf weights and a -1 norm row for such a field
    from document_search_engine_b200.scoring import BM25F
    norm = BM25F().norm_tables(ix)
    assert (norm[1] == -1.0).all() and (norm[0] > 0).all()
    # a flat index file keeps the flag (and the stored fields)
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        ix2 = FlatIndex.from_documents(docs, ["body", "book"], id_fields=["book"], stored=["book"])
        ix2.save(os.path.join(d, "ix.npz"))
        back = FlatIndex.load(os.path.join(d, "ix.npz"))
        assert back.scorable == [True, False] and back.stored_fields(3) == {"book": "deavf1"}
        assert np.array_equal(back.docids, ix2.docids) and back.term_id("book", "ss") == ix2.term_id("book", "ss")


def test_normalize_like_whoosh():
    """CompoundQuery.normalize ([W] query/compound.py) as the parser applies it (my_flask.py:189-193): equal
    subqueries once, nested same-class nodes merged with their boost, null children dropped; ``lower`` itself does
    not de-duplicate (Searcher.search scores the tree it is given)."""
    a, b = Term("f", "a"), Term("f", "b")
    assert And([a, a, b]).normalize() == And([a, b])
    assert Or([a, Or([b, a], boost=2.0)]).normalize() == Or([a, Term("f", "b", boost=2.0), Term("f", "a", boost=2.0)])
    assert And([a, NullQuery]).normalize() == a and Or([NullQuery]).normalize() == NullQuery
    assert And([Or([a], boost=3.0)], boost=2.0).normalize() == Term("f", "a", boost=6.0)
    assert QueryParser("f").parse("walk Walk home") == And([Term("f", "walk"), Term("f", "home")])
    leaves, g, kind = lower(And([a, a, b]))
    assert [(lf.text, lf.group) for lf in leaves] == [("a", 0), ("a", 1), ("b", 2)] and g == 3
    assert lower(And([a, NullQuery]))[2] == "null" and lower(Or([a, NullQuery]))[1] == 1


def _books_index():
    rng = np.random.default_rng(11)
    books = ["ss", "nopr", "deavf1", "deavf2", "tes1", "tes2", "tes9", "test", "tps"]
    docs = []
    for d in range(400):
        toks = ["w%d" % t for t in rng.zipf(1.4, size=int(rng.integers(4, 40))) if t < 200] or ["w1"]
        docs.append({"body": toks, "book": books[int(rng.integers(0, len(books)))]})
    return FlatIndex.from_documents(docs, ["body", "book"], id_fields=["book"])


PATTERN_QUERIES = [Wildcard("book", "tes?"), Prefix("book", "dea"), Wildcard("book", "t*s"), Wildcard("book", "x*"),
                   Wildcard("book", "tes[12]", boost=3.0), Prefix("book", "nop", boost=3.0), Prefix("body", "w1"),
                   And([Term("body", "w1"), Wildcard("book", "tes?")]), And([Term("body", "w2"), Not(Prefix("book", "dea"))]),
                   Or([Term("body", "w3"), Prefix("book", "t", boost=0.5)]), And([Prefix("body", "w19"), Wildcard("book", "q?")])]


def test_pattern_queries_f3():
    """Prefix / Wildcard (reference UI ``book:tes?``, search-form.html:20-40): expansion over the field's lexicon in
    lexicon order, one word -> plain Term without the pattern's boost, none -> nothing ([W] MultiTerm.matcher); the
    two oracles expand independently of the engine's host rewrite and must agree with each other and with it."""
    ix = _books_index()
    assert ix.lexicon("book") == sorted(["ss", "nopr", "deavf1", "deavf2", "tes1", "tes2", "tes9", "test", "tps"])
    assert str(expand_multiterms(Wildcard("book", "tes?"), ix.lexicon)) == "(book:tes1 OR book:tes2 OR book:tes9 OR book:test)"
    assert expand_multiterms(Prefix("book", "nop", boost=3.0), ix.lexicon) == Term("book", "nopr")
    assert expand_multiterms(Wildcard("book", "x*"), ix.lexicon) == NullQuery
    assert QueryParser("body").parse("w1 book:tes? NOT book:dea*") == And([Term("body", "w1"), Wildcard("book", "tes?"), Not(Prefix("book", "dea"))])
    a, b = OracleSearcher(ix), NumpyOracle(ix)
    for q in PATTERN_QUERIES:
        ta, na = a.search(q, limit=None)
        tb, nb = b.search(q, limit=None)
        assert na == nb and [d for _, d in ta] == [d for _, d in tb], q
        assert [s for s, _ in ta] == pytest.approx([s for s, _ in tb], rel=1e-12), q
        # ... and with the expansion done by the engine's host code, scored as a plain tree
        te, ne = a.search(expand_multiterms(q, ix.lexicon), limit=None)
        assert ne == na and [d for _, d in te] == [d for _, d in ta], q


class _HostOnlySearcher(object):
    """The host half of Searcher (no engine): enough for the key-term arithmetic."""

    def __new__(cls, ix):
        from document_search_engine_b200.searching import Searcher
        s = object.__new__(Searcher)
        s.ix = s.stats_ix = ix
        return s


def test_key_terms_f4():
    """searcher.key_terms / key_terms_from_text (reference my_index.py:100, my_flask.py:431-434): Whoosh's Bo1 expansion
    model, the engine's host code against the oracle's restatement; ties broken by the word, weights normalised."""
    ix = _books_index()
    s, o = _HostOnlySearcher(ix), OracleSearcher(ix)
    text = "w1 w7 w7 w150 w3 nosuchword w7 w9"
    got = s.key_terms_from_text("body", text, numterms=4)
    want = o.key_terms([(t, 1) for t in text.split()], "body", numterms=4)
    assert [w for w, _ in got] == [w for w, _ in want] and len(got) == 4
    assert [x for _, x in got] == pytest.approx([x for _, x in want], rel=1e-12)
    assert got[0][1] > got[-1][1] > 0 and got[0][1] <= 1.0 + 1e-12
    assert "nosuchword" not in [w for w, _ in s.key_terms_from_text("body", text, numterms=50)]
    # from a document's term vector
    d = 17
    vec = ix.doc_terms(d, "body")
    assert sorted(w for w, _ in vec) == sorted(set(t for t in ["w%d" % i for i in range(200)] if ix.term_id("body", t) >= 0
                                                   and d in ix.postings(ix.term_id("body", t))[0].tolist()))
    got = s.key_terms([d], "body", numterms=10)
    want = o.key_terms(vec, "body", numterms=10)
    assert got == [(w, pytest.approx(x, rel=1e-12)) for w, x in want]
    assert s.key_terms_from_text("body", "", numterms=3) == [] and s.key_terms_from_text("nofield", "w1") == []
