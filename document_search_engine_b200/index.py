"""Flattened, upload-ready inverted index (CSR posting store).

The reference opens a Whoosh index directory (``my_index.py:226-234``) and hands
it to the front ends as the module global ``ix`` (``my_flask.py:549``,
``cli.py:25``).  The engine replaces the *inside* of that object for the scoring
path: everything the BM25F scorer reads (SURVEY.md §8 b, "Data layout across
the boundary") is flattened into a handful of arrays that are uploaded to HBM
once per process:

* ``term_offsets[n_terms+1]`` u64 CSR row pointers; a "term" is a (field, text)
  pair, numbered field-major;
* ``docids[P]`` u32, ascending inside a term; ``tfs[P]`` f32 posting weights (W7);
* ``len_bytes[n_fields, n_docs_all]`` u8 quantised field lengths (W5/W6);
* ``field_length_total[n_fields]`` exact token totals (W4), ``df`` as stored (W3),
  ``deleted`` flags (W9) and ``doc_base`` for document shards (W8).

Corpus parsing, analyzers and the on-disk Whoosh format are out of scope
(SURVEY.md §2); ``from_documents`` exists so tests and small tools can build an
index from already-tokenised documents.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Mapping, Optional, Sequence, Tuple

import itertools
import json
import threading

import numpy as np

from .numeric import lengths_to_bytes

FORMAT_VERSION = 1
_TOKENS = itertools.count(1)


class Schema:
    """Just enough of ``whoosh.fields.Schema`` for ``QueryParser`` and the UI."""

    def __init__(self, names: Sequence[str], stored: Sequence[str] = ()):
        self._names = list(names)
        self._stored = list(stored)

    def names(self):
        return list(self._names)

    def stored_names(self):
        return list(self._stored)

    def __contains__(self, name):
        return name in self._names


class IndexReader:
    """``searcher.ixreader`` surface used by the reference (``my_flask.py:254``)."""

    def __init__(self, ix: "FlatIndex"):
        self._ix = ix

    def frequency(self, fieldname, text) -> float:
        tid = self._ix.term_id(fieldname, text)
        if tid < 0:
            return 0.0
        a, b = int(self._ix.term_offsets[tid]), int(self._ix.term_offsets[tid + 1])
        return float(self._ix.tfs[a:b].sum(dtype=np.float64)) if self._ix.term_weight_total is None \
            else float(self._ix.term_weight_total[tid])

    def doc_frequency(self, fieldname, text) -> int:
        tid = self._ix.term_id(fieldname, text)
        return 0 if tid < 0 else int(self._ix.df[tid])

    def doc_count_all(self):
        return self._ix.doc_count_all()

    def doc_count(self):
        return self._ix.doc_count()

    def field_length(self, fieldname):
        return self._ix.field_length(fieldname)

    def __contains__(self, term):
        return self._ix.term_id(term[0], term[1]) >= 0


class FlatIndex:
    def __init__(self, *, field_names: Sequence[str], n_docs_all: int,
                 term_offsets: np.ndarray, docids: np.ndarray, tfs: np.ndarray,
                 term_field: np.ndarray, len_bytes: np.ndarray,
                 field_length_total: np.ndarray,
                 terms: Optional[Dict[Tuple[int, object], int]] = None,
                 vocab_size: Optional[int] = None,
                 df: Optional[np.ndarray] = None,
                 deleted: Optional[np.ndarray] = None,
                 stored: Optional[Sequence[Mapping]] = None,
                 doc_base: int = 0,
                 global_doc_count_all: Optional[int] = None,
                 term_weight_total: Optional[np.ndarray] = None,
                 scorable: Optional[Sequence[bool]] = None,
                 positions: Optional[Dict[int, Tuple[np.ndarray, np.ndarray]]] = None):
        self.field_names = list(field_names)
        self.n_docs_all = int(n_docs_all)
        self.term_offsets = np.ascontiguousarray(term_offsets, dtype=np.uint64)
        self.docids = np.ascontiguousarray(docids, dtype=np.uint32)
        self.tfs = np.ascontiguousarray(tfs, dtype=np.float32)
        self.term_field = np.ascontiguousarray(term_field, dtype=np.uint8)
        self.len_bytes = np.ascontiguousarray(len_bytes, dtype=np.uint8).reshape(len(self.field_names), self.n_docs_all)
        self.field_length_total = np.ascontiguousarray(field_length_total, dtype=np.uint64)
        self.terms = terms
        self.vocab_size = vocab_size
        n_terms = self.term_offsets.size - 1
        if n_terms != self.term_field.size:
            raise ValueError("term_field must have one entry per posting list")
        if int(self.term_offsets[-1]) != self.docids.size or self.docids.size != self.tfs.size:
            raise ValueError("posting arrays do not match term_offsets")
        # W3: document frequency *as stored* (deleted documents still counted)
        self.df = (np.diff(self.term_offsets).astype(np.uint32) if df is None
                   else np.ascontiguousarray(df, dtype=np.uint32))
        self.deleted = None if deleted is None else np.ascontiguousarray(deleted, dtype=np.uint8)
        self.stored = stored
        self.doc_base = int(doc_base)
        # W8: idf / avgfl come from the whole corpus, never from a shard
        self.global_doc_count_all = int(self.n_docs_all if global_doc_count_all is None else global_doc_count_all)
        self.term_weight_total = term_weight_total
        #: W15: per field, Whoosh's ``schema[field].scorable``.  TEXT fields are; an ID field like the reference's
        #: ``book`` (``my_index.py:152``, ``:171``) is not: its terms score their posting weight (WeightScorer)
        self.scorable = [True] * len(self.field_names) if scorable is None else [bool(x) for x in scorable]
        if len(self.scorable) != len(self.field_names):
            raise ValueError("scorable must have one entry per field")
        #: word order, for phrases (Whoosh: the ``positions`` posting format of a ``TEXT(phrase=True)`` field; reference
        #: ``my_index.py:172-177``): per field index ``f`` the documents' token sequences as posting-list ids,
        #: ``(offsets[n_docs_all + 1], ids[sum of lengths])``, -1 for a token that is not indexed.  A searcher uploads a
        #: field's word order to the device the first time a phrase on the field reaches it (``bm25f_put_positions``).
        self.positions = {int(f): (np.ascontiguousarray(o, dtype=np.int64), np.ascontiguousarray(i, dtype=np.int32))
                          for f, (o, i) in (positions or {}).items()}
        self.schema = Schema(self.field_names, stored=self._stored_names())
        #: identifies this index object in caches that must not hold on to it (Searcher.pack)
        self.token = next(_TOKENS)
        self._engine_cache = {}
        self._lexicons = {}
        self._forward = {}
        self._text_of = None
        self._engine_cache_lock = threading.Lock()

    # ---- Whoosh Index surface -------------------------------------------------
    def doc_count_all(self) -> int:
        return self.global_doc_count_all

    def doc_count(self) -> int:
        """Undeleted documents (``ix.doc_count()``, ``my_flask.py:225``)."""
        if self.deleted is None:
            return self.global_doc_count_all
        return self.global_doc_count_all - int(self.deleted.sum())

    def is_empty(self):
        return self.doc_count() == 0

    def reader(self):
        return IndexReader(self)

    def searcher(self, weighting=None, **kwargs):
        from .searching import Searcher
        return Searcher(self, weighting=weighting, **kwargs)

    # ---- dictionary -----------------------------------------------------------
    @property
    def n_terms(self) -> int:
        return self.term_offsets.size - 1

    @property
    def n_postings(self) -> int:
        return self.docids.size

    def field_index(self, fieldname) -> int:
        try:
            return self.field_names.index(fieldname)
        except ValueError:
            return -1

    def term_id(self, fieldname, text) -> int:
        """Posting-list id of (field, text), or -1 (unknown term/field → empty matcher, W10)."""
        f = self.field_index(fieldname)
        if f < 0:
            return -1
        if self.terms is not None:
            return self.terms.get((f, text), -1)
        # numeric vocabulary: term text is the rank, or "t0000123"
        try:
            r = int(text[1:]) if isinstance(text, str) and text[:1] == "t" else int(text)
        except (TypeError, ValueError):
            return -1
        if r < 0 or r >= self.vocab_size:
            return -1
        return f * self.vocab_size + r

    def is_scorable(self, fieldname) -> bool:
        f = self.field_index(fieldname)
        return f < 0 or self.scorable[f]

    def lexicon(self, fieldname) -> List[str]:
        """The words of a field, sorted (what Whoosh's ``reader.lexicon(fieldname)`` iterates): the expansion
        domain of ``Prefix`` / ``Wildcard`` queries.  Needs a string vocabulary."""
        f = self.field_index(fieldname)
        if f < 0:
            return []
        lex = self._lexicons.get(f)
        if lex is None:
            if self.terms is None:
                raise NotImplementedError("pattern queries need a string vocabulary (this index numbers its terms)")
            lex = self._lexicons[f] = sorted(t for (ff, t) in self.terms if ff == f and isinstance(t, str))
        return lex

    def doc_terms(self, docnum: int, fieldname) -> List[Tuple[object, float]]:
        """``[(text, weight)]`` of one document in one field: its term vector as Whoosh's ``Expander.add_document``
        reads it (``searcher.key_terms([docnum], field)``, reference ``my_index.py:100``).  Served from a
        per-field forward map (the posting store transposed once, on first use)."""
        f = self.field_index(fieldname)
        if f < 0:
            return []
        fw = self._forward.get(f)
        if fw is None:
            tids = np.nonzero(self.term_field == f)[0]
            if tids.size == 0:
                fw = (np.zeros(self.n_docs_all + 1, np.int64), np.zeros(0, np.int64), np.zeros(0, np.float32))
            else:
                a, b = int(self.term_offsets[tids[0]]), int(self.term_offsets[tids[-1] + 1])
                if not (np.diff(tids) == 1).all():
                    raise NotImplementedError("the posting lists of a field must be contiguous")
                lens = np.diff(self.term_offsets[tids[0]:tids[-1] + 2].astype(np.int64))
                term_of = np.repeat(tids, lens)
                d = self.docids[a:b].astype(np.int64)
                order = np.argsort(d, kind="stable")
                starts = np.zeros(self.n_docs_all + 1, np.int64)
                np.cumsum(np.bincount(d, minlength=self.n_docs_all), out=starts[1:])
                fw = (starts, term_of[order], self.tfs[a:b][order])
            self._forward[f] = fw
            if self.terms is not None and self._text_of is None:
                self._text_of = {tid: t for (ff, t), tid in self.terms.items()}
        starts, term_of, w = fw
        local = docnum - self.doc_base
        lo, hi = int(starts[local]), int(starts[local + 1])
        text = (lambda tid: self._text_of[tid]) if self.terms is not None else (lambda tid: tid - f * self.vocab_size)
        return [(text(int(t)), float(x)) for t, x in zip(term_of[lo:hi], w[lo:hi])]

    def term_frequency(self, fieldname, text) -> float:
        """Whoosh ``reader.frequency``: the total weight of the term in the collection."""
        return self.reader().frequency(fieldname, text)

    def field_length(self, fieldname) -> int:
        f = self.field_index(fieldname)
        return 0 if f < 0 else int(self.field_length_total[f])

    def avg_field_length(self, fieldname) -> float:
        """W4: ``field_length / (doc_count_all or 1)``, then ``or 1``."""
        return (self.field_length(fieldname) / (self.doc_count_all() or 1)) or 1.0

    def postings(self, tid: int):
        a, b = int(self.term_offsets[tid]), int(self.term_offsets[tid + 1])
        return self.docids[a:b], self.tfs[a:b]

    def stored_fields(self, docnum: int) -> Mapping:
        local = docnum - self.doc_base
        if self.stored is None:
            return {}
        return self.stored[local]

    def _stored_names(self):
        if not self.stored:
            return []
        names = []
        for d in self.stored[:16]:
            for k in d:
                if k not in names:
                    names.append(k)
        return names

    # ---- construction ---------------------------------------------------------
    @classmethod
    def from_documents(cls, docs: Sequence[Mapping[str, object]], fields: Sequence[str],
                       analyzer=None, stored: Optional[Sequence[str]] = None,
                       deleted: Iterable[int] = (), id_fields: Sequence[str] = (),
                       date_fields: Sequence[str] = ()) -> "FlatIndex":
        """Build from tokenised documents: ``doc[field]`` is a token list or a string
        split on whitespace by default.  Token boosts are all 1 so ``tf`` is the term
        count (W7).  ``id_fields``: fields indexed like Whoosh's ``ID`` type (the reference's ``book``,
        ``my_index.py:152``): the whole value is one term, posting weight 1 (Existence format), no length
        is stored and the field is not scorable (W15).  ``date_fields``: fields whose value is a date (the
        reference's ``date=DATETIME``, ``my_index.py:150-175``): filed under a year, a month and a day token
        (``dates.tier_tokens``) so that ``DateRange`` queries become OR-groups of posting lists; not scorable either.
        A date field that is not in ``fields`` is appended to them."""
        from .dates import tier_tokens
        fields = list(fields) + [f for f in date_fields if f not in fields]
        id_fields = list(id_fields) + list(date_fields)
        analyzer = analyzer or (lambda text: text.split())
        n = len(docs)
        nf = len(fields)
        postings: Dict[Tuple[int, object], Dict[int, float]] = {}
        nf = len(fields)
        lengths = np.zeros((nf, n), dtype=np.int64)
        sequences: Dict[int, List[list]] = {f: [] for f, name in enumerate(fields) if name not in id_fields}
        for d, doc in enumerate(docs):
            for f, name in enumerate(fields):
                v = doc.get(name)
                if v is None:
                    continue
                if name in date_fields:
                    for tok in tier_tokens(v):
                        postings.setdefault((f, tok), {})[d] = 1.0
                    continue
                if name in id_fields:
                    postings.setdefault((f, v), {})[d] = 1.0
                    continue
                toks = analyzer(v) if isinstance(v, str) else list(v)
                while len(sequences[f]) < d:
                    sequences[f].append([])
                sequences[f].append(toks)
                lengths[f, d] = len(toks)
                for t in toks:
                    p = postings.setdefault((f, t), {})
                    p[d] = p.get(d, 0.0) + 1.0
        keys = sorted(postings.keys(), key=lambda k: (k[0], str(k[1])))
        terms = {k: i for i, k in enumerate(keys)}
        offs = np.zeros(len(keys) + 1, dtype=np.uint64)
        dl: List[int] = []
        tl: List[float] = []
        for i, k in enumerate(keys):
            items = sorted(postings[k].items())
            dl.extend(d for d, _ in items)
            tl.extend(w for _, w in items)
            offs[i + 1] = len(dl)
        lb = np.stack([lengths_to_bytes(lengths[f]) for f in range(nf)]) if nf else np.zeros((0, n), np.uint8)
        # a field a document does not have keeps length byte 0 (W5: scored with fl=1)
        del_arr = None
        deleted = list(deleted)
        if deleted:
            del_arr = np.zeros(n, dtype=np.uint8)
            del_arr[deleted] = 1
        stored_docs = None
        if stored:
            stored_docs = [{k: doc[k] for k in stored if k in doc} for doc in docs]
        positions = {}
        for f, seqs in sequences.items():
            seqs = seqs + [[]] * (n - len(seqs))
            po = np.zeros(n + 1, dtype=np.int64)
            np.cumsum([len(x) for x in seqs], out=po[1:])
            positions[f] = (po, np.fromiter((terms[(f, t)] for x in seqs for t in x), dtype=np.int32, count=int(po[-1])))
        return cls(field_names=fields, n_docs_all=n, term_offsets=offs, positions=positions,
                   docids=np.array(dl, dtype=np.uint32), tfs=np.array(tl, dtype=np.float32),
                   term_field=np.array([k[0] for k in keys], dtype=np.uint8),
                   len_bytes=lb, field_length_total=lengths.sum(axis=1).astype(np.uint64),
                   terms=terms, deleted=del_arr, stored=stored_docs,
                   scorable=[name not in id_fields for name in fields])

    # ---- document sharding (W8, SURVEY.md §8 e) ------------------------------
    def shard(self, g: int, n_shards: int) -> "FlatIndex":
        """Contiguous document-range shard ``g`` of ``n_shards`` with local docids.

        Global statistics (``df``, ``doc_count_all``, field totals) are carried
        over unchanged so that idf and avgfl are those of the whole corpus.
        """
        if not (0 <= g < n_shards):
            raise ValueError("shard index out of range")
        lo = (self.n_docs_all * g) // n_shards
        hi = (self.n_docs_all * (g + 1)) // n_shards
        keep = (self.docids >= lo) & (self.docids < hi)
        csum = np.concatenate([[0], np.cumsum(keep, dtype=np.uint64)])
        offs = csum[self.term_offsets.astype(np.int64)]
        return FlatIndex(field_names=self.field_names, n_docs_all=hi - lo, term_offsets=offs,
                         docids=(self.docids[keep] - np.uint32(lo)), tfs=self.tfs[keep],
                         term_field=self.term_field, len_bytes=self.len_bytes[:, lo:hi],
                         field_length_total=self.field_length_total, terms=self.terms,
                         vocab_size=self.vocab_size, df=self.df,
                         deleted=None if self.deleted is None else self.deleted[lo:hi],
                         stored=None if self.stored is None else self.stored[lo:hi],
                         doc_base=self.doc_base + lo,
                         global_doc_count_all=self.global_doc_count_all,
                         term_weight_total=self.term_weight_total, scorable=self.scorable,
                         positions={f: (o[lo:hi + 1] - o[lo], i[int(o[lo]):int(o[hi])]) for f, (o, i) in self.positions.items()})

    # ---- phrases (CPU reference of the device filter, bm25f_phrase_lists; SURVEY.md section 8 f3) --------------
    def phrase_docs(self, fieldname, words: Sequence[object], slop: int = 1) -> np.ndarray:
        """Local docnums (ascending) in which ``words`` occur in this order, every word at most ``slop`` positions
        after the one before (``slop=1``: adjacent) - the documents Whoosh's ``Phrase(fieldname, words, slop)`` lets
        through its ``SpanNear`` chain.  Needs the field's word order (``positions``)."""
        f = self.field_index(fieldname)
        if f < 0:
            return np.zeros(0, np.uint32)
        if f not in self.positions:
            raise NotImplementedError("field %r was flattened without positions: no phrase queries on it" % fieldname)
        tids = [self.term_id(fieldname, w) for w in words]
        if not tids or min(tids) < 0:
            return np.zeros(0, np.uint32)
        cand = None
        for t in sorted(set(tids), key=lambda t: int(self.term_offsets[t + 1] - self.term_offsets[t])):
            d = self.docids[int(self.term_offsets[t]):int(self.term_offsets[t + 1])]
            cand = d if cand is None else np.intersect1d(cand, d, assume_unique=True)
            if cand.size == 0:
                return np.zeros(0, np.uint32)
        offs, ids = self.positions[f]
        out = []
        for d in cand.tolist():
            seq = ids[int(offs[d]):int(offs[d + 1])]
            ends = np.nonzero(seq == tids[0])[0]
            for t in tids[1:]:
                if ends.size == 0:
                    break
                pos = np.nonzero(seq == t)[0]
                # keep the positions that follow some kept position of the previous word by 1 .. slop
                j = np.searchsorted(ends, pos, side="left")             # ends[j - 1] < pos
                ok = (j > 0) & (pos - ends[np.maximum(j - 1, 0)] <= slop)
                ends = pos[ok]
            if ends.size:
                out.append(d)
        return np.asarray(out, dtype=np.uint32)

    # ---- persistence (the "checkpoint": a flattened index file) --------------
    def save(self, path: str) -> None:
        if self.terms is not None:
            tf_ = np.array([k[0] for k in self.terms], dtype=np.uint8)
            tt_ = np.array([str(k[1]) for k in self.terms])
            ti_ = np.array(list(self.terms.values()), dtype=np.int64)
        else:
            tf_, tt_, ti_ = np.zeros(0, np.uint8), np.zeros(0, "U1"), np.zeros(0, np.int64)
        np.savez(path, version=FORMAT_VERSION, field_names=np.array(self.field_names),
                 n_docs_all=self.n_docs_all, term_offsets=self.term_offsets, docids=self.docids,
                 tfs=self.tfs, term_field=self.term_field, len_bytes=self.len_bytes,
                 field_length_total=self.field_length_total, df=self.df,
                 deleted=self.deleted if self.deleted is not None else np.zeros(0, np.uint8),
                 vocab_size=-1 if self.vocab_size is None else self.vocab_size,
                 doc_base=self.doc_base, global_doc_count_all=self.global_doc_count_all,
                 dict_field=tf_, dict_text=tt_, dict_id=ti_, scorable=np.array(self.scorable, dtype=np.uint8),
                 term_weight_total=(self.term_weight_total if self.term_weight_total is not None else np.zeros(0, np.float64)),
                 stored_json=np.array("" if self.stored is None else json.dumps(list(self.stored), default=str)),
                 pos_fields=np.array(sorted(self.positions), dtype=np.int64),
                 **{"pos_%s_%d" % (kind, f): arr for f, pair in self.positions.items() for kind, arr in zip(("off", "ids"), pair)})

    @classmethod
    def load(cls, path: str) -> "FlatIndex":
        z = np.load(path, allow_pickle=False)
        if int(z["version"]) != FORMAT_VERSION:
            raise ValueError("unsupported flat index version %s" % z["version"])
        terms = None
        if z["dict_id"].size:
            terms = {(int(f), str(t)): int(i) for f, t, i in zip(z["dict_field"], z["dict_text"], z["dict_id"])}
        vs = int(z["vocab_size"])
        return cls(field_names=[str(s) for s in z["field_names"]], n_docs_all=int(z["n_docs_all"]),
                   term_offsets=z["term_offsets"], docids=z["docids"], tfs=z["tfs"],
                   term_field=z["term_field"], len_bytes=z["len_bytes"],
                   field_length_total=z["field_length_total"], terms=terms,
                   vocab_size=None if vs < 0 else vs, df=z["df"],
                   deleted=z["deleted"] if z["deleted"].size else None,
                   doc_base=int(z["doc_base"]), global_doc_count_all=int(z["global_doc_count_all"]),
                   scorable=[bool(x) for x in z["scorable"]] if "scorable" in z.files else None,
                   term_weight_total=(z["term_weight_total"] if "term_weight_total" in z.files and z["term_weight_total"].size else None),
                   stored=(json.loads(str(z["stored_json"])) if "stored_json" in z.files and str(z["stored_json"]) else None),
                   positions=({int(f): (z["pos_off_%d" % f], z["pos_ids_%d" % f]) for f in z["pos_fields"]} if "pos_fields" in z.files else None))
