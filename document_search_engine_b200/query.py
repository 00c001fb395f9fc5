"""Query tree nodes with the Whoosh surface the reference relies on.

The reference builds its trees with ``whoosh.qparser.QueryParser`` (default
group AND, ``OR`` keyword; reference ``my_flask.py:189-193``, ``:302``) and
greps ``str(query)`` for ``"<field>:"`` (``my_flask.py:201-205``).  The engine
needs ``Term`` / ``And`` / ``Or`` (SURVEY.md §8 a6, b) plus ``Every`` for the
CLI probe (``cli.py:8-9``) and ``Not`` for the UI's ``a NOT b``
(``search-form.html:20-40``).  A tiny parser for the ``a b OR c NOT e field:d``
subset is provided so the front ends have something to call; the rest of the
query language (phrases, wildcards, ranges) is out of scope (SURVEY.md §8 f3).

``normalize()`` lowers a tree to the engine's input form: an AND of groups,
each group an OR of weighted leaves.  ``Or`` of plain leaves is the one-group
case.
"""
from __future__ import annotations

import re
from dataclasses import dataclass
from typing import Iterable, List, Sequence, Tuple


class Query:
    boost: float = 1.0

    def __and__(self, other):
        return And([self, other])

    def __or__(self, other):
        return Or([self, other])

    def leaves(self) -> Iterable["Term"]:
        raise NotImplementedError

    def all_terms(self):
        return {(t.fieldname, t.text) for t in self.leaves()}

    def normalize(self) -> "Query":
        return self

    def __getstate__(self):
        # the lowered form Searcher.pack remembers on a query belongs to one index: it does not travel
        d = dict(self.__dict__)
        d.pop("_lowered", None)
        return d

    def __ne__(self, other):
        return not self.__eq__(other)


class _Null(Query):
    """Matches nothing (what the parser returns for an empty string)."""

    def __repr__(self):
        return "<_NullQuery>"

    def __str__(self):
        return ""

    def __eq__(self, other):
        return isinstance(other, _Null)

    def __hash__(self):
        return hash("_Null")

    def leaves(self):
        return iter(())


NullQuery = _Null()


class Term(Query):
    def __init__(self, fieldname: str, text, boost: float = 1.0):
        self.fieldname = fieldname
        self.text = text
        self.boost = float(boost)

    def __eq__(self, other):
        return (isinstance(other, Term) and other.fieldname == self.fieldname
                and other.text == self.text and other.boost == self.boost)

    def __hash__(self):
        return hash((self.fieldname, self.text, self.boost))

    def __repr__(self):
        r = "Term(%r, %r" % (self.fieldname, self.text)
        if self.boost != 1.0:
            r += ", boost=%s" % self.boost
        return r + ")"

    def __str__(self):
        # the reference looks for "<field>:" in this rendering (my_flask.py:203)
        t = "%s:%s" % (self.fieldname, self.text)
        if self.boost != 1.0:
            t += "^%s" % self.boost
        return t

    def leaves(self):
        yield self


class Every(Query):
    """All documents that have any term in ``fieldname`` (cli.py:8-9)."""

    def __init__(self, fieldname: str = None, boost: float = 1.0):
        self.fieldname = fieldname
        self.boost = float(boost)

    def __eq__(self, other):
        return (isinstance(other, Every) and other.fieldname == self.fieldname
                and other.boost == self.boost)

    def __hash__(self):
        return hash(("Every", self.fieldname, self.boost))

    def __repr__(self):
        return "Every(%r)" % (self.fieldname,)

    def __str__(self):
        return "%s:*" % (self.fieldname or "*")

    def leaves(self):
        return iter(())


class _Compound(Query):
    JOINT = " ? "

    def __init__(self, subqueries: Sequence[Query], boost: float = 1.0):
        for q in subqueries:
            if not isinstance(q, Query):
                raise TypeError("%r is not a query" % (q,))
        self.subqueries = list(subqueries)
        self.boost = float(boost)

    def __eq__(self, other):
        return (type(other) is type(self) and other.subqueries == self.subqueries
                and other.boost == self.boost)

    def __hash__(self):
        h = hash(type(self).__name__) ^ hash(self.boost)
        for q in self.subqueries:
            h ^= hash(q)
        return h

    def __repr__(self):
        r = "%s(%r" % (type(self).__name__, self.subqueries)
        if self.boost != 1.0:
            r += ", boost=%s" % self.boost
        return r + ")"

    def __str__(self):
        r = "(" + self.JOINT.join(str(q) for q in self.subqueries) + ")"
        if self.boost != 1.0:
            r += "^%s" % self.boost
        return r

    def __iter__(self):
        return iter(self.subqueries)

    def __len__(self):
        return len(self.subqueries)

    def __getitem__(self, i):
        return self.subqueries[i]

    def leaves(self):
        for q in self.subqueries:
            yield from q.leaves()

    def normalize(self):
        """What Whoosh's ``CompoundQuery.normalize`` does to the trees this path serves ([W] query/compound.py;
        ``QueryParser.parse`` normalizes by default, so every query the reference hands to ``search`` has been
        through it, ``my_flask.py:189-193``): nested nodes of the same class are merged (the child's boost goes
        into its subqueries), null children are dropped, EQUAL SUBQUERIES ARE KEPT ONCE (a stemmed field turns
        ``walk walking`` into two equal terms: Whoosh scores the term once), a single survivor is returned
        with the boosts multiplied."""
        subs: List[Query] = []
        for q in self.subqueries:
            q = q.normalize()
            if type(q) is type(self):
                subs.extend(_with_boost(s, s.boost * q.boost) for s in q.subqueries)
            else:
                subs.append(q)
        seen = set()
        kept: List[Query] = []
        for q in subs:
            if isinstance(q, _Null) or q in seen:
                continue
            seen.add(q)
            kept.append(q)
        if not kept:
            return NullQuery
        if len(kept) == 1:
            return _with_boost(kept[0], kept[0].boost * self.boost)
        return type(self)(kept, boost=self.boost)

    def flattened(self):
        """Score-neutral restructuring for ``lower`` (no de-duplication: ``Searcher.search`` scores the tree it is
        given, as Whoosh does): nested nodes of the same class are merged, their boost pushed into the children."""
        subs: List[Query] = []
        for q in self.subqueries:
            if isinstance(q, _Compound):
                q = q.flattened()
            if type(q) is type(self):
                subs.extend(_with_boost(s, s.boost * q.boost) for s in q.subqueries)
            else:
                subs.append(q)
        return type(self)(subs, boost=self.boost)


class And(_Compound):
    JOINT = " AND "


class MultiTerm(Query):
    """``Prefix`` / ``Wildcard`` (the reference's UI documents ``book:tes?``, ``search-form.html:20-40``; Whoosh
    ``query/terms.py``).  [W] ``MultiTerm.matcher`` expands the pattern over the field's lexicon, in lexicon order,
    into ``Or([Term(field, word), ...], boost=self.boost)`` - a single matching word becomes its plain ``Term``
    matcher (the boost is NOT applied in that case), none a NullMatcher - and although pattern queries ask for a
    constant score, ``Searcher.postings`` falls back to the searcher's weighting, so the expansion is scored by BM25F
    like any other ``Or``.  The engine does the same rewrite on the host (``expand_multiterms``) and scores the
    ``Or`` on the flat-OR kernels."""

    def __init__(self, fieldname: str, text: str, boost: float = 1.0):
        self.fieldname = fieldname
        self.text = text
        self.boost = float(boost)

    def __eq__(self, other):
        return (type(other) is type(self) and other.fieldname == self.fieldname and other.text == self.text
                and other.boost == self.boost)

    def __hash__(self):
        return hash((type(self).__name__, self.fieldname, self.text, self.boost))

    def __repr__(self):
        return "%s(%r, %r%s)" % (type(self).__name__, self.fieldname, self.text, "" if self.boost == 1.0 else ", boost=%s" % self.boost)

    def leaves(self):
        return iter(())

    def matches(self, word: str) -> bool:
        raise NotImplementedError

    def literal_prefix(self) -> str:
        """Every matching word starts with this (narrows the scan of the sorted lexicon)."""
        raise NotImplementedError

    def expand(self, lexicon: Sequence[str]) -> Query:
        """``lexicon``: the field's words, sorted."""
        from bisect import bisect_left
        pre = self.literal_prefix()
        words = []
        for i in range(bisect_left(lexicon, pre), len(lexicon)):
            w = lexicon[i]
            if not w.startswith(pre):
                break
            if self.matches(w):
                words.append(w)
        if not words:
            return NullQuery
        if len(words) == 1:
            return Term(self.fieldname, words[0])                 # Whoosh drops the pattern's boost here
        return Or([Term(self.fieldname, w) for w in words], boost=self.boost)


class Prefix(MultiTerm):
    def __str__(self):
        return "%s:%s*" % (self.fieldname, self.text)

    def matches(self, word):
        return word.startswith(self.text)

    def literal_prefix(self):
        return self.text


class Wildcard(MultiTerm):
    """``?`` one character, ``*`` any run, ``[...]`` a character class (fnmatch rules, as Whoosh)."""
    SPECIAL_CHARS = frozenset("*?[")

    def __str__(self):
        return "%s:%s" % (self.fieldname, self.text)

    def _regex(self):
        r = self.__dict__.get("_rx")
        if r is None:
            import fnmatch
            r = self.__dict__["_rx"] = re.compile(fnmatch.translate(self.text))
        return r

    def matches(self, word):
        return self._regex().match(word) is not None

    def literal_prefix(self):
        for i, ch in enumerate(self.text):
            if ch in self.SPECIAL_CHARS:
                return self.text[:i]
        return self.text

    def normalize(self):
        # [W] Wildcard.normalize: no special character -> Term; "*" -> Every; one trailing "*" -> Prefix
        text = self.text
        if text == "*":
            return Every(self.fieldname, boost=self.boost)
        if not any(ch in self.SPECIAL_CHARS for ch in text):
            return Term(self.fieldname, text, boost=self.boost)
        if text.endswith("*") and not any(ch in self.SPECIAL_CHARS for ch in text[:-1]):
            return Prefix(self.fieldname, text[:-1], boost=self.boost)
        return self


class DateRange(MultiTerm):
    """``date:[oct 1970 to dec 8 1970]`` / ``date:"feb 1964"`` (reference ``search-form.html:26``, ``:39``; parsed by
    Whoosh's ``DateParserPlugin``, ``my_flask.py:189-193``).  [W] ``query.DateRange`` is a ``NumericRange`` over the
    DATETIME field: it compiles to the ``Or`` of the tiered numeric terms that cover the range inside a
    ``ConstantScoreQuery(boost)`` - a matching document scores ``boost``, and adds it to the other clauses' scores
    inside an ``And``.  The flat index files every document date under a year, a month and a day token of a
    non-scorable field (``dates.py``), so the same rewrite gives an OR-group of ordinary posting lists whose
    postings score exactly ``boost``.  ``start`` / ``end`` are datetimes or dates, inclusive, ``None`` = open."""

    def __init__(self, fieldname: str, start=None, end=None, boost: float = 1.0):
        MultiTerm.__init__(self, fieldname, "[%s to %s]" % ("" if start is None else start, "" if end is None else end), boost)
        self.start = start
        self.end = end

    def __str__(self):
        return "%s:%s" % (self.fieldname, self.text)

    def expand(self, lexicon: Sequence[str]) -> Query:
        from . import dates
        days = [w for w in lexicon if w.startswith("D")]
        if not days:
            return NullQuery
        lo = dates.first_day(self.start) if self.start is not None else dates.date(int(days[0][1:5]), 1, 1)
        hi = dates.last_day(self.end) if self.end is not None else dates.date(int(days[-1][1:5]), 12, 31)
        have = set(lexicon)
        toks = [t for t in dates.range_cover(lo, hi) if t in have]
        if not toks:
            return NullQuery
        if len(toks) == 1:
            return Term(self.fieldname, toks[0], boost=self.boost)
        return Or([Term(self.fieldname, t, boost=self.boost) for t in toks])


#: pseudo-field of the leaves that stand for a per-batch document list (``Phrase`` filters); never in a schema
FILTER_FIELD = "\x00filter"


class Phrase(Query):
    """``"dead sea"`` / ``exact:"way toward health"~2`` (reference ``search-form.html:20-40``; Whoosh ``query.Phrase``).
    [W] ``Phrase.matcher``: a word that is not in the field -> NullMatcher; else the ``SpanNear`` chain of the words'
    term matchers, ordered, every word 1 .. ``slop`` positions after the one before (``slop=1``: adjacent), over an
    IntersectionMatcher - so a matching document scores the SUM of its words' BM25F scores, and the positions only
    decide whether it matches.  The engine does the same in two steps: a positional filter on the device finds the
    documents that pass (``bm25f_phrase_lists``, over the candidates of the rarest word; ``FlatIndex.phrase_docs`` is
    its CPU reference) and keeps them as a per-batch posting list, and the query runs as ``And(words..., that list)`` -
    the list is the smallest group, so the candidate-driven kernel walks it and looks the words' postings up."""

    def __init__(self, fieldname: str, words: Sequence[object], slop: int = 1, boost: float = 1.0):
        self.fieldname = fieldname
        self.words = list(words)
        self.slop = int(slop)
        self.boost = float(boost)

    def __eq__(self, other):
        return (isinstance(other, Phrase) and other.fieldname == self.fieldname and other.words == self.words
                and other.slop == self.slop and other.boost == self.boost)

    def __hash__(self):
        return hash(("Phrase", self.fieldname, tuple(self.words), self.slop, self.boost))

    def __repr__(self):
        return "Phrase(%r, %r%s%s)" % (self.fieldname, self.words, "" if self.slop == 1 else ", slop=%d" % self.slop,
                                      "" if self.boost == 1.0 else ", boost=%s" % self.boost)

    def __str__(self):
        return '%s:"%s"%s' % (self.fieldname, " ".join(str(w) for w in self.words), "" if self.slop == 1 else "~%d" % self.slop)

    def leaves(self):
        return iter(())

    def normalize(self):
        # [W] Phrase.normalize: no words -> NullQuery, one word -> its Term
        if not self.words:
            return NullQuery
        if len(self.words) == 1:
            return Term(self.fieldname, self.words[0], boost=self.boost)
        return self


def has_phrase(q: Query) -> bool:
    if isinstance(q, Phrase):
        return True
    if isinstance(q, _Compound):
        return any(has_phrase(s) for s in q.subqueries)
    if isinstance(q, Not):
        return has_phrase(q.query)
    return False


def expand_phrases(q: Query, register) -> Query:
    """Replace every ``Phrase`` by ``And(its words..., Term(FILTER_FIELD, i))`` where ``i = register(phrase)`` numbers
    the document list that will stand for the phrase's positional test in this batch (``Not(Phrase)``: the list alone)."""
    if isinstance(q, Phrase):
        q = q.normalize()
        if not isinstance(q, Phrase):
            return q
        return And([Term(q.fieldname, w) for w in q.words] + [Term(FILTER_FIELD, register(q))], boost=q.boost)
    if isinstance(q, _Compound):
        return type(q)([expand_phrases(s, register) for s in q.subqueries], boost=q.boost)
    if isinstance(q, Not):
        if isinstance(q.query, Phrase) and len(q.query.words) > 1:
            return Not(Term(FILTER_FIELD, register(q.query)))
        return Not(expand_phrases(q.query, register))
    return q


def has_multiterm(q: Query) -> bool:
    if isinstance(q, MultiTerm):
        return True
    if isinstance(q, _Compound):
        return any(has_multiterm(s) for s in q.subqueries)
    if isinstance(q, Not):
        return has_multiterm(q.query)
    return False


def expand_multiterms(q: Query, lexicon_of) -> Query:
    """Replace every ``Prefix`` / ``Wildcard`` node by its expansion; ``lexicon_of(fieldname)`` -> sorted words."""
    if isinstance(q, MultiTerm):
        return q.expand(lexicon_of(q.fieldname))
    if isinstance(q, _Compound):
        return type(q)([expand_multiterms(s, lexicon_of) for s in q.subqueries], boost=q.boost)
    if isinstance(q, Not):
        return Not(expand_multiterms(q.query, lexicon_of))
    return q


class Or(_Compound):
    JOINT = " OR "


class Not(Query):
    """Excludes the documents matching ``query``.  Served inside ``And`` (Whoosh turns ``And([a, Not(b)])``
    into an AndNot matcher: the documents of ``a`` that are not in ``b``, scored by ``a`` alone);
    reference UI help ``search-form.html:20-40``."""

    def __init__(self, query: Query, boost: float = 1.0):
        if not isinstance(query, Query):
            raise TypeError("%r is not a query" % (query,))
        self.query = query
        self.boost = float(boost)

    def __eq__(self, other):
        return isinstance(other, Not) and other.query == self.query

    def __hash__(self):
        return hash(("Not", self.query))

    def __repr__(self):
        return "Not(%r)" % (self.query,)

    def __str__(self):
        return "NOT " + str(self.query)

    def leaves(self):
        return iter(())              # a negated term is not a scoring leaf

    def normalize(self):
        q = self.query.normalize()
        if isinstance(q, _Null):
            return NullQuery         # NOT nothing: no constraint (dropped by the enclosing And)
        return Not(q)


def _with_boost(q: Query, boost: float) -> Query:
    if boost == q.boost:
        return q
    if isinstance(q, Term):
        return Term(q.fieldname, q.text, boost=boost)
    if isinstance(q, Every):
        return Every(q.fieldname, boost=boost)
    if isinstance(q, _Compound):
        return type(q)(q.subqueries, boost=boost)
    if isinstance(q, MultiTerm):
        return type(q)(q.fieldname, q.text, boost=boost)
    return q                     # Not / Null carry no score


#: ``Leaf.group`` of a leaf inside a NOT clause (BM25F_GROUP_NOT in include/bm25f.h)
GROUP_NOT = 255

# --------------------------------------------------------------------------
# Lowering to the engine's input form
# --------------------------------------------------------------------------

@dataclass
class Leaf:
    fieldname: str
    text: object
    boost: float
    group: int


class UnsupportedQuery(NotImplementedError):
    """Raised for trees the GPU path does not serve (no CPU fallback exists)."""


def lower(q: Query) -> Tuple[List[Leaf], int, str]:
    """Lower ``q`` to ``(leaves, n_groups, kind)``.

    ``kind`` is ``"groups"`` (AND of OR-groups; ``Or`` of leaves is one group),
    ``"every"`` or ``"null"``.  Boosts on compound nodes are pushed into the
    leaves, which is exact because W10 scores are sums of leaf scores.
    """
    if isinstance(q, _Compound):
        q = q.flattened()
        if len(q.subqueries) == 1 and not isinstance(q.subqueries[0], Not):
            return lower(_with_boost(q.subqueries[0], q.subqueries[0].boost * q.boost))
    if isinstance(q, _Null):
        return [], 0, "null"
    if isinstance(q, Every):
        return [Leaf(q.fieldname, None, q.boost, 0)], 1, "every"
    if isinstance(q, Term):
        return [Leaf(q.fieldname, q.text, q.boost, 0)], 1, "groups"
    if isinstance(q, Not):
        # Whoosh's root-level Not is an InverseMatcher over every document of the index, a full scan
        # outside this path.
        raise UnsupportedQuery("a top-level Not() has no positive part to score: %r" % (q,))
    if isinstance(q, (And, Or)):
        # Whoosh's compound matcher pulls the Not children out, builds the matcher of the rest and
        # wraps it in AndNotMatcher(rest, union of the negated queries); nothing positive -> no hits.
        conj = isinstance(q, And)
        leaves: List[Leaf] = []
        negatives: List[Leaf] = []
        g = 0
        for s in q.subqueries:
            if isinstance(s, _Null):
                if conj:
                    return [], 0, "null"          # Whoosh: an And with a NullMatcher child matches nothing
                continue
            if isinstance(s, _Compound) and len(s.subqueries) == 1 and isinstance(s.subqueries[0], Term):
                s = _with_boost(s.subqueries[0], s.subqueries[0].boost * s.boost)
            if isinstance(s, Term):
                leaves.append(Leaf(s.fieldname, s.text, s.boost * q.boost, g))
            elif isinstance(s, Or) and conj:
                for t in s.subqueries:
                    if not isinstance(t, Term):
                        raise UnsupportedQuery("And(Or(...)) groups may only contain Term leaves: %r" % (t,))
                    leaves.append(Leaf(t.fieldname, t.text, t.boost * s.boost * q.boost, g))
            elif isinstance(s, Not):
                nq = s.query.flattened() if isinstance(s.query, _Compound) else s.query
                inner = nq.subqueries if isinstance(nq, Or) else [nq]
                for t in inner:
                    if isinstance(t, _Null):
                        continue                  # NOT nothing: no constraint
                    if not isinstance(t, Term):
                        raise UnsupportedQuery("Not() may contain a Term or an Or of Terms: %r" % (t,))
                    negatives.append(Leaf(t.fieldname, t.text, 1.0, GROUP_NOT))
                continue
            elif conj:
                raise UnsupportedQuery("And() may contain Term, Or(Term...) or Not(...) children: %r" % (s,))
            else:
                raise UnsupportedQuery("Or() may contain Term or Not(...) children on the GPU path: %r" % (s,))
            if conj:
                g += 1
        if not leaves:
            return [], 0, "null"
        return leaves + negatives, (g if conj else 1), "groups"
    raise UnsupportedQuery("unsupported query node %r" % (q,))


# --------------------------------------------------------------------------
# Minimal parser (Term / AND / OR / field:term / parentheses-free)
# --------------------------------------------------------------------------

_TOKEN_RE = re.compile(r"\s*(?:(\w+):)?([^\s()]+)")
_DATE_EXPR_RE = re.compile(r"\b(\w+):(?:\[([^\]]*)\]|\"([^\"]*)\")")
_PHRASE_RE = re.compile(r"(?:\b(\w+):)?\"([^\"]*)\"(?:~(\d+))?")


class QueryParser:
    """``QueryParser(fieldname, schema)`` for the subset ``a b``, ``a AND b``,
    ``a OR b``, ``a NOT b``, ``field:a``.  AND binds tighter than OR, as in Whoosh's default
    grammar.  ``analyzer`` maps a raw token to zero or more index terms
    (lower-casing, stemming ...); the default lower-cases.
    """

    def __init__(self, fieldname: str, schema=None, analyzer=None, termclass=Term, date_fields=("date",)):
        self.fieldname = fieldname
        self.schema = schema
        self.analyzer = analyzer or (lambda field, text: [text.lower()])
        self.termclass = termclass
        #: fields whose values are dates: ``field:[a to b]``, ``field:"feb 1964"``, ``field:1964`` become ``DateRange``
        #: (what ``qp.add_plugin(DateParserPlugin())`` does in the reference, ``my_flask.py:190``)
        self.date_fields = tuple(date_fields)

    def add_plugin(self, plugin):  # accepted for call-compatibility (my_flask.py:190)
        return None

    def parse(self, text: str) -> Query:
        from . import dates
        held: List[Query] = []

        def hold(m):
            if m.group(1) not in self.date_fields:
                return m.group(0)
            expr = m.group(2) if m.group(2) is not None else m.group(3)
            start, end = dates.parse_range(expr)                 # DateParseError: the caller redirects (my_flask.py:193-196)
            held.append(DateRange(m.group(1), start, end))
            return " \x00%d " % (len(held) - 1)
        text = _DATE_EXPR_RE.sub(hold, text or "")

        def hold_phrase(m):
            # Whoosh's PhrasePlugin: the quoted words are analysed like any other text of the field
            field = m.group(1) or self.fieldname
            if m.group(1) and self.schema is not None and hasattr(self.schema, "names") and field not in self.schema.names():
                field = self.fieldname
            words = [t for w in m.group(2).split() for t in self.analyzer(field, w)]
            held.append(Phrase(field, words, slop=int(m.group(3) or 1)).normalize())
            return " \x00%d " % (len(held) - 1)
        text = _PHRASE_RE.sub(hold_phrase, text)
        nodes: List[object] = []          # Query nodes and the markers "AND" / "OR"
        for m in _TOKEN_RE.finditer(text or ""):
            field, tok = m.group(1), m.group(2)
            if field is None and tok in ("AND", "OR", "NOT"):
                nodes.append(tok)
                continue
            if field is None and tok.startswith("\x00"):
                nodes.append(held[int(tok[1:])])
                continue
            if field in self.date_fields:
                start, end = dates.parse_span(tok)
                nodes.append(DateRange(field, start, end))
                continue
            field = field or self.fieldname
            if any(ch in Wildcard.SPECIAL_CHARS for ch in tok):
                # Whoosh's WildcardPlugin: the pattern is not analysed (lower-cased only)
                known = self.schema is None or not hasattr(self.schema, "names") or field in self.schema.names()
                nodes.append(Wildcard(field if known else self.fieldname, tok.lower() if known else "%s:%s" % (field, tok.lower())).normalize())
                continue
            if self.schema is not None and hasattr(self.schema, "names") and field not in self.schema.names():
                tok, field = "%s:%s" % (field, tok), self.fieldname
            terms = [self.termclass(field, t) for t in self.analyzer(field, tok)]
            if len(terms) == 1:
                nodes.append(terms[0])
            elif terms:
                nodes.append(And(terms))
        # NOT negates the node that follows it
        out0: List[object] = []
        i = 0
        while i < len(nodes):
            if nodes[i] == "NOT":
                if i + 1 < len(nodes) and isinstance(nodes[i + 1], Query):
                    out0.append(Not(nodes[i + 1]))
                    i += 2
                else:
                    i += 1             # dangling NOT: drop it
                continue
            out0.append(nodes[i])
            i += 1
        nodes = out0
        # Infix operators take their immediate neighbours, AND before OR; what is
        # left side by side is joined by the default group (AND), as the
        # reference's form explains ("both words", search-form.html:21).
        for op, cls in (("AND", And), ("OR", Or)):
            out: List[object] = []
            i = 0
            while i < len(nodes):
                n = nodes[i]
                if n == op and out and isinstance(out[-1], Query) and i + 1 < len(nodes) \
                        and isinstance(nodes[i + 1], Query):
                    out[-1] = cls([out[-1], nodes[i + 1]])
                    i += 2
                    continue
                if n == op:         # dangling operator: drop it
                    i += 1
                    continue
                out.append(n)
                i += 1
            nodes = out
        nodes = [n for n in nodes if isinstance(n, Query)]
        return And(nodes).normalize() if nodes else NullQuery
