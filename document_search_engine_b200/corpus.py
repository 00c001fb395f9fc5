"""Synthetic Zipf corpora and query batches (SURVEY.md §8 d).

The reference ships no corpus (the indexed books are copyrighted;
``my_index.py:184`` reads ``books/<abbr>.txt`` which is absent), so every parity
and throughput figure comes from the generator specified in SURVEY.md §8 d:

* vocabulary of ``V`` ranks, ``p(r) ∝ r^-1``;
* document length ``clip(round(lognormal(5.0, 0.6)), 8, 4096)`` (title field of
  config 5: ``clip(round(lognormal(2.0, 0.4)), 1, 32)``);
* ``tf`` = multiplicity of the term in the document;
* a stateless counter-based hash (SplitMix64 finaliser keyed by seed, field,
  docid, position), so any document can be regenerated anywhere.

The generator is written with torch integer ops only, so the same code builds a
10k-document index on the CPU for tests and a 10M-document one on a B200 in
seconds.  It is data plumbing, not part of the scoring path.  The result is a
``FlatIndex`` over host (numpy) arrays with a numeric vocabulary (term text is
the rank, printable as ``t0000123``).
"""
from __future__ import annotations

from dataclasses import dataclass, field as dc_field
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from .index import FlatIndex
from .numeric import lengths_to_bytes
from .query import And, Or, Query, Term

_M1 = 0xBF58476D1CE4E5B9 - (1 << 64)
_M2 = 0x94D049BB133111EB - (1 << 64)
_GOLD = 0x9E3779B97F4A7C15 - (1 << 64)


def _lsr(x: torch.Tensor, s: int) -> torch.Tensor:
    return (x >> s) & ((1 << (64 - s)) - 1)


def _mix(x: torch.Tensor) -> torch.Tensor:
    """SplitMix64 finaliser on int64 tensors (two's-complement wrap-around)."""
    x = (x ^ _lsr(x, 30)) * _M1
    x = (x ^ _lsr(x, 27)) * _M2
    return x ^ _lsr(x, 31)


def _uniform(h: torch.Tensor) -> torch.Tensor:
    """float64 in [0, 1) from the top 53 bits."""
    return _lsr(h, 11).to(torch.float64) * (1.0 / 9007199254740992.0)


def _salt(seed: int, fieldno: int, stream: int) -> int:
    v = (seed * 0x9E3779B97F4A7C15 + fieldno * 0xD1B54A32D192ED03 + stream * 0x8CB92BA72F3D8DD7) & ((1 << 64) - 1)
    return v - (1 << 64) if v >= (1 << 63) else v


def zipf_cdf(V: int, s: float = 1.0) -> np.ndarray:
    p = 1.0 / np.arange(1, V + 1, dtype=np.float64) ** s
    c = np.cumsum(p)
    c /= c[-1]
    c[-1] = 1.0
    return c


@dataclass
class FieldSpec:
    name: str
    mu: float = 5.0
    sigma: float = 0.6
    lo: int = 8
    hi: int = 4096


BODY = FieldSpec("body")
TITLE = FieldSpec("title", mu=2.0, sigma=0.4, lo=1, hi=32)


def doc_lengths(n_docs: int, seed: int, fieldno: int, spec: FieldSpec, device="cpu",
                start: int = 0) -> torch.Tensor:
    d = torch.arange(start, start + n_docs, dtype=torch.int64, device=device)
    u1 = _uniform(_mix(d * _GOLD + _salt(seed, fieldno, 1)))
    u2 = _uniform(_mix(d * _GOLD + _salt(seed, fieldno, 2)))
    z = torch.sqrt(-2.0 * torch.log1p(-u1)) * torch.cos(2.0 * torch.pi * u2)
    L = torch.round(torch.exp(spec.mu + spec.sigma * z))
    return L.clamp_(spec.lo, spec.hi).to(torch.int64)


def _field_postings(n_docs: int, V: int, seed: int, fieldno: int, spec: FieldSpec, cdf: torch.Tensor,
                    device, chunk_tokens: int, tokens: Optional[list] = None):
    """(sorted unique key=term*n_docs+doc, tf counts, lengths) for one field.  ``tokens``: a list that receives the
    field's ranks in document order (int32 chunks), when the caller wants the word order."""
    lengths = doc_lengths(n_docs, seed, fieldno, spec, device)
    csum = torch.cumsum(lengths, 0)
    keys_out, cnt_out = [], []
    d0 = 0
    salt = _salt(seed, fieldno, 3)
    while d0 < n_docs:
        # largest doc range whose token count fits the chunk budget
        base = int(csum[d0 - 1]) if d0 else 0
        d1 = int(torch.searchsorted(csum, torch.tensor(base + chunk_tokens, device=device), right=True))
        d1 = max(d1, d0 + 1)
        d1 = min(d1, n_docs)
        ls = lengths[d0:d1]
        ntok = int(ls.sum())
        doc = torch.repeat_interleave(torch.arange(d0, d1, dtype=torch.int64, device=device), ls,
                                      output_size=ntok)
        first = torch.cumsum(ls, 0) - ls
        pos = torch.arange(ntok, dtype=torch.int64, device=device) - torch.repeat_interleave(first, ls, output_size=ntok)
        u = _uniform(_mix(_mix((doc << 13) + pos + salt)))
        del pos
        rank = torch.searchsorted(cdf, u, right=True).clamp_(max=V - 1)
        del u
        if tokens is not None:
            tokens.append(rank.to(torch.int32).cpu())
        key = rank * n_docs + doc
        del rank, doc
        key, _ = torch.sort(key)
        uk, cnt = torch.unique_consecutive(key, return_counts=True)
        keys_out.append(uk)
        cnt_out.append(cnt)
        d0 = d1
    keys = torch.cat(keys_out)
    cnts = torch.cat(cnt_out)
    if len(keys_out) > 1:
        keys, order = torch.sort(keys)
        cnts = cnts[order]
    return keys, cnts, lengths


def make_corpus(n_docs: int, vocab: int, seed: int, fields: Sequence[FieldSpec] = (BODY,),
                device: Optional[str] = None, chunk_tokens: int = 1 << 28, zipf_s: float = 1.0,
                positions: bool = False) -> FlatIndex:
    """Generate the flattened index of a synthetic corpus.  ``positions``: also keep every field's word order
    (``FlatIndex.positions``: token ``fno * vocab + rank`` in document order), so that phrase queries can run on it."""
    if device is None:
        device = "cuda" if torch.cuda.is_available() else "cpu"
    cdf = torch.from_numpy(zipf_cdf(vocab, zipf_s)).to(device)
    offs_parts, doc_parts, tf_parts, lb_parts, totals = [], [], [], [], []
    base = 0
    word_order = {}
    for fno, spec in enumerate(fields):
        toks = [] if positions else None
        keys, cnts, lengths = _field_postings(n_docs, vocab, seed, fno, spec, cdf, device, chunk_tokens, toks)
        if positions:
            po = np.zeros(n_docs + 1, dtype=np.int64)
            np.cumsum(lengths.cpu().numpy(), out=po[1:])
            ids = torch.cat(toks).numpy() if toks else np.zeros(0, np.int32)
            ids += np.int32(fno * vocab)
            word_order[fno] = (po, ids)
            del toks
        term = torch.div(keys, n_docs, rounding_mode="floor")
        doc = keys - term * n_docs
        df = torch.bincount(term, minlength=vocab)
        offs = torch.cumsum(df, 0) + base
        offs_parts.append(offs.cpu().numpy().astype(np.uint64))
        doc_parts.append(doc.to(torch.int32).cpu().numpy().view(np.uint32))
        tf_parts.append(cnts.to(torch.float32).cpu().numpy())
        lcpu = lengths.cpu().numpy()
        lb_parts.append(lengths_to_bytes(lcpu))
        totals.append(int(lcpu.sum()))
        base += int(keys.numel())
        del keys, cnts, term, doc, df, offs
    term_offsets = np.concatenate([np.zeros(1, np.uint64)] + offs_parts)
    term_field = np.repeat(np.arange(len(fields), dtype=np.uint8), vocab)
    return FlatIndex(field_names=[f.name for f in fields], n_docs_all=n_docs, term_offsets=term_offsets,
                     docids=np.concatenate(doc_parts), tfs=np.concatenate(tf_parts), term_field=term_field,
                     len_bytes=np.stack(lb_parts), field_length_total=np.array(totals, dtype=np.uint64),
                     vocab_size=vocab, positions=word_order)


# --------------------------------------------------------------------------
# Query batches
# --------------------------------------------------------------------------

_U64 = np.uint64


def _mix_np(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64)
    with np.errstate(over="ignore"):
        x = (x ^ (x >> _U64(30))) * _U64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> _U64(27))) * _U64(0x94D049BB133111EB)
    return x ^ (x >> _U64(31))


def _uniform_np(h: np.ndarray) -> np.ndarray:
    return (h >> _U64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def _draw_ranks(seed: int, n_queries: int, max_terms: int, vocab: int, skip_top: int, zipf_s: float) -> np.ndarray:
    """``[n_queries, max_terms]`` distinct Zipf ranks >= skip_top per row."""
    cdf = zipf_cdf(vocab, zipf_s)
    c0 = cdf[skip_top - 1] if skip_top > 0 else 0.0
    cq = (cdf[skip_top:] - c0) / (1.0 - c0)
    cq[-1] = 1.0
    out = np.zeros((n_queries, max_terms), dtype=np.int64)
    q = np.arange(n_queries, dtype=np.uint64)
    with np.errstate(over="ignore"):
        for j in range(max_terms):
            attempt = np.zeros(n_queries, dtype=np.uint64)
            pending = np.ones(n_queries, dtype=bool)
            while pending.any():
                h = _mix_np(_mix_np(q * _U64(64) + _U64(j) + _U64(seed) * _U64(0x9E3779B97F4A7C15))
                            + attempt * _U64(0xD1B54A32D192ED03))
                r = skip_top + np.minimum(np.searchsorted(cq, _uniform_np(h), side="right"), cq.size - 1)
                dup = np.zeros(n_queries, dtype=bool)
                for i in range(j):
                    dup |= out[:, i] == r
                ok = pending & ~dup
                out[ok, j] = r[ok]
                pending &= dup
                attempt += _U64(1)
    return out


@dataclass
class QuerySet:
    """A batch of queries in two forms: trees for the façade/oracle and the
    rank matrix they were drawn from."""
    queries: List[Query]
    ranks: np.ndarray
    n_terms: np.ndarray
    is_and: np.ndarray


def variant_partner(r: np.ndarray, skip_top: int = 50) -> np.ndarray:
    """Config-3 synthetic spelling-variant involution: ``r <-> r+1`` for even ``r - skip_top``."""
    r = np.asarray(r)
    return np.where((r - skip_top) % 2 == 0, r + 1, r - 1)


def make_queries(n_queries: int, vocab: int, seed: int, min_terms: int = 2, max_terms: int = 4,
                 mode: str = "mixed", fields: Sequence[str] = ("body",), field_boosts: Sequence[float] = (1.0,),
                 variants: bool = False, skip_top: int = 50, zipf_s: float = 1.0) -> QuerySet:
    """``mode``: ``"and"``, ``"or"`` or ``"mixed"`` (50/50).  With ``variants`` every term
    becomes ``Or(term, partner)`` and the query is the AND of those groups (config 3).
    With several ``fields`` every term is searched in each field (OR across fields,
    boosts applied as leaf boosts: config 5)."""
    if variants:
        vocab_draw = vocab - 1 if (vocab - skip_top) % 2 else vocab     # keep partners in range
    else:
        vocab_draw = vocab
    ranks = _draw_ranks(seed, n_queries, max_terms, vocab_draw, skip_top, zipf_s)
    q = np.arange(n_queries, dtype=np.uint64)
    with np.errstate(over="ignore"):
        h = _mix_np(q * _U64(0x9E3779B97F4A7C15) + _U64(seed) + _U64(77))
    n_terms = (min_terms + (h % _U64(max_terms - min_terms + 1))).astype(np.int64)
    if mode == "mixed":
        is_and = ((h >> _U64(32)) & _U64(1)).astype(bool)
    else:
        is_and = np.full(n_queries, mode == "and")
    queries: List[Query] = []
    multi = len(fields) > 1
    for i in range(n_queries):
        subs = []
        for j in range(int(n_terms[i])):
            r = int(ranks[i, j])
            alts = [r, int(variant_partner(r, skip_top))] if variants else [r]
            leaves = [Term(f, a, boost=b) for a in alts for f, b in zip(fields, field_boosts)]
            subs.append(leaves[0] if len(leaves) == 1 else Or(leaves))
        if variants or is_and[i]:
            queries.append(And(subs) if len(subs) > 1 else subs[0])
        else:
            flat = []
            for s in subs:
                flat.extend(s.subqueries if isinstance(s, Or) else [s])
            queries.append(Or(flat) if len(flat) > 1 else flat[0])
    return QuerySet(queries, ranks, n_terms, is_and | variants)


# BASELINE.json configs (SURVEY.md §8 d): seeds 20260000 + config#, 20261000 + config#
CONFIGS = {
    1: dict(n_docs=10_000, vocab=50_000, n_queries=1_000, min_terms=2, max_terms=2, mode="and", k=10),
    2: dict(n_docs=1_000_000, vocab=200_000, n_queries=10_000, min_terms=2, max_terms=4, mode="mixed", k=10),
    3: dict(n_docs=1_000_000, vocab=200_000, n_queries=10_000, min_terms=4, max_terms=4, mode="and", k=10,
            variants=True, corpus_of=2),
    4: dict(n_docs=10_000_000, vocab=500_000, n_queries=100_000, min_terms=2, max_terms=4, mode="mixed", k=100),
    5: dict(n_docs=50_000_000, vocab=1_000_000, n_queries=1_000_000, min_terms=2, max_terms=4, mode="mixed",
            k=10, fields=("title", "body"), field_boosts=(2.0, 1.0)),
}


def config_corpus(cfg: int, device=None, n_docs: Optional[int] = None) -> FlatIndex:
    c = CONFIGS[cfg]
    corpus_cfg = c.get("corpus_of", cfg)
    specs = (TITLE, BODY) if "fields" in c else (BODY,)
    return make_corpus(n_docs or c["n_docs"], c["vocab"], 20260000 + corpus_cfg, specs, device=device)


def config_queries(cfg: int, n_queries: Optional[int] = None) -> QuerySet:
    c = CONFIGS[cfg]
    return make_queries(n_queries or c["n_queries"], c["vocab"], 20261000 + cfg, c["min_terms"], c["max_terms"],
                        c["mode"], fields=c.get("fields", ("body",)), field_boosts=c.get("field_boosts", (1.0,)),
                        variants=c.get("variants", False))
