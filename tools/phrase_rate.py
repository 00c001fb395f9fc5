#!/usr/bin/env python
"""Phrase queries on the config-2-sized corpus (1M documents, 200k words, word order kept): the host positional test
the engine used before (``FlatIndex.phrase_docs``) against the device filter (``bm25f_phrase_lists``), and what a
user sees: ``search(phrase, limit=10)`` latency, ``search_page(phrase, 2, 150)`` and ``search_batch`` throughput.

Phrases are 2-3 words cut from real adjacent tokens of sampled documents (ranks below 50 skipped), bucketed by the
document frequency of their rarest word: that word's live postings are the filter's candidates.

    python tools/phrase_rate.py [out.json]
"""
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from document_search_engine_b200 import BM25F, Phrase
from document_search_engine_b200 import _ffi
from document_search_engine_b200.corpus import make_corpus

BUCKETS = [(0, 1_000), (1_000, 10_000), (10_000, 100_000), (100_000, 1 << 40)]
SKIP_TOP = 50


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def cut_phrases(ix, n, seed):
    rng = np.random.default_rng(seed)
    offs, ids = ix.positions[0]
    out, seen = [], set()
    while len(out) < n:
        d = int(rng.integers(ix.n_docs_all))
        a, b = int(offs[d]), int(offs[d + 1])
        w = int(rng.integers(2, 4))
        if b - a < w:
            continue
        p = int(rng.integers(a, b - w + 1))
        ranks = tuple(ids[p:p + w].tolist())
        if min(ranks) < SKIP_TOP or ranks in seen:
            continue
        seen.add(ranks)
        out.append(Phrase("body", list(ranks)))
    return out


def rare_df(ix, p):
    return min(int(ix.df[ix.term_id("body", w)]) for w in p.words)


def pct(a):
    a = np.asarray(a, dtype=np.float64)
    return {"median": float(np.median(a)), "p90": float(np.percentile(a, 90)), "p99": float(np.percentile(a, 99)), "n": int(a.size)}


def main(out_path):
    if not torch.cuda.is_available():
        raise SystemExit("phrase_rate.py measures the device path: it needs a CUDA device")
    t0 = time.perf_counter()
    ix = make_corpus(1_000_000, 200_000, 20260002, positions=True)
    gen_s = time.perf_counter() - t0
    res = {"card": card(), "corpus": "make_corpus(1_000_000, 200_000, 20260002, positions=True)", "generate_s": gen_s,
           "tokens": int(ix.positions[0][1].size)}
    pool = cut_phrases(ix, 12_000, 5)
    dfs = np.array([rare_df(ix, p) for p in pool])
    by_bucket = {"%d-%d" % b: [p for p, df in zip(pool, dfs) if b[0] <= df < b[1]] for b in BUCKETS}
    res["bucket_sizes"] = {k: len(v) for k, v in by_bucket.items()}

    # the host positional test (the old path): ms per phrase, a sample of every bucket, at most ~60 s in all
    host = {}
    for k, ps in by_bucket.items():
        times = []
        for p in ps[:10]:
            t = time.perf_counter()
            ix.phrase_docs(p.fieldname, p.words, p.slop)
            times.append((time.perf_counter() - t) * 1e3)
            if sum(times) > 15_000:
                break
        host[k] = {"ms_mean": float(np.mean(times)) if times else None, "n": len(times),
                   "candidates_mean": float(np.mean([rare_df(ix, p) for p in ps[:len(times)]])) if times else None}
    res["host_phrase_docs"] = host

    with ix.searcher(weighting=BM25F, filter_postings=1 << 24) as s:
        eng = s.engine
        t = time.perf_counter()
        s.search(pool[0], limit=10)                                   # first phrase: uploads the word order
        res["first_phrase_with_upload_ms"] = (time.perf_counter() - t) * 1e3
        res["device_bytes"] = int(eng.stats()["device_bytes"])
        for p in pool[:50]:                                           # warm-up
            s.search(p, limit=10)
            s.search_page(p, 2, 150)

        # the filter alone: a host clock around a synchronised bm25f_phrase_lists call
        def filter_ms(ps, reps):
            words = [[ix.term_id("body", w) for w in p.words] for p in ps]
            slops = [p.slop for p in ps]
            eng.phrase_lists(words, slops)
            ts = []
            for _ in range(reps):
                eng.synchronize()
                t = time.perf_counter()
                eng.phrase_lists(words, slops)
                ts.append((time.perf_counter() - t) * 1e3)
            return float(np.median(ts))
        res["filter_one_phrase_ms"] = {k: (float(np.median([filter_ms([p], 3) for p in ps[:30]])) if ps else None)
                                       for k, ps in by_bucket.items()}
        res["filter_batch_ms"] = {"1000": filter_ms(pool[1000:2000], 5), "4000": filter_ms(pool[2000:6000], 3)}

        lat, lat_b = [], {k: [] for k in by_bucket}
        sample = pool[200:1200]
        for p in sample:
            t = time.perf_counter()
            s.search(p, limit=10)
            us = (time.perf_counter() - t) * 1e6
            lat.append(us)
            df = rare_df(ix, p)
            for (lo, hi), k in zip(BUCKETS, by_bucket):
                if lo <= df < hi:
                    lat_b[k].append(us)
        res["search_limit10_us"] = pct(lat)
        res["search_limit10_us_by_bucket"] = {k: pct(v) for k, v in lat_b.items() if v}
        pg = []
        for p in pool[1200:1500]:
            t = time.perf_counter()
            s.search_page(p, 2, 150)
            pg.append((time.perf_counter() - t) * 1e6)
        res["search_page_2_150_us"] = pct(pg)

        # throughput: batches of phrase queries (at most 4096 distinct phrases, BM25F_MAX_FILTER_LISTS, a call)
        def qps(qs, reps):
            s.search_batch(qs[:4000], limit=10)
            best = None
            for _ in range(reps):
                t = time.perf_counter()
                for a in range(0, len(qs), 4000):
                    s.search_batch(qs[a:a + 4000], limit=10)
                dt = time.perf_counter() - t
                best = dt if best is None else min(best, dt)
            return len(qs) / best
        res["search_batch_qps"] = {"1000": qps(pool[:1000], 5), "10000 (3 calls of <= 4000)": qps(pool[:10_000], 3)}
    txt = json.dumps(res, indent=1)
    print(txt)
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write(txt + "\n")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
