#!/usr/bin/env python
"""Benchmark of the BM25F scoring + top-k hot path (BASELINE.json metric).

``python bench.py --gpus N --steps K --warmup W`` prints ONE JSON line on rank 0.

A *step* is one pass of the hot path over one batch of synthetic queries:
BASELINE.json ``configs[1]`` — 1M synthetic documents (Zipf vocabulary 200k), 10k batched
2-4-term AND/OR queries, top-10.  For N > 1 (one process per GPU, launched by torchrun) the same
corpus is document-sharded over the ranks and the local top-k lists are merged after an NCCL
all-gather, so total work is fixed (``"scaling": "strong"``).

* ``value``   queries/s with the packed query batch and the plan already resident in HBM;
              timed with CUDA events on the launching stream, max over ranks.
* ``e2e``     the same metric with HOST buffers: host planning, H2D of the batch, kernels,
              (all-gather + merge), D2H of the results, every step, all inside the timed region.
              ``e2e.value`` goes through the pipelined entry (``bm25f_submit`` / ``bm25f_collect``
              at N = 1, ``ShardedSearcher.search_packed_stream`` at N > 1: two batches in flight,
              the host side of step i + 1 overlaps the GPU side of step i); ``e2e.serial_value``
              is one blocking ``bm25f_search_batch`` / ``search_packed`` per step.  Wall clock,
              max over ranks, median of three repetitions of ``--steps`` steps.
* ``roofline`` achieved algorithmic posting bytes/s of the scoring kernel (9 B per posting
              touched, SURVEY.md §8 d) from the library's CUDA events around that kernel, over the
              same timed steps, against the measured HBM copy bandwidth in MEASURED_PEAKS.json.
* ``cpu_baseline`` the oracle's doc-at-a-time Whoosh-semantics port (``oracle/whoosh_port.py``;
              Whoosh itself is pure Python and not installable here) on a bounded query sample,
              one worker process per host core.

``--impl reference`` times that CPU port alone (the reference's own implementation of the path
is Whoosh, which is absent; see DESIGN.md) on the same config/metric/unit.

``--dump-outputs DIR`` writes what the last timed step of ``value`` returned (``scores`` float32 [Q, k], 0 in the
empty slots past ``counts``; ``docids``, ``counts`` and ``totals`` as float64) to ``DIR/<name>.npy``; the inputs
depend only on the arguments, so two builds of the library can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_POSTING = 9.0      # u32 docid + f32 weight + u8 length byte (SURVEY.md §8 d)
FALLBACK_HBM_GBS = 6650.0    # B200_PROFILING.md fallback if MEASURED_PEAKS.json is absent


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------------------------
# CPU baseline (the oracle port; the only place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------
_CPU_IX = None
_CPU_K = 10


def _cpu_worker(queries):
    from oracle.whoosh_port import OracleSearcher
    s = OracleSearcher(_CPU_IX)
    t = time.perf_counter()
    n = 0
    for q in queries:
        s.search(q, limit=_CPU_K)
        n += 1
    return n, time.perf_counter() - t


def cpu_baseline(ix, queries, k, target_seconds=15.0, cores=None):
    """Whole-machine throughput of the Whoosh-semantics port on a bounded sample."""
    global _CPU_IX, _CPU_K
    _CPU_IX, _CPU_K = ix, k
    cores = cores or os.cpu_count() or 1
    # pilot on one core to size the sample
    pilot = queries[:8]
    _, dt = _cpu_worker(pilot)
    per_q = max(dt / len(pilot), 1e-6)
    n = int(min(len(queries), max(cores * 4, target_seconds * cores / per_q)))
    sample = queries[:n]
    chunks = [sample[i::cores] for i in range(cores)]
    chunks = [c for c in chunks if c]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(len(chunks)) as pool:
        done = pool.map(_cpu_worker, chunks)
    wall = time.perf_counter() - t0
    nq = sum(d[0] for d in done)
    return {"value": nq / wall, "unit": "queries/s", "cores": len(chunks), "kind": "port",
            "sample": "first %d of the step's queries, doc-at-a-time Python port of Whoosh 2.7.4 semantics "
                      "(oracle/whoosh_port.py), %d fork workers, %.1f s wall" % (nq, len(chunks), wall)}


# ----------------------------------------------------------------------------------------------
# clocks
# ----------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1]))
                mx.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


#: --dump-outputs writes at most this many bytes; a larger batch is cut to a fixed, seeded sample of its queries
DUMP_LIMIT_BYTES = 64_000_000 - 65_536       # (minus room for the .npy headers)


def step_outputs(b):
    """Host copies of what ``ShardedSearcher.run_plan`` hands its caller, per query: the top-k scores and docids in
    W11 order, the length of that list and the match count.  Slots past the list's length (a query with fewer than k
    matches) are decoded as score -inf and docid 0xFFFFFFFF; their score is written as 0 so that every value is
    finite, and ``counts`` tells which slots hold hits."""
    Q = b["totals"].numel()
    k = b["scores"].numel() // Q
    scores = b["scores"].cpu().numpy().reshape(Q, k)
    counts = b["counts"].cpu().numpy().view(np.uint32)
    live = np.arange(k)[None, :] < counts[:, None]
    return {"scores": np.where(live, scores, 0).astype(np.float32),
            "docids": b["docids"].cpu().numpy().view(np.uint32).reshape(Q, k).astype(np.float64),
            "counts": counts.astype(np.float64),
            "totals": b["totals"].cpu().numpy().view(np.uint64).astype(np.float64)}


def write_outputs(path, arrays):
    """``path/<name>.npy`` per array.  Above DUMP_LIMIT_BYTES only the rows of a seeded sample of the queries are
    written, and their indices go to ``query_index.npy``."""
    Q = arrays["totals"].shape[0]
    row_bytes = sum(a[:1].nbytes for a in arrays.values())
    if Q * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(Q, DUMP_LIMIT_BYTES // (row_bytes + 8), replace=False))
        arrays = dict({name: a[rows] for name, a in arrays.items()}, query_index=rows.astype(np.float64))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


#: DRAM traffic is not measured inside a bench run (it needs ncu's counters, and a number taken under a profiler is
#: not a bench value): the line carries null and points at the dated capture of this same command
TRAFFIC_PROFILE = "profiles/r02_traffic.json (ncu --set full capture of this command: dram__bytes_read.sum + dram__bytes_write.sum per launch)"


def whoosh_module():
    """Real Whoosh (reference requirements.txt:6) if it can be imported here, also from a driver-provided install
    under baseline/_ref; None in this image."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    if os.path.isdir(ref) and ref not in sys.path:
        sys.path.append(ref)
    try:
        import whoosh
        return whoosh
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------
def workload(args):
    from document_search_engine_b200.corpus import CONFIGS
    c = dict(CONFIGS[args.config])
    if args.docs:
        c["n_docs"] = args.docs
    if args.queries:
        c["n_queries"] = args.queries
    if args.k:
        c["k"] = args.k
    return c


def config_json(args, c, world):
    return {"workload": "BASELINE configs[%d]: %d synthetic docs (Zipf s=1 vocab %d, lognormal(5,0.6) lengths), "
                        "%d batched %d-%d-term %s queries, top-%d" % (
                            args.config - 1, c["n_docs"], c["vocab"], c["n_queries"], c["min_terms"], c["max_terms"],
                            "AND-of-variant-OR" if c.get("variants") else {"mixed": "AND/OR", "and": "AND", "or": "OR"}[c["mode"]],
                            c["k"]),
            "n_docs": c["n_docs"], "n_queries": c["n_queries"], "k": c["k"],
            "sharding": "none" if world == 1 else "documents, %d contiguous ranges, NCCL all-gather of local top-k" % world,
            "l2": "inputs larger than L2: a step streams the batch's posting lists out of a %.2f GiB "
                  "device-resident index (L2 is 126 MB)"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from document_search_engine_b200.corpus import config_corpus, config_queries
    c = workload(args)
    t0 = time.perf_counter()
    ix = config_corpus(args.config, device="cpu" if not _cuda() else None, n_docs=c["n_docs"])
    qs = config_queries(args.config, c["n_queries"])
    log("reference arm: corpus ready in %.1f s" % (time.perf_counter() - t0))
    target = max(4.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    vals = []
    last = None
    if whoosh_module() is not None and c["n_docs"] <= 50_000:
        return run_reference_whoosh(args, c, ix, qs)
    for i in range(args.warmup + args.steps):
        # rotate the sample so steps do not re-time identical queries
        off = (i * 997) % max(1, len(qs.queries) - 1)
        sample = qs.queries[off:] + qs.queries[:off]
        last = cpu_baseline(ix, sample, c["k"], target_seconds=target)
        if i >= args.warmup:
            vals.append(last["value"])
    v = float(np.mean(vals))
    cfg = config_json(args, c, 1)
    cfg["l2"] = "n/a (CPU)"
    last["value"] = v
    out = {"impl": "reference", "metric": "BM25F top-%d queries/sec" % c["k"], "value": v, "unit": "queries/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": 1000.0 * c["n_queries"] / v, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": cfg, "cpu_baseline": last,
           "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "note": "Whoosh 2.7.4 (pure Python, reference requirements.txt:6) is not installable here; this is the "
                   "oracle's doc-at-a-time port of its semantics on all host cores; each step is a bounded "
                   "sample of the workload and ms_per_step is extrapolated to the full batch"}
    print(json.dumps(out), flush=True)
    return 0


def run_reference_whoosh(args, c, ix, qs):
    """The reference arm on real Whoosh (only when it can be imported, and for corpora a pure-Python indexer can
    build in the bench's time: BASELINE configs[0]): index the corpus as 't%07d' tokens with a whitespace
    tokenizer, time searcher.search(q, limit=k) with weighting=BM25F (my_flask.py:183-184, :208) on one core."""
    import tempfile
    from whoosh import fields, index, query as wq, scoring
    from whoosh.analysis import SpaceSeparatedTokenizer
    docs = [[] for _ in range(ix.n_docs_all)]
    for tid in range(ix.n_terms):
        d, tf = ix.postings(tid)
        tok = "t%07d" % (tid - int(ix.term_field[tid]) * ix.vocab_size)
        for dn, n in zip(d.tolist(), tf.tolist()):
            docs[dn].extend([tok] * int(n))
    tmp = tempfile.mkdtemp(prefix="bm25f_whoosh_")
    wix = index.create_in(tmp, fields.Schema(body=fields.TEXT(analyzer=SpaceSeparatedTokenizer(), phrase=False)))
    w = wix.writer()
    for toks in docs:
        w.add_document(body=" ".join(toks))
    w.commit()

    def conv(q):
        n = type(q).__name__
        if n == "Term":
            return wq.Term("body", "t%07d" % q.text, boost=q.boost)
        return {"And": wq.And, "Or": wq.Or}[n]([conv(s) for s in q.subqueries], boost=q.boost)
    wqs = [conv(q) for q in qs.queries]
    vals = []
    with wix.searcher(weighting=scoring.BM25F) as s:
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            for q in wqs:
                s.search(q, limit=c["k"])
            if i >= args.warmup:
                vals.append(len(wqs) / (time.perf_counter() - t0))
    v = float(np.mean(vals))
    cfg = config_json(args, c, 1)
    cfg["l2"] = "n/a (CPU)"
    cb = {"value": v, "unit": "queries/s", "cores": 1, "kind": "whoosh",
          "sample": "the whole batch through whoosh %s Searcher.search, one process" % getattr(__import__("whoosh"), "versionstring", lambda: "?")()}
    print(json.dumps({"impl": "reference", "metric": "BM25F top-%d queries/sec" % c["k"], "value": v, "unit": "queries/s",
                      "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * c["n_queries"] / v,
                      "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": cfg, "cpu_baseline": cb,
                      "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)
    return 0


def _cuda():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2)
    ap.add_argument("--docs", type=int, default=0)
    ap.add_argument("--queries", type=int, default=0)
    ap.add_argument("--k", type=int, default=0)
    ap.add_argument("--opt", action="append", default=[], metavar="NAME=VALUE",
                    help="engine option (a bm25f_options field, include/bm25f.h), e.g. --opt variant=3")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg")
    ap.add_argument("--check", type=int, default=200, help="queries checked against the oracle before timing")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's results (scores, docids, counts, totals) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.warmup < 3 and args.impl == "ours":
        log("note: the timing rules ask for >= 3 warm-up steps")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    from document_search_engine_b200.corpus import config_corpus, config_queries
    from document_search_engine_b200.scoring import BM25F
    from document_search_engine_b200.distributed import ShardedSearcher

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200; there is no CPU fallback for the product path")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log("note: --gpus %d but WORLD_SIZE %d; using WORLD_SIZE" % (args.gpus, world))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    c = workload(args)
    k = c["k"]

    t0 = time.perf_counter()
    ix = config_corpus(args.config, device="cuda:%d" % local_rank, n_docs=c["n_docs"])
    qs = config_queries(args.config, c["n_queries"])
    if rank == 0:
        log("corpus: %d docs, %d postings, generated in %.1f s" % (ix.n_docs_all, ix.n_postings, time.perf_counter() - t0))
    torch.cuda.empty_cache()
    t0 = time.perf_counter()
    # run on a side stream: the legacy default stream would serialise the library's second stream
    side = torch.cuda.Stream(device=local_rank)
    torch.cuda.set_stream(side)
    engine_opts = {}
    for o in args.opt:
        name, _, value = o.partition("=")
        engine_opts[name.strip()] = int(value, 0)
    ss = ShardedSearcher(ix, rank=rank, world=world, device=local_rank, weighting=BM25F, **engine_opts)
    eng = ss.engine
    batch = ss.pack(qs.queries)
    if rank == 0:
        log("upload + pack: %.1f s; engine %s" % (time.perf_counter() - t0, eng.stats()))

    # ---- parity gate on a sample before any number is reported --------------------------------
    if args.check:
        from oracle.numpy_oracle import NumpyOracle
        from tests.parity import assert_query_parity
        scores, docids, counts, totals = ss.search_packed(batch, k)
        if rank == 0:
            o = NumpyOracle(ix)
            step = max(1, len(qs.queries) // args.check)
            for i in range(0, len(qs.queries), step):
                n = int(counts[i])
                assert_query_parity(o, qs.queries[i], list(zip(scores[i, :n].tolist(), docids[i, :n].tolist())),
                                    int(totals[i]), k, ctx="bench query %d" % i)
            log("parity gate: %d sampled queries match the oracle" % len(range(0, len(qs.queries), step)))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: plan resident in HBM, CUDA events on the launching stream ----------------------
    plan = eng.prepare(batch, k)
    for _ in range(args.warmup):
        ss.run_plan(plan)
    barrier()
    eng.synchronize()
    eng.reset_stats()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for _ in range(args.steps):
        last = ss.run_plan(plan)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    # the result buffers are reused by the e2e legs below, so the last step's results are copied out now
    dumped = step_outputs(last) if args.dump_outputs and rank == 0 else None
    eng.synchronize()
    st = eng.stats()
    clk = clocks.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ms_per_step = ms / args.steps
    value = c["n_queries"] / (ms_per_step * 1e-3)

    # roofline of the dominant kernel (k_score_stream: the flat ORs, every posting read and accumulated):
    # algorithmic bytes of ITS items on this rank / ITS launch duration (CUDA events around that launch;
    # k_score_isect runs beside it on a second stream, so this is its duration under that sharing)
    peak, peak_src = measured_peak()
    nex = max(1, st["n_executes"])
    ms_score = st["ms_score"] / nex
    ms_stream = st["ms_stream"] / nex
    achieved = BYTES_PER_POSTING * st["postings_stream"] / (ms_stream * 1e-3) / 1e9 if ms_stream > 0 else 0.0
    roof_kernel = "k_score_stream (flat OR queries: every posting read once and accumulated)"
    roof_ms, roof_bytes = ms_stream, BYTES_PER_POSTING * st["postings_stream"]
    if st["postings_stream"] == 0 and st["postings_lookup"] > 0:
        # a workload without flat ORs (config 3: AND of OR groups): the candidate-driven kernel is the step
        roof_kernel = ("k_score_isect (AND queries: the smallest group's postings are read, the other lists are searched; "
                       "algorithmic bytes count every leaf's full list as SURVEY 8d does, so this is not a bandwidth claim)")
        roof_ms, roof_bytes = ms_score, BYTES_PER_POSTING * st["postings_lookup"]
        achieved = roof_bytes / (roof_ms * 1e-3) / 1e9 if roof_ms > 0 else 0.0
    step_gbs = BYTES_PER_POSTING * st["postings_touched"] / (ms_score * 1e-3) / 1e9 if ms_score > 0 else 0.0
    # kernels of the library per timed step: the plan's own launches, run_plan's decode of the (merged) keys,
    # and for N > 1 the merge of the gathered lists
    launches = (int(st["n_launches"]) + 1 + (1 if world > 1 else 0)) * args.steps

    # ---- e2e: host buffers through the public entry point ---------------------------------------
    h2d = batch.nbytes
    d2h = batch.n_queries * (k * 8 + 4 + 8)
    for _ in range(min(2, args.warmup)):
        ss.search_packed(batch, k) if world > 1 else eng.search_batch(batch, k)

    def median_of_three(run_steps):
        """Wall time of ``run_steps()`` (exactly ``--steps`` steps), max over ranks, median of three
        repetitions: the region is tens of milliseconds of host + GPU work, one host hiccup would
        otherwise move the figure by 10 %."""
        times = []
        for _ in range(3):
            barrier()
            eng.synchronize()
            t0 = time.perf_counter()
            run_steps()
            barrier()
            t = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            times.append(float(t.item()))
        return sorted(times)[1]

    def serial_steps():
        for _ in range(args.steps):
            if world > 1:
                ss.search_packed(batch, k)
            else:
                eng.search_batch(batch, k)

    def pipelined_steps():
        n_out = 0
        for res in ss.search_packed_stream((batch for _ in range(args.steps)), k):
            n_out += res[0].shape[0]
        assert n_out == c["n_queries"] * args.steps

    serial_value = c["n_queries"] * args.steps / median_of_three(serial_steps)
    # The same steps through the pipelined entry (N = 1: bm25f_submit / bm25f_collect; N > 1:
    # ShardedSearcher.search_packed_stream), two batches in flight: every step still plans its batch
    # from the host arrays, uploads it, and reads its results back into host arrays; the host side of
    # step i + 1 overlaps the GPU side of step i.
    # (untimed) the pipelined entry must return what the blocking one returns, batch after batch; a mismatch is
    # reported in the line (e2e.pipelined_check), it does not stop the measurement
    pipelined_check = "ok"
    want = ss.search_packed(batch, k) if world > 1 else eng.search_batch(batch, k)
    for got in ss.search_packed_stream((batch for _ in range(max(3, min(2, args.warmup)))), k):
        for name, g_, w_ in zip(("scores", "docids", "counts", "totals"), got, want):
            if name in ("scores", "docids"):
                live = np.arange(g_.shape[1])[None, :] < want[2][:, None]
                same = np.array_equal(g_[live], w_[live])
            else:
                same = np.array_equal(g_, w_)
            if not same and pipelined_check == "ok":
                pipelined_check = "MISMATCH: pipelined %s differ from the blocking call's" % name
                log(pipelined_check)
    e2e_value = c["n_queries"] * args.steps / median_of_three(pipelined_steps)
    e2e_extra = {"pipeline_depth": 2, "pipelined_check": pipelined_check, "serial_value": serial_value, "timing": "median of 3 repetitions of --steps steps",
                 "note": "value: search_packed_stream (N = 1: bm25f_submit / bm25f_collect), the host side of batch "
                         "i+1 overlaps the GPU side of batch i; serial_value: one blocking search per step"}
    plan.close()

    # The Whoosh-shaped entry: a list of Query objects in, Results out (Searcher.search_batch: lowering of the
    # trees, packing, the same C-ABI call, result objects on demand).  "warm": the same query objects as the step
    # before (their lowered form is remembered on them); "cold": fresh query objects every step.
    facade = None
    if world == 1:
        from document_search_engine_b200.corpus import config_queries as _cq
        searcher = ss.local

        def facade_steps(fresh):
            def run():
                for i in range(args.steps):
                    queries = _fresh[i] if fresh else qs.queries
                    res = searcher.search_batch(queries, limit=k)
                    assert len(res) == c["n_queries"] and res[0].scored_length() <= k
            return run
        _fresh = [_cq(args.config, c["n_queries"]).queries for _ in range(args.steps)]
        searcher.search_batch(qs.queries, limit=k)
        facade = {"warm_value": c["n_queries"] * args.steps / median_of_three(facade_steps(False))}
        t0 = time.perf_counter()
        facade_steps(True)()
        facade["cold_value"] = c["n_queries"] * args.steps / (time.perf_counter() - t0)
        facade["note"] = ("Searcher.search_batch(list of Query trees, limit) -> sequence of Results; warm: lowered forms "
                          "cached on the query objects, cold: new query objects every step (one repetition)")

    if rank == 0:
        cfg = config_json(args, c, world)
        cfg["l2"] = cfg["l2"] % (st["device_bytes"] / 2 ** 30)
        cfg["engine"] = {"options": engine_opts, "ctas_per_sm": st["ctas_per_sm"],
                         "packed_payload": bool(st["packed_payload"]), "work_items": int(st["n_items"]),
                         "kernels_per_step": int(st["n_launches"])}
        out = {"metric": "BM25F top-%d queries/sec" % k, "value": value, "unit": "queries/s", "n_gpus": world,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
               "e2e": dict({"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": int(h2d),
                            "d2h_bytes_per_step": int(d2h), "facade": facade}, **e2e_extra),
               "gpu_launches": launches,
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                            "frac": achieved / peak, "traffic": None, "traffic_profile": TRAFFIC_PROFILE, "peak_source": peak_src,
                            "kernel": roof_kernel,
                            "kernel_ms_per_step": roof_ms,
                            "algorithmic_bytes_per_launch": roof_bytes,
                            "frac_of_nominal_8000": achieved / 8000.0,
                            "whole_step": {"algorithmic_GBs": step_gbs, "frac": step_gbs / peak,
                                           "ms": ms_score, "algorithmic_bytes": BYTES_PER_POSTING * st["postings_touched"],
                                           "postings_by_kernel": {"k_score_stream": int(st["postings_stream"]),
                                                                  "k_score_isect": int(st["postings_lookup"]),
                                                                  "k_score_team": int(st["postings_team"]),
                                                                  "cta_kernels": int(st["postings_cta"])},
                                           "note": "the whole-step figure counts every leaf's full list (SURVEY 8d) although "
                                                   "k_score_isect, like Whoosh's IntersectionMatcher, reads only the smallest "
                                                   "group's postings and searches the other lists; it is not a bandwidth claim"}},
               "kernel_ms": {"bounds": st["ms_bounds"] / max(1, st["n_executes"]), "score": ms_score,
                             "stream_kernel": ms_stream,
                             "merge": st["ms_merge"] / max(1, st["n_executes"]),
                             # the rest of ms_per_step on rank 0: for N > 1 the all-gather of the shards' top-k lists
                             # and match counts (one NCCL collective) + bm25f_merge_gathered, waits for the slowest
                             # rank included; for N = 1 the device-to-device copy and decode of run_plan
                             "exchange_and_final_merge": max(0.0, ms_per_step - st["ms_total"] / max(1, st["n_executes"]))},
               "clocks": clk}
        if not args.no_cpu:
            out["cpu_baseline"] = cpu_baseline(ix, qs.queries, k)
        if dumped is not None:
            write_outputs(args.dump_outputs, dumped)
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
