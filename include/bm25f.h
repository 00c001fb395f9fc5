/*
 * bm25f.h — C ABI of libbm25f.so, the B200-native BM25F scoring + top-k engine.
 *
 * This is the drop-in boundary for one hot path of CodeOptimist/document-search-engine.
 * The reference is pure Python on top of Whoosh 2.7.4 (reference requirements.txt:6); it
 * has no FFI of its own, so the entry points below are what a ctypes binding for the
 * scoring path replaces, call site by call site:
 *
 *   bm25f_create / bm25f_destroy
 *       <- the index handle the front ends keep for the life of the process:
 *          `ix = my_index.get_idx('index')`            reference my_flask.py:549, cli.py:25
 *          (open at my_index.py:226-234).  create uploads the flattened index to HBM once.
 *   bm25f_set_weighting
 *       <- `ix.searcher(weighting=BM25F | AscDateBM25F | DescDateBM25F)`
 *                                                      reference my_flask.py:183-184
 *          (B, K1, per-field B and the corpus avgfl are folded into per-field norm tables).
 *   bm25f_search_batch  (= bm25f_prepare_arena + bm25f_execute + bm25f_fetch)
 *       <- `searcher.search_page(qp, pagenum, pagelen)` reference my_flask.py:208, :211
 *          `searcher.search(qp, limit=3)`               reference my_flask.py:304
 *          `ix.searcher().search(Every('session'), limit=None)`   reference cli.py:9
 *          i.e. Whoosh Searcher.search -> matcher tree -> BM25FScorer -> TopCollector.
 *   bm25f_merge_keys / bm25f_decode_keys
 *       <- Whoosh's multi-segment collection (global docnum = segment offset + local docnum,
 *          one collector over all segments); here: merge of per-GPU local top-k lists
 *          after the NCCL all-gather.
 *   bm25f_plan_gather_span / bm25f_merge_gathered
 *       <- the same, as one exchange: the plan's keys and match counts are one device span (one all-gather), then
 *          merge + decode + sum of the counts in one call.
 *   bm25f_set_final_date / bm25f_fetch_final / bm25f_merge_final_lists
 *       <- `DateBM25F.final()` of the reference's date-ordered weightings   reference my_whoosh.py:127-154
 *   bm25f_put_positions / bm25f_phrase_lists
 *       <- Whoosh's Phrase matcher (quoted phrases of the search form, reference templates/search-form.html:20-40):
 *          the fields' word order lives in HBM, a positional filter on the device finds the documents that pass,
 *          and they become posting lists of one batch.  (bm25f_put_lists takes such lists found elsewhere.)
 *   bm25f_submit / bm25f_collect
 *       <- no counterpart in the reference (one request at a time): two batches in flight for servers that batch.
 *   bm25f_get_stats
 *       <- `Results.runtime` (Whoosh records wall time per search; the reference never reads it).
 *
 * Conventions: every function returns 0 on success or a negative BM25F_E* code; the message
 * is available from bm25f_last_error() (thread-local).  No exceptions or abort() cross this
 * boundary.  A handle is not thread-safe: one in-flight call per handle.  The caller owns all
 * host buffers; the library copies what it needs and owns all device memory until destroy.
 * Pointers in bm25f_index_desc may be host or device pointers (the copy uses UVA);
 * term_offsets and term_field must be host pointers.
 */
#ifndef BM25F_H_
#define BM25F_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BM25F_ABI_VERSION 3

#define BM25F_OK          0
#define BM25F_EINVAL     -1   /* bad argument */
#define BM25F_ECUDA      -2   /* CUDA runtime error */
#define BM25F_ENCCL      -3   /* reserved: collective error (collectives run in the host layer) */
#define BM25F_ENOMEM     -4   /* out of (device or host) memory */
#define BM25F_EABI       -5   /* ABI version mismatch */

#define BM25F_MAX_LEAVES_PER_QUERY 256
#define BM25F_MAX_K               1024
#define BM25F_TERM_UNKNOWN 0xFFFFFFFFu  /* leaf_term value for a term/field not in the index (empty matcher) */
#define BM25F_GROUP_NOT 0xFFu            /* leaf_group value of a leaf inside a NOT clause: its documents are excluded from
                                            the query's matches and it contributes no score (Whoosh AndNot); such leaves
                                            come last in the query (groups are non-decreasing) */
#define BM25F_TERM_EVERY_BASE 0xFFFFFF00u  /* leaf_term = BASE + field: Whoosh's Every(field) - every live document
                                              that has the field, constant score = leaf_weight (reference cli.py:9) */

typedef struct bm25f_handle bm25f_handle;
typedef struct bm25f_plan bm25f_plan;

/* Flattened index of one document shard (SURVEY.md §8 b). */
typedef struct {
  uint32_t abi_version;          /* must be BM25F_ABI_VERSION */
  uint32_t n_fields;
  uint64_t n_docs_all;           /* documents in this shard, deleted ones included */
  uint64_t n_terms;              /* posting lists; a "term" is a (field, text) pair */
  uint64_t n_postings;
  uint64_t doc_base;             /* global docnum of local document 0 (Whoosh segment offset) */
  const uint64_t* term_offsets;  /* [n_terms + 1] CSR row pointers (host) */
  const uint8_t*  term_field;    /* [n_terms] field index of every posting list (host) */
  const uint32_t* docids;        /* [n_postings] local docids, ascending inside a term */
  const float*    tfs;           /* [n_postings] posting weights (term count x field boost) */
  const uint8_t*  len_bytes;     /* [n_fields * n_docs_all] quantised field lengths */
  const uint8_t*  deleted;       /* [n_docs_all] 1 = deleted, or NULL */
} bm25f_index_desc;

/* Engine options; zero means "library default". */
typedef struct {
  uint32_t tile_docs;            /* documents per shared-memory score tile (<= 65536) */
  uint32_t threads;              /* threads per CTA of the scoring kernel */
  uint32_t split_postings;       /* target postings per work item */
  uint32_t variant;              /* scoring kernel: 0 = auto (where eligible - k <= 256, <= 8 leaves, positive
                                    weights, no paging bound - flat ORs on warp streams (small ones by
                                    candidate-driven lookups), ANDs whose smallest
                                    group is far sparser than the rest by candidate-driven lookups, other
                                    ANDs on warp teams; else the bulk-copy pipeline),
                                    1 = bulk-copy pipeline, 2 = direct loads, 3 = warp streams,
                                    4 = warp teams (same eligibility as 3),
                                    5 = candidate-driven lookups for every eligible query (<= 32 leaves) */
  uint32_t chunk_postings;       /* pipeline: postings per shared-memory stage (multiple of 16) */
  uint32_t stages;               /* pipeline: ring depth (2..32) */
  uint32_t subtile_docs;         /* stream kernel: documents per warp-private sub-range of a flat OR
                                    (4-byte accumulators; AND queries use half as many 8-byte slots);
                                    multiple of 128 */
  uint32_t warp_split;           /* stream kernel: target work (posting-equivalents) per work item */
  uint32_t stream_warps;         /* stream kernel: warps (independent workers) per CTA, 1..16 */
  uint32_t prefetch_postings;    /* stream kernel: bulk L2 prefetch distance (multiple of 512;
                                    0xFFFFFFFF = off; also switches the tile kernel's prefetch) */
  uint32_t cta_warps;            /* team kernel: warps per CTA, 1..16 */
  uint32_t cta_prefetch;         /* team kernel: slices ahead to bulk-prefetch into L2 (0xFFFFFFFF = off) */
  uint32_t cta_split;            /* team kernel: target work (posting-equivalents) per work item */
  uint32_t cta_slice_docs;       /* team kernel: documents per warp-private slice of a flat OR (AND: half);
                                    multiple of 128 */
  uint32_t isect_ratio;          /* candidate-driven AND: used when (postings of the smallest group) x
                                    (leaves - 1) x isect_ratio < postings of the query; default 1 */
  uint32_t isect_split;          /* candidate-driven AND: target candidates per work item; default 2048 */
  uint32_t isect_or_limit;       /* a flat OR goes the candidate-driven way when postings x (leaves - 1) is
                                    below this (0xFFFFFFFF = never); default 40000 x n_docs_all / 1e6, within
                                    2000..40000: the sweep it avoids is as long as the shard's document space */
  uint32_t serial_streams;       /* 1: the candidate-driven / team kernels run after, not beside, the flat-OR kernel */
  uint32_t host_plan;            /* 1: always plan batches on the host (default: batches of >= 256 queries that the warp
                                    kernels serve alone - <= 8 leaves a query, positive weights, no NOT clause, no paging
                                    bound, no final() step, k <= 256 - are planned by three small kernels on the device) */
  uint32_t compact_store;        /* 1: release the raw postings (docid, tf, length byte: 8 of the 16 bytes a posting) after
                                    the first bm25f_set_weighting; the handle then serves that weighting only, and only
                                    queries the warp kernels take (k <= 256, <= 32 leaves, positive weights, no paging
                                    bound past BM25F_MAX_K) - anything else is a loud BM25F_EINVAL */
  uint32_t filter_postings;      /* room for the per-batch document lists of bm25f_put_lists, in postings (8 bytes each);
                                    default 1 << 20 */
} bm25f_options;

/* A batch of lowered queries: every query is an AND of groups, every group an OR of leaves
 * (an OR query is the one-group case).  Leaves of a query are contiguous and sorted by group. */
typedef struct {
  uint32_t n_queries;
  uint32_t n_leaves;
  const uint32_t* query_leaf_offsets;  /* [n_queries + 1] */
  const uint8_t*  query_n_groups;      /* [n_queries]; 0 = null query (matches nothing) */
  const uint32_t* leaf_term;           /* [n_leaves] posting-list id or BM25F_TERM_UNKNOWN */
  const float*    leaf_weight;         /* [n_leaves] idf * (K1 + 1) * boost, rounded from float64 */
  const uint8_t*  leaf_group;          /* [n_leaves] group index inside the query, or BM25F_GROUP_NOT */
  const uint64_t* after_keys;          /* [n_queries] or NULL: only hits ordered strictly after this
                                          key are collected (paging past BM25F_MAX_K); 0 = no bound.
                                          While a final() step is set the bound is the 96-bit key of the last hit already
                                          returned: after_keys = the float64 final value made orderable (sign bit set for
                                          v >= 0, all bits inverted for v < 0), after_lo = 0xFFFFFFFF - its docnum */
  const uint32_t* after_lo;            /* [n_queries] or NULL (see after_keys) */
} bm25f_query_batch;

typedef struct {
  uint64_t postings_touched;     /* sum over leaves of live df, last execute */
  uint64_t n_items;              /* work items of the last execute */
  uint64_t n_launches;           /* kernels launched by the last execute */
  uint64_t n_executes;           /* executes folded into the ms_* sums since the last reset */
  float    ms_bounds;            /* summed device time of the tile-boundary kernel (CUDA events; CTA kernels only) */
  float    ms_score;             /* summed device time of the scoring + top-k kernel */
  float    ms_merge;             /* summed device time of the merge + decode kernels */
  float    ms_total;             /* summed first-launch-to-last-kernel-end time */
  uint32_t tile_docs;
  uint32_t threads;
  uint32_t ctas_per_sm;
  uint32_t packed_payload;       /* 1: (tf,lb) packed in 32 bits; 0: float tf + length byte */
  uint64_t device_bytes;         /* device memory held by the index */
  /* last execute, algorithmic postings (sum of live df over leaves) per kernel class: */
  uint64_t postings_stream;      /* k_score_stream: every posting is read and accumulated */
  uint64_t postings_team;        /* k_score_team: every posting of the slices not skipped is read */
  uint64_t postings_cta;         /* k_score_pipe / k_score_topk */
  uint64_t postings_lookup;      /* k_score_isect: postings of the smallest group are read, the other lists are
                                    searched (skip_to), so most of these postings are NOT read */
  uint64_t reserved0;
  float    ms_stream;            /* summed device time of k_score_stream alone (it overlaps k_score_isect) */
  uint32_t reserved1;
} bm25f_stats;

int  bm25f_abi_version(void);
const char* bm25f_last_error(void);

int  bm25f_create(const bm25f_index_desc* desc, int device, const bm25f_options* opts, bm25f_handle** out);
void bm25f_destroy(bm25f_handle* h);

/* norm: [n_fields * 256] float32, norm[f][b] = K1 * ((1 - B_f) + B_f * fl(b) / avgfl_f).
 * A row of 256 x -1.0 marks a field that is not scorable (Whoosh: schema[field].scorable is false, e.g. the
 * reference's `book` ID field, my_index.py:152): BM25F.scorer() gives its terms a WeightScorer, the score of a
 * posting is its weight x the leaf weight (which the caller then sets to the query boost alone: no idf). */
int  bm25f_set_weighting(bm25f_handle* h, const float* norm);

/* A weighting with a final() step (reference my_whoosh.py:127-154, DescDateBM25F / AscDateBM25F, selected at
 * my_flask.py:183): Whoosh applies final(searcher, docnum, score) to EVERY match before the top-k collector.
 * date_add: [n_docs_all] float64, for a dated document (its date score in seconds + 1.0), NaN for a document
 * without a date.  While set, a match with BM25F score s ranks by the float64 value
 *     v = 1 - 1/s                      (no date)
 *     v = ((1 - 1/s) + date_add) / 1e9 (dated)
 * descending, docnum ascending; plans are fetched with bm25f_fetch_final (which returns v), k <= 256 per pass
 * (deeper pages: another pass with after_keys / after_lo), at most 32 leaves per query, and
 * bm25f_search_batch / bm25f_submit / bm25f_fetch are refused.  NULL switches the step off again. */
int  bm25f_set_final_date(bm25f_handle* h, const double* date_add);

/* Host planning + upload of one batch.  The plan can be executed any number of times. */
int  bm25f_prepare(bm25f_handle* h, const bm25f_query_batch* batch, int k, bm25f_plan** out);
/* Same, but the plan's buffers live in the handle's reusable workspaces (no allocation): the plan is valid
 * until the second next bm25f_prepare_arena / bm25f_search_batch / bm25f_submit on this handle (there are two
 * workspaces, used alternately).  This is what the sharded host layer
 * uses per batch (the per-GPU half of `Searcher.search`, reference my_flask.py:208, :211, :304). */
int  bm25f_prepare_arena(bm25f_handle* h, const bm25f_query_batch* batch, int k, bm25f_plan** out);
/* Launch the kernels of a plan on the handle's stream (asynchronous). */
int  bm25f_execute(bm25f_handle* h, bm25f_plan* plan);
/* Wait for the plan's kernels and copy the results to host buffers:
 * out_scores/out_docids [n_queries * k] (unused slots: -inf / 0xFFFFFFFF),
 * out_counts [n_queries] hits written, out_totals [n_queries] exact number of matching documents. */
int  bm25f_fetch(bm25f_handle* h, bm25f_plan* plan, float* out_scores, uint32_t* out_docids,
                 uint32_t* out_counts, uint64_t* out_totals);
/* bm25f_fetch for a plan prepared while a final() step was set: out_final [n_queries * k] float64 final
 * values (unused slots: -inf); the other outputs as bm25f_fetch. */
int  bm25f_fetch_final(bm25f_handle* h, bm25f_plan* plan, double* out_final, uint32_t* out_docids,
                       uint32_t* out_counts, uint64_t* out_totals);
/* Device-resident results of a plan: keys [n_queries * k] (0 = empty slot), totals [n_queries]. */
int  bm25f_plan_device_results(bm25f_plan* plan, uint64_t** d_keys, uint64_t** d_totals);
int  bm25f_synchronize(bm25f_handle* h);
/* Launch on the caller's stream (a cudaStream_t; e.g. the host framework's current stream) so the
 * caller's events and collectives order with the library's kernels.  NULL is the legacy default
 * stream.  use_own != 0 restores the library's own non-blocking stream. */
int  bm25f_set_stream(bm25f_handle* h, void* stream, int use_own);
void bm25f_plan_destroy(bm25f_plan* plan);

/* prepare + execute + fetch */
int  bm25f_search_batch(bm25f_handle* h, const bm25f_query_batch* batch, int k, float* out_scores,
                        uint32_t* out_docids, uint32_t* out_counts, uint64_t* out_totals);

/* Pipelined form of bm25f_search_batch (same reference call sites: my_flask.py:208, :211, :304) for a stream of
 * batches (a server answering request batches back to back): bm25f_submit plans the batch on the host, uploads
 * it on a copy stream, launches its kernels and the device-to-host copy of its results into pinned memory, and returns without waiting; bm25f_collect waits for
 * that batch, copies the results to the caller's buffers (same layout as bm25f_fetch) and frees the plan.
 * Two batches may be in flight (the handle has two workspaces), so the host side of batch i + 1 overlaps the
 * GPU side of batch i; a third bm25f_submit before the oldest is collected is refused (BM25F_EINVAL), and
 * batches are collected in submission order (a refused bm25f_collect leaves the batch in flight; any other
 * outcome frees the plan).  The query arrays may be reused as soon as bm25f_submit returns. */
int  bm25f_submit(bm25f_handle* h, const bm25f_query_batch* batch, int k, bm25f_plan** out);
int  bm25f_collect(bm25f_handle* h, bm25f_plan* plan, float* out_scores, uint32_t* out_docids,
                   uint32_t* out_counts, uint64_t* out_totals);

/* Merge n_lists device-resident top-k key lists per query (layout [n_lists][n_queries][k], as an
 * all-gather of per-shard results produces: every list in descending key order, empty slots 0 at its end, which
 * is how bm25f_execute and this call write them) into d_out_keys [n_queries][k].  Runs on `stream`
 * (a cudaStream_t, or NULL for the handle's current stream). */
int  bm25f_merge_keys(bm25f_handle* h, const uint64_t* d_keys, int n_lists, uint32_t n_queries, int k,
                      uint64_t* d_out_keys, void* stream);
/* The exchange step of a document-sharded batch with ONE collective: a plan keeps its
 * [n_queries * k] keys and its [n_queries] match counts in one span of 64-bit words (bm25f_plan_gather_span: first word,
 * length, offset of the counts), so a single all-gather of that span moves both; bm25f_merge_gathered then merges the
 * n_lists key lists per query (W11 order, as Whoosh's one collector over all segments), adds up the counts and decodes:
 * d_keys [n_queries * k] merged keys, d_scores / d_docids [n_queries * k], d_counts / d_totals [n_queries]. */
int  bm25f_plan_gather_span(bm25f_plan* plan, uint64_t** d_base, uint64_t* span_words, uint64_t* totals_offset_words);
int  bm25f_merge_gathered(bm25f_handle* h, const uint64_t* d_gathered, int n_lists, uint64_t span_words,
                          uint64_t totals_offset_words, uint32_t n_queries, int k, uint64_t* d_keys, float* d_scores,
                          uint32_t* d_docids, uint32_t* d_counts, uint64_t* d_totals, void* stream);
/* Final mode (my_whoosh.py:127-154) across document shards (Whoosh segments with doc offsets, W8).
 * bm25f_plan_device_final: the device-resident results of a plan
 * prepared under a final() step (final values [n_queries * k] float64, global docnums [n_queries * k] with
 * 0xFFFFFFFF in unused slots, totals [n_queries]).  bm25f_merge_final_lists merges n_lists such result lists
 * per query (layout [n_lists][n_queries][k], as an all-gather over the shards produces) into the k best by
 * (final value descending, docnum ascending) and counts them.  k <= 256. */
int  bm25f_plan_device_final(bm25f_plan* plan, double** d_final, uint32_t** d_docids, uint64_t** d_totals);
int  bm25f_merge_final_lists(bm25f_handle* h, const double* d_vals, const uint32_t* d_docids, int n_lists,
                             uint32_t n_queries, int k, double* d_out_final, uint32_t* d_out_docids,
                             uint32_t* d_out_counts, void* stream);
/* Decode device keys to device arrays of scores / docids / counts (any may be NULL). */
int  bm25f_decode_keys(bm25f_handle* h, const uint64_t* d_keys, uint32_t n_queries, int k,
                       float* d_scores, uint32_t* d_docids, uint32_t* d_counts, void* stream);

/* Timings are folded in by bm25f_synchronize / bm25f_fetch. */
/* Per-batch document lists (phrase queries: reference search-form.html:20-40, `"dead sea"`; Whoosh query.Phrase).
 * Whoosh scores a phrase as the AND of its words and lets the positions decide only WHETHER a document matches; the
 * host finds the documents that pass the positional test and hands them over as posting lists with impact 1: list i of
 * this call is leaf_term `*first_term + i` until the next call replaces them all.  A phrase is then the query
 * And(words..., its list) with a tiny positive weight (e.g. 1e-29) on the list's leaf.  Such leaves are served by
 * every kernel (the CTA kernels too: k > 256, more than 32 leaves, paging bounds); docids are local, strictly
 * ascending, < n_docs_all; `offsets` [n_lists + 1] starts at 0.  Waits for the handle's stream; refused while a
 * submitted batch is in flight. */
#define BM25F_MAX_FILTER_LISTS 4096
int  bm25f_put_lists(bm25f_handle* h, uint32_t n_lists, const uint64_t* offsets, const uint32_t* docids, uint32_t* first_term);

/* Word order of one field for the positional filter (Whoosh: the positions of a TEXT(phrase=True) field, reference
 * my_index.py:172-177), document-major as FlatIndex.positions holds it: document d's tokens, as posting-list ids in
 * document order, are tokens[doc_offsets[d] .. doc_offsets[d + 1]) (doc_offsets [n_docs_all + 1] starts at 0 and never
 * decreases; a token that is no posting list of the field may be any other value, e.g. 0xFFFFFFFF).  Host pointers,
 * copied.  A second call for the same field replaces the first; the bytes count in device_bytes.  4 bytes a token. */
int  bm25f_put_positions(bm25f_handle* h, uint32_t field, const uint64_t* doc_offsets, const uint32_t* tokens);
/* The positional filter (reference: quoted phrases, search-form.html:20-40; `searcher.search_page(qp, ...)` of a query
 * that holds them, my_flask.py:208, :211).  Phrase i is words[word_offsets[i] .. word_offsets[i + 1]) (posting-list
 * ids of one field whose word order was uploaded, at most 32; BM25F_TERM_UNKNOWN makes the list empty) with slops[i]:
 * a live document matches iff kept_{n-1} is not empty, where kept_0 = the positions of word 0 and kept_j = the
 * positions p of word j with some e in kept_{j-1}, 1 <= p - e <= slop.  The candidates are the live postings of the
 * phrase's rarest word.  Afterwards the handle is in the state bm25f_put_lists leaves it in, with phrase i's matches
 * (ascending) as list i: leaf_term `*first_term + i`.  Same limits (BM25F_MAX_FILTER_LISTS, option filter_postings)
 * and the same waits and refusals as bm25f_put_lists. */
int  bm25f_phrase_lists(bm25f_handle* h, uint32_t n_phrases, const uint32_t* word_offsets, const uint32_t* words,
                        const uint32_t* slops, uint32_t* first_term);

int  bm25f_get_stats(bm25f_handle* h, bm25f_stats* out);
int  bm25f_reset_stats(bm25f_handle* h);

#ifdef __cplusplus
}
#endif
#endif /* BM25F_H_ */
