// libbm25f — B200-native BM25F scoring + top-k over a device-resident CSR posting store.
//
// Replaces the inside of Whoosh's Searcher.search() for Term/And/Or trees as the reference
// calls it (reference my_flask.py:184, :208, :211, :304; cli.py:9).  See include/bm25f.h for
// the boundary and DESIGN.md for the data layout and the kernels.
//
// Kernel inventory (all hand-written for sm_100a; DESIGN.md section 4 has the table):
//   k_check_tf / k_pack_postings          index upload: fold (tf, length byte) into one 32-bit payload
//   k_live_counts / k_compact_lists       index upload: drop the postings of deleted documents (W9)
//   k_impacts                             re-weighting: {docid, tf / (tf + norm)} pairs, the scoring store
//   k_score_stream    (stream.cuh)        flat ORs: independent warps, accumulators in shared memory
//   k_score_isect     (isect.cuh)         ANDs: candidate-driven lookups (IntersectionMatcher + skip_to)
//   k_score_team      (team.cuh)          symmetric ANDs: CTA-built bounds table, private slices
//   k_tile_bounds, k_score_pipe, k_score_topk   general fallback (k > 256, many leaves, paging, odd weights)
//   k_merge_topk_warp / k_merge_topk      merge of per-item (or per-GPU) top-k lists
//   k_decode_keys                         keys -> (score, docid, count)
#include "../../include/bm25f.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <vector>

namespace {

thread_local std::string g_err;

int fail(int code, const char* fmt, ...) __attribute__((format(printf, 2, 3)));
int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}

#define CU(x)                                                                               \
  do {                                                                                      \
    cudaError_t e_ = (x);                                                                   \
    if (e_ != cudaSuccess)                                                                  \
      return fail(e_ == cudaErrorMemoryAllocation ? BM25F_ENOMEM : BM25F_ECUDA, "%s: %s",   \
                  #x, cudaGetErrorString(e_));                                              \
  } while (0)

// ------------------------------------------------------------------------------------------
// Device-side records
// ------------------------------------------------------------------------------------------
struct LeafRec {            // 32 B
  unsigned long long off;   // first posting of the list
  uint32_t df;              // postings in the list (this shard)
  float w;                  // idf * (K1 + 1) * boost
  uint32_t norm_off;        // field * 256
  uint32_t group;           // group index after sorting groups by size
  uint32_t qleaf0;          // first leaf of the owning query (global leaf index)
  uint32_t qnl;             // leaves in the owning query
};

struct QueryRec {           // 32 B
  uint32_t leaf_begin;
  uint16_t n_leaves;
  uint16_t n_groups;
  uint32_t flags;           // bit0: one group, all weights > 0 -> "acc == 0" marks a fresh slot
  uint32_t after_lo;        // final mode: low part (~docnum) of the paging bound; after_key is its high part
  unsigned long long after_key;
  uint32_t part_begin;      // first partial top-k list of this query
  uint32_t n_parts;
};

struct ItemRec {            // 16 B
  uint32_t q;
  uint32_t tile_begin;
  uint32_t tile_end;
  uint32_t part;            // which partial list this item writes
};

constexpr uint32_t QF_SIMPLE_OR = 1u;
constexpr int MAXL = BM25F_MAX_LEAVES_PER_QUERY;
constexpr int FAST_MAX_K = 256;           // largest k of the warp kernels: 8 keys per lane (the reference's listing page asks for 150)

// W11 order as one unsigned 64-bit key: score descending, docnum ascending.  All keys of
// distinct documents are distinct, so "top-k by key" is exactly the reference collector.
__host__ __device__ __forceinline__ unsigned long long make_key(float score, uint32_t gdoc) {
#ifdef __CUDA_ARCH__
  uint32_t u = __float_as_uint(score);
#else
  uint32_t u;
  memcpy(&u, &score, 4);
#endif
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ((unsigned long long)u << 32) | (unsigned long long)(0xFFFFFFFFu - gdoc);
}

__host__ __device__ __forceinline__ float key_score(unsigned long long key) {
  uint32_t u = (uint32_t)(key >> 32);
  u = (u & 0x80000000u) ? (u & 0x7FFFFFFFu) : ~u;
#ifdef __CUDA_ARCH__
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}

__host__ __device__ __forceinline__ uint32_t key_doc(unsigned long long key) {
  return 0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull);
}

// ------------------------------------------------------------------------------------------
// Index upload kernels
// ------------------------------------------------------------------------------------------
// Posting weights are term counts in the reference's schema (no field_boost, SURVEY W7); when
// every weight is a positive integer < 2^24 the (tf, length byte) pair is packed in 32 bits.
__global__ void k_check_tf(const float* __restrict__ tfs, unsigned long long n, int* __restrict__ flag) {
  unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  int bad = 0;
  for (; i < n; i += stride) {
    float t = tfs[i];
    if (!(t >= 1.0f && t < 16777216.0f && t == floorf(t))) bad = 1;
  }
  if (bad) atomicOr(flag, 1);
}

// payload[i] = (tf << 8) | len_byte[field][docid]   (packed)   or float bits of tf + separate byte;
// postings of deleted documents get tf = 0, which the scoring kernels skip
__global__ void k_pack_postings(const uint32_t* __restrict__ docids, const float* __restrict__ tfs,
                                const uint8_t* __restrict__ len_bytes_field, const uint8_t* __restrict__ deleted,
                                unsigned long long begin, unsigned long long end, int packed,
                                uint32_t* __restrict__ payload, uint8_t* __restrict__ lb_out) {
  unsigned long long i = begin + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (; i < end; i += stride) {
    const uint32_t d = docids[i];
    uint32_t lb = len_bytes_field[d];
    float t = tfs[i];
    if (deleted != nullptr && deleted[d]) t = 0.0f;   // W9: the kernels skip tf == 0
    if (packed) {
      payload[i] = ((uint32_t)t << 8) | lb;
    } else {
      payload[i] = __float_as_uint(t);
      lb_out[i] = (uint8_t)lb;
    }
  }
}

// pairs[i] = {docid, impact} with impact = tf / (tf + norm[lb]) for the postings [begin, end) of one
// field (float64 divide, rounded once); refreshed whenever the weighting changes.
// score = leaf weight * impact.
//
// weight_only: the field is not scorable (Whoosh gives such a field's terms a WeightScorer: the score of a posting is
// its weight, no idf, no length norm - e.g. the reference's `book` ID field, my_index.py:152, :171): impact = tf.
__global__ void k_impacts(const uint32_t* __restrict__ docids, const uint32_t* __restrict__ payload, const uint8_t* __restrict__ lb,
                          const float* __restrict__ norm_field, unsigned long long begin, unsigned long long end,
                          int packed, int weight_only, uint2* __restrict__ pairs) {
  unsigned long long i = begin + blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
  for (; i < end; i += stride) {
    const uint32_t pl = payload[i];
    double tf;
    uint32_t b;
    if (packed) { tf = (double)(pl >> 8); b = pl & 255u; }
    else { tf = (double)__uint_as_float(pl); b = lb[i]; }
    const float u = tf > 0.0 ? (weight_only ? (float)tf : (float)(tf / (tf + (double)norm_field[b]))) : 0.0f;
    pairs[i] = make_uint2(docids[i], __float_as_uint(u));
  }
}

// The caller's promise about the posting lists (include/bm25f.h: docids < n_docs_all, ascending inside a list) is
// checked once at upload: an out-of-range docid would index the length bytes, the deleted flags and the kernels'
// accumulators out of bounds.  flag[0] = 1 + the first offending list (the smallest such list wins).
__global__ void k_check_docids(const uint32_t* __restrict__ docids, const unsigned long long* __restrict__ offs,
                               unsigned long long n_terms, uint32_t n_docs, unsigned long long* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  unsigned long long t = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) >> 5;
  const unsigned long long stride = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
  for (; t < n_terms; t += stride) {
    bool bad = false;
    const unsigned long long b = offs[t], e = offs[t + 1];
    for (unsigned long long i = b + lane; i < e; i += 32) {
      const uint32_t d = docids[i];
      if (d >= n_docs || (i > b && docids[i - 1] >= d)) bad = true;
    }
    if (__any_sync(0xFFFFFFFFu, bad) && lane == 0) atomicMin(flag, t + 1ull);
  }
}

// W9: postings of deleted documents never match.  They are removed from the device store at
// upload (df / dc used for idf stay the stored ones: those are host-side statistics).
__global__ void k_live_counts(const uint32_t* __restrict__ docids, const unsigned long long* __restrict__ offs,
                              unsigned long long n_terms, const uint8_t* __restrict__ deleted, uint32_t* __restrict__ counts) {
  const int lane = threadIdx.x & 31;
  unsigned long long t = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) >> 5;
  const unsigned long long stride = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
  for (; t < n_terms; t += stride) {
    uint32_t c = 0;
    for (unsigned long long i = offs[t] + lane; i < offs[t + 1]; i += 32) c += deleted[docids[i]] ? 0u : 1u;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xFFFFFFFFu, c, o);
    if (lane == 0) counts[t] = c;
  }
}

__global__ void k_compact_lists(const uint32_t* __restrict__ docids, const float* __restrict__ tfs,
                                const unsigned long long* __restrict__ offs, const unsigned long long* __restrict__ new_offs,
                                unsigned long long n_terms, const uint8_t* __restrict__ deleted,
                                uint32_t* __restrict__ out_docids, float* __restrict__ out_tfs) {
  const int lane = threadIdx.x & 31;
  unsigned long long t = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) >> 5;
  const unsigned long long stride = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
  for (; t < n_terms; t += stride) {
    unsigned long long w = new_offs[t];
    const unsigned long long e = offs[t + 1];
    for (unsigned long long i0 = offs[t]; i0 < e; i0 += 32) {
      const unsigned long long i = i0 + lane;
      uint32_t d = 0;
      bool keep = false;
      if (i < e) { d = docids[i]; keep = !deleted[d]; }
      const unsigned m = __ballot_sync(0xFFFFFFFFu, keep);
      if (keep) {
        const unsigned long long o = w + __popc(m & ((1u << lane) - 1u));
        out_docids[o] = d;
        out_tfs[o] = tfs[i];
      }
      w += __popc(m);
    }
  }
}

// ------------------------------------------------------------------------------------------
// Tile boundaries: bounds[q][j][l] = first posting of leaf l with docid >= j * S
// ------------------------------------------------------------------------------------------
__global__ void k_tile_bounds(const LeafRec* __restrict__ leaves, uint32_t n_leaves, uint32_t T,
                              uint32_t S, const uint32_t* __restrict__ docids,
                              uint32_t* __restrict__ bounds) {
  unsigned long long gid = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x;
  unsigned long long total = (unsigned long long)n_leaves * (T + 1);
  if (gid >= total) return;
  uint32_t leaf = (uint32_t)(gid / (T + 1));
  uint32_t j = (uint32_t)(gid % (T + 1));
  LeafRec L = leaves[leaf];
  uint32_t lo = 0, hi = L.df;
  if (j == T) {
    lo = L.df;
  } else if (j > 0) {
    unsigned long long target = (unsigned long long)j * S;
    const uint32_t* d = docids + L.off;
    while (lo < hi) {
      uint32_t mid = (lo + hi) >> 1;
      if ((unsigned long long)__ldg(d + mid) < target) lo = mid + 1; else hi = mid;
    }
  }
  size_t base = (size_t)L.qleaf0 * (T + 1);
  bounds[base + (size_t)j * L.qnl + (leaf - L.qleaf0)] = lo;
}

// ------------------------------------------------------------------------------------------
// A "team" is the set of threads that cooperate on one work item: the whole CTA (barrier 0) in
// k_score_topk, the consumer warps (named barrier 1) in k_score_pipe.
// ------------------------------------------------------------------------------------------
struct Team {
  int tid;   // rank inside the team
  int nt;    // team size (multiple of 32)
  int bar;   // hardware barrier id
  __device__ __forceinline__ void sync() const {
    asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(nt) : "memory");
  }
};

// Shared-memory bitonic sort (descending) of n = 2^m keys by all threads of the team
__device__ void bitonic_sort_desc(unsigned long long* a, int n, const Team& tm) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tm.tid; i < n; i += tm.nt) {
        int x = i ^ j;
        if (x > i) {
          unsigned long long ai = a[i], ax = a[x];
          bool desc = (i & k) == 0;
          if (desc ? (ai < ax) : (ai > ax)) { a[i] = ax; a[x] = ai; }
        }
      }
      tm.sync();
    }
  }
}

__device__ __forceinline__ int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

// Keep the k largest keys of keys[0..*nkeys) (sorted descending), update the admission threshold.
// Must be called by all threads of the team; contains barriers.  Returns the new count (uniform).
__device__ int prune_topk(unsigned long long* keys, int* nkeys, unsigned long long* thr, int k, const Team& tm) {
  tm.sync();
  const int n = *nkeys;
  if (n > 1) {
    const int np = next_pow2(n);
    for (int i = n + tm.tid; i < np; i += tm.nt) keys[i] = 0ull;
    tm.sync();
    bitonic_sort_desc(keys, np, tm);
    if (tm.tid == 0 && n >= k) { *nkeys = k; *thr = keys[k - 1]; }
    tm.sync();
  }
  return min(n, k);
}

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// The hot kernel.  One CTA per work item = (query, range of document tiles).
//
// Per tile of S documents the CTA owns, in shared memory:  acc[S] f32 score accumulators,
// cnt[S] u8 "groups matched so far" counters and cand[S] u16 slots touched by the first
// group.  Leaves are walked in group order (smallest group first) with a barrier between
// leaves, so every accumulator is updated by one thread at a time, in a fixed order: the plan's
// leaf order, acc = fmaf(w, impact, acc) over the {docid, impact} pairs, as in the warp kernels,
// so a document gets the same float32 score whichever kernel serves its query.
// A posting of group g contributes only to slots with cnt == g (first hit of the group:
// cnt becomes g + 1) or cnt == g + 1 (another leaf of the same group already hit).  After the
// last leaf the candidates with cnt == n_groups are the tile's matches: they are counted,
// turned into 64-bit keys and offered to the CTA's top-k buffer.
// ------------------------------------------------------------------------------------------
struct ScoreParams {
  const uint2* pairs;           // {docid, impact} per posting (the warp kernels' store)
  const LeafRec* leaves;
  const QueryRec* queries;
  const ItemRec* items;
  const uint32_t* bounds;
  unsigned long long* part_keys;   // [n_parts * k]
  unsigned long long* totals;      // [Q]
  uint32_t S;
  uint32_t T;
  uint32_t n_docs;
  uint32_t doc_base;
  int k;
  int cap;                      // key buffer capacity (power of two)
  unsigned long long* prof;     // BM25F_PROFILE builds: 16 cycle counters, else null
};

__global__ void __launch_bounds__(512) k_score_topk(ScoreParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tid = threadIdx.x;
  const int nt = blockDim.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int nwarps = nt >> 5;
  const uint32_t S = p.S;
  const Team tm{tid, nt, 0};

  // carve shared memory
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  float* acc = reinterpret_cast<float*>(keys + p.cap);
  uint16_t* cand = reinterpret_cast<uint16_t*>(acc + S);
  uint8_t* cnt = reinterpret_cast<uint8_t*>(cand + S);
  __shared__ LeafRec s_leaf[MAXL];
  __shared__ uint32_t s_bounds[3][MAXL];
  __shared__ int s_ncand[2];
  __shared__ int s_nkeys;
  __shared__ unsigned long long s_thr;
  __shared__ unsigned long long s_total;

  const ItemRec item = p.items[blockIdx.x];
  const QueryRec q = p.queries[item.q];
  const int L = (int)q.n_leaves;
  const int G = (int)q.n_groups;
  const bool simple_or = (q.flags & QF_SIMPLE_OR) != 0;
  const unsigned long long upper = q.after_key ? q.after_key : ~0ull;

  for (int i = tid; i < L; i += nt) s_leaf[i] = p.leaves[q.leaf_begin + i];
  for (uint32_t i = tid; i < S; i += nt) { acc[i] = 0.0f; cnt[i] = 0; }
  if (tid == 0) { s_ncand[0] = 0; s_ncand[1] = 0; s_nkeys = 0; s_thr = 0ull; s_total = 0ull; }
  const uint32_t* qbounds = p.bounds + (size_t)q.leaf_begin * (p.T + 1);
  // rows tile_begin and tile_begin + 1 of the boundary table
  for (int i = tid; i < 2 * L; i += nt) {
    int r = i / L, l = i - r * L;
    s_bounds[(item.tile_begin + r) % 3][l] = qbounds[(size_t)(item.tile_begin + r) * L + l];
  }
  __syncthreads();

  unsigned int my_total = 0;
  int budget = p.cap;                  // keys that can still be appended without overflow (uniform)

  for (uint32_t t = item.tile_begin; t < item.tile_end; ++t) {
    const uint32_t t0 = t * S;
    int* ncand_ctr = &s_ncand[t & 1];
    // prefetch the boundary row of tile t + 2 (consumed by tile t + 1 as its upper bounds)
    if (t + 2 <= p.T && tid < L) cp_async4(&s_bounds[(t + 2) % 3][tid], qbounds + (size_t)(t + 2) * L + tid);
    const uint32_t* blo = s_bounds[t % 3];
    const uint32_t* bhi = s_bounds[(t + 1) % 3];

    for (int l = 0; l < L; ++l) {
      const uint32_t lo = blo[l], hi = bhi[l];
      if (lo < hi) {
        const LeafRec lf = s_leaf[l];
        const unsigned long long base = lf.off + lo;
        const unsigned long long end = lf.off + hi;
        const float w = lf.w;
        const uint32_t g = lf.group;
        // 32-byte aligned groups of four postings, one group per lane per step
        for (unsigned long long wb = (base & ~3ull) + (unsigned long long)warp * 128ull; wb < end;
             wb += (unsigned long long)nwarps * 128ull) {
          const unsigned long long i = wb + (unsigned long long)lane * 4ull;
          uint2 r[4] = {};
          if (i < end) {
            const uint4 a = __ldg(reinterpret_cast<const uint4*>(p.pairs + i));
            const uint4 b = __ldg(reinterpret_cast<const uint4*>(p.pairs + i + 2));
            r[0] = make_uint2(a.x, a.y); r[1] = make_uint2(a.z, a.w);
            r[2] = make_uint2(b.x, b.y); r[3] = make_uint2(b.z, b.w);
          }
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const bool valid = (i + e >= base) && (i + e < end);
            bool fresh = false;
            uint32_t slot = 0;
            if (valid) {
              slot = r[e].x - t0;
              const float u = __uint_as_float(r[e].y);
              if (!(u > 0.0f)) {
                // impact 0: a posting weight of 0 is not a match
              } else if (simple_or) {
                const float old = acc[slot];
                acc[slot] = fmaf(w, u, old);             // the warp kernels' arithmetic, in leaf order
                fresh = (old == 0.0f);
              } else {
                const uint32_t c = cnt[slot];
                if (c == g) {
                  cnt[slot] = (uint8_t)(g + 1);
                  acc[slot] = fmaf(w, u, acc[slot]);
                  fresh = (g == 0);
                } else if (c == g + 1) {
                  acc[slot] = fmaf(w, u, acc[slot]);
                }
              }
            }
            const unsigned m = __ballot_sync(0xFFFFFFFFu, fresh);
            if (m) {
              int b = 0;
              const int leader = __ffs(m) - 1;
              if (lane == leader) b = atomicAdd(ncand_ctr, __popc(m));
              b = __shfl_sync(0xFFFFFFFFu, b, leader);
              if (fresh) cand[b + __popc(m & ((1u << lane) - 1u))] = (uint16_t)slot;
            }
          }
        }
        __syncthreads();   // the next leaf may touch the same slots
      }
    }

    // ---- tile epilogue: matches -> total, keys -> top-k buffer, reset touched slots --------
    const int ncand = *ncand_ctr;
    for (int j0 = 0; j0 < ncand; j0 += nt) {
      if (budget < nt) {               // the bound is conservative: look at the real count first
        __syncthreads();
        int n = s_nkeys;
        __syncthreads();
        if (p.cap - n < nt) n = prune_topk(keys, &s_nkeys, &s_thr, p.k, tm);
        budget = p.cap - n;
      }
      budget -= nt;
      const int j = j0 + tid;
      bool push = false;
      unsigned long long key = 0ull;
      if (j < ncand) {
        const uint32_t slot = cand[j];
        const float sc = acc[slot];
        acc[slot] = 0.0f;
        bool match = true;
        if (!simple_or) { match = (cnt[slot] == (uint8_t)G); cnt[slot] = 0; }
        const uint32_t doc = t0 + slot;
        if (match) {
          ++my_total;
          key = make_key(sc, p.doc_base + doc);
          push = (key > s_thr) && (key < upper);
        }
      }
      const unsigned m = __ballot_sync(0xFFFFFFFFu, push);
      if (m) {
        int b = 0;
        const int leader = __ffs(m) - 1;
        if (lane == leader) b = atomicAdd(&s_nkeys, __popc(m));
        b = __shfl_sync(0xFFFFFFFFu, b, leader);
        if (push) keys[b + __popc(m & ((1u << lane) - 1u))] = key;
      }
    }
    cp_async_wait_all();
    __syncthreads();                   // end of tile: slots are clean, boundary row t + 2 has landed
    if (tid == 0) *ncand_ctr = 0;      // next used by tile t + 2, ordered by the barrier of tile t + 1
    budget = p.cap - s_nkeys;          // nobody appends before the next tile's leaf barrier
  }

  // ---- item epilogue -------------------------------------------------------------------
  const int n = prune_topk(keys, &s_nkeys, &s_thr, p.k, tm);
  unsigned long long* out = p.part_keys + (size_t)item.part * p.k;
  for (int i = tid; i < p.k; i += nt) out[i] = (i < n) ? keys[i] : 0ull;
  // match count of this item
  for (int o = 16; o > 0; o >>= 1) my_total += __shfl_down_sync(0xFFFFFFFFu, my_total, o);
  if (lane == 0 && my_total) atomicAdd(&s_total, (unsigned long long)my_total);
  __syncthreads();
  if (tid == 0 && s_total) atomicAdd(p.totals + item.q, s_total);
}

// ------------------------------------------------------------------------------------------
// mbarrier / bulk-copy (TMA) primitives, sm_90+ PTX
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(unsigned long long* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(a), "r"(parity)
        : "memory");
  } while (!ok);
}
// 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------------------------------
// The hot kernel, pipelined.  Same algorithm and data structures as k_score_topk, but DRAM
// latency is decoupled from the per-leaf accumulate phases: the last warp of the CTA is a
// PRODUCER that walks the item's static (tile, leaf, chunk) schedule ahead of the consumers and
// stages chunks of {docid, impact} pairs into a ring of shared-memory stages with 1-D bulk
// copies (cp.async.bulk, completion on an mbarrier per stage).  The CONSUMER warps wait on the
// stage's "full" barrier, accumulate one posting per lane from shared memory, release the stage
// on its "empty" barrier, and synchronise among themselves (named barrier 1) only where the
// algorithm needs it: between two leaves of a tile and around the tile epilogue.
// ------------------------------------------------------------------------------------------
#ifdef BM25F_PROFILE
#define PROF_DECL long long pt_[8] = {0, 0, 0, 0, 0, 0, 0, 0}; long long pt0_ = 0
#define PROF_T0() pt0_ = clock64()
#define PROF_ADD(i) do { long long n_ = clock64(); pt_[i] += n_ - pt0_; pt0_ = n_; } while (0)
#define PROF_FLUSH(base, on) do { if (on && p.prof) for (int i_ = 0; i_ < 8; ++i_) atomicAdd(p.prof + (base) + i_, (unsigned long long)pt_[i_]); } while (0)
#else
#define PROF_DECL
#define PROF_T0()
#define PROF_ADD(i)
#define PROF_FLUSH(base, on)
#endif

constexpr int PIPE_MAX_STAGES = 32;
constexpr int PIPE_BROWS = 4;          // boundary rows kept by the producer
constexpr int HOTCAP = 512;            // per-tile list of documents whose score crossed the threshold
constexpr uint32_t SF_LEAF_END = 1u, SF_TILE_END = 2u, SF_END = 4u, SF_LAST_GROUP = 8u;

struct __align__(16) StageMeta {   // 32 B: two 128-bit shared loads
  uint32_t t0;        // first document of the tile
  uint32_t n;         // postings staged (multiple of 16, includes alignment padding)
  uint32_t vbeg;      // valid range inside the stage
  uint32_t vend;
  float w;            // leaf weight
  uint32_t group;     // leaf's group rank
  uint32_t flags;
  uint32_t pad;
};

struct PipeParams {
  ScoreParams sp;
  uint32_t chunk;       // postings per stage (multiple of 16)
  uint32_t stages;      // ring depth (<= PIPE_MAX_STAGES)
  uint32_t prune_at;    // sort + cut the key buffer when it holds this many keys
};

// Requires every leaf weight > 0 (scores only grow while a tile is accumulated); batches with a
// non-positive weight are routed to k_score_topk by the host.
//
// Matches are COUNTED while accumulating (a slot's first hit for OR, the hit that completes the
// last group for AND), so the tile epilogue does no per-candidate work beyond clearing the touched
// slots.  A document is offered to the top-k buffer only if its running score crosses the current
// k-th best score ("hot"); until k hits exist the threshold is the smallest positive float, every
// match is hot, the hot list overflows and the epilogue falls back to walking all candidates.
__global__ void __launch_bounds__(544) k_score_pipe(PipeParams pp) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const ScoreParams& p = pp.sp;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int NC = (int)blockDim.x - 32;          // consumer threads
  const int producer_warp = NC >> 5;
  const uint32_t S = p.S, CH = pp.chunk, NS = pp.stages;

  // carve shared memory
  unsigned long long* keys = reinterpret_cast<unsigned long long*>(smem_raw);
  float* acc = reinterpret_cast<float*>(keys + p.cap);
  uint16_t* cand = reinterpret_cast<uint16_t*>(acc + S);
  uint8_t* cnt = reinterpret_cast<uint8_t*>(cand + S);
  uint2* spair = reinterpret_cast<uint2*>(smem_raw + (((size_t)p.cap * 8 + (size_t)S * 7 + 15) & ~(size_t)15));
  uint16_t* hot = reinterpret_cast<uint16_t*>(spair + (size_t)NS * CH);
  __shared__ LeafRec s_leaf[MAXL];
  __shared__ uint32_t s_brow[PIPE_BROWS][MAXL];
  __shared__ StageMeta s_meta[PIPE_MAX_STAGES];
  __shared__ __align__(8) unsigned long long s_full[PIPE_MAX_STAGES];
  __shared__ __align__(8) unsigned long long s_empty[PIPE_MAX_STAGES];
  __shared__ int s_ncand[2];
  __shared__ int s_nhot[2];
  __shared__ int s_nkeys;
  __shared__ unsigned long long s_thr;
  __shared__ float s_thr_score;
  __shared__ unsigned long long s_total;

  const ItemRec item = p.items[blockIdx.x];
  const QueryRec q = p.queries[item.q];
  const int L = (int)q.n_leaves;
  const int G = (int)q.n_groups;
  const bool simple_or = (q.flags & QF_SIMPLE_OR) != 0;
  const unsigned long long upper = q.after_key ? q.after_key : ~0ull;
  const uint32_t* qbounds = p.bounds + (size_t)q.leaf_begin * (p.T + 1);

  for (int i = tid; i < L; i += blockDim.x) s_leaf[i] = p.leaves[q.leaf_begin + i];
  for (uint32_t i = tid; i < S; i += blockDim.x) { acc[i] = 0.0f; cnt[i] = 0; }
  if (tid == 0) {
    s_ncand[0] = 0; s_ncand[1] = 0; s_nhot[0] = 0; s_nhot[1] = 0; s_nkeys = 0; s_thr = 0ull; s_total = 0ull;
    s_thr_score = 1.17549435e-38f;    // FLT_MIN: every first hit crosses it
    for (uint32_t i = 0; i < NS; ++i) { mbar_init(&s_full[i], 1); mbar_init(&s_empty[i], (uint32_t)producer_warp); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (warp == producer_warp) {
    // =============================== PRODUCER ===============================================
    for (int r = 0; r < PIPE_BROWS; ++r) {
      const uint32_t row = item.tile_begin + r;
      if (row <= p.T)
        for (int l = lane; l < L; l += 32) s_brow[row % PIPE_BROWS][l] = qbounds[(size_t)row * L + l];
    }
    __syncwarp();
    PROF_DECL;
    PROF_T0();
    uint32_t stage = 0, phase = 0;
    for (uint32_t t = item.tile_begin; t < item.tile_end; ++t) {
      if (t > item.tile_begin) {
        // rows t and t + 1 are needed: at most the two youngest prefetch groups may be pending
        asm volatile("cp.async.wait_group 2;" ::: "memory");
        __syncwarp();
      }
      PROF_ADD(0);                        // [8] producer: boundary rows
      const uint32_t* blo = s_brow[t % PIPE_BROWS];
      const uint32_t* bhi = s_brow[(t + 1) % PIPE_BROWS];
      if (lane == 0) {
        // which leaves have postings in this tile; an AND with an empty group skips the tile
        int last = -1;
        bool skip = false;
        uint32_t cur_g = 0;
        bool g_has = false;
        for (int l = 0; l < L; ++l) {
          const uint32_t g = s_leaf[l].group;
          if (g != cur_g) { if (!g_has) skip = true; cur_g = g; g_has = false; }
          if (blo[l] < bhi[l]) { last = l; g_has = true; }
        }
        if (!g_has) skip = true;
        if (simple_or) skip = (last < 0);
        if (!skip) {
          for (int l = 0; l <= last; ++l) {
            const uint32_t lo = blo[l], hi = bhi[l];
            if (lo >= hi) continue;
            const LeafRec lf = s_leaf[l];
            const unsigned long long a = lf.off + lo, b = lf.off + hi;
            for (unsigned long long c0 = a & ~15ull; c0 < b; c0 += CH) {
              unsigned long long rem = ((b - c0) + 15ull) & ~15ull;
              const uint32_t n = (uint32_t)(rem < CH ? rem : CH);
              PROF_ADD(1);                // [9] producer: schedule arithmetic
              mbar_wait(&s_empty[stage], phase ^ 1u);
              PROF_ADD(2);                // [10] producer: wait for a free stage
              StageMeta m;
              m.t0 = t * S;
              m.n = n;
              m.vbeg = (uint32_t)(a > c0 ? a - c0 : 0);
              m.vend = (uint32_t)(b < c0 + n ? b - c0 : n);
              m.w = lf.w;
              m.group = lf.group;
              const bool last_chunk = (c0 + CH >= b);
              m.flags = (last_chunk ? SF_LEAF_END : 0u) | ((last_chunk && l == last) ? SF_TILE_END : 0u) |
                        ((int)lf.group == G - 1 ? SF_LAST_GROUP : 0u);
              m.pad = 0u;
              s_meta[stage] = m;
              mbar_arrive_expect_tx(&s_full[stage], n * 8u);
              bulk_g2s(spair + (size_t)stage * CH, p.pairs + c0, n * 8u, &s_full[stage]);
              if (++stage == NS) { stage = 0; phase ^= 1u; }
              PROF_ADD(3);                // [11] producer: meta + issue
            }
          }
        }
      }
      __syncwarp();
      const uint32_t row = t + PIPE_BROWS;
      if (row <= p.T)
        for (int l = lane; l < L; l += 32) cp_async4(&s_brow[row % PIPE_BROWS][l], qbounds + (size_t)row * L + l);
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    if (lane == 0) {
      mbar_wait(&s_empty[stage], phase ^ 1u);
      StageMeta m = {0u, 0u, 0u, 0u, 0.0f, 0u, SF_END, 0u};
      s_meta[stage] = m;
      mbar_arrive(&s_full[stage]);
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    PROF_ADD(4);
    PROF_FLUSH(8, lane == 0);
    return;
  }

  // ================================= CONSUMERS ================================================
  const Team tm{tid, NC, 1};
  unsigned int my_total = 0;
  uint32_t stage = 0, phase = 0, seq = 0;
  PROF_DECL;
  PROF_T0();
  for (;;) {
    mbar_wait(&s_full[stage], phase);
    PROF_ADD(0);                          // [0] consumer: wait for a full stage
    const StageMeta m = s_meta[stage];
    if (m.flags & SF_END) break;
    {
      const float w = m.w;
      const float thr_s = s_thr_score;
      const uint2* __restrict__ sp = spair + (size_t)stage * CH;
      int* ncand_ctr = &s_ncand[seq & 1u];
      int* nhot_ctr = &s_nhot[seq & 1u];
      if (simple_or) {
        for (uint32_t i0 = (uint32_t)(warp * 32); i0 < m.n; i0 += (uint32_t)NC) {
          const uint32_t i = i0 + lane;
          bool fresh = false;
          uint32_t slot = 0;
          if (i >= m.vbeg && i < m.vend) {
            const uint2 r = sp[i];
            const float u = __uint_as_float(r.y);
            if (u > 0.0f) {                                     // impact 0: a posting weight of 0 is not a match
              slot = r.x - m.t0;
              const float old = acc[slot];
              const float nw = fmaf(w, u, old);                 // the warp kernels' arithmetic, in leaf order
              acc[slot] = nw;
              fresh = (old == 0.0f);
              if (nw >= thr_s && old < thr_s) {
                const int h = atomicAdd(nhot_ctr, 1);
                if (h < HOTCAP) hot[h] = (uint16_t)slot;
              }
            }
          }
          const unsigned mk = __ballot_sync(0xFFFFFFFFu, fresh);
          if (mk) {
            int b = 0;
            if (lane == 0) b = atomicAdd(ncand_ctr, __popc(mk));
            b = __shfl_sync(0xFFFFFFFFu, b, 0);
            if (fresh) cand[b + __popc(mk & ((1u << lane) - 1u))] = (uint16_t)slot;
            if (lane == 0) my_total += __popc(mk);              // a first hit is a match (OR)
          }
        }
      } else {
        const uint32_t g = m.group;
        const bool last_group = (m.flags & SF_LAST_GROUP) != 0;
        for (uint32_t i0 = (uint32_t)(warp * 32); i0 < m.n; i0 += (uint32_t)NC) {
          const uint32_t i = i0 + lane;
          bool fresh = false, matched = false;
          uint32_t slot = 0;
          if (i >= m.vbeg && i < m.vend) {
            const uint2 r = sp[i];
            slot = r.x - m.t0;
            const uint32_t c = cnt[slot];
            if (c == g || c == g + 1) {                         // alive: earlier groups all matched
              const float u = __uint_as_float(r.y);
              if (u > 0.0f) {
                const float old = acc[slot];
                const float nw = fmaf(w, u, old);
                acc[slot] = nw;
                bool crossing = (nw >= thr_s);
                if (c == g) {
                  cnt[slot] = (uint8_t)(g + 1);
                  fresh = (g == 0);
                  matched = last_group;                         // this hit completes the last group
                } else {
                  crossing = crossing && (old < thr_s);
                }
                if (last_group && crossing) {
                  const int h = atomicAdd(nhot_ctr, 1);
                  if (h < HOTCAP) hot[h] = (uint16_t)slot;
                }
              }
            }
          }
          const unsigned mk = __ballot_sync(0xFFFFFFFFu, fresh);
          if (mk) {
            int b = 0;
            if (lane == 0) b = atomicAdd(ncand_ctr, __popc(mk));
            b = __shfl_sync(0xFFFFFFFFu, b, 0);
            if (fresh) cand[b + __popc(mk & ((1u << lane) - 1u))] = (uint16_t)slot;
          }
          if (last_group) {
            const unsigned mm = __ballot_sync(0xFFFFFFFFu, matched);
            if (lane == 0) my_total += __popc(mm);
          }
        }
      }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive(&s_empty[stage]);       // this warp no longer reads the stage
    if (++stage == NS) { stage = 0; phase ^= 1u; }
    PROF_ADD(1);                                        // [1] consumer: accumulate
    if (m.flags & SF_LEAF_END) tm.sync();               // the next leaf may touch the same slots
    PROF_ADD(2);                                        // [2] consumer: leaf barrier
    if (m.flags & SF_TILE_END) {
      // ---- tile epilogue ----------------------------------------------------------------------
      int* ncand_ctr = &s_ncand[seq & 1u];
      int* nhot_ctr = &s_nhot[seq & 1u];
      const int ncand = *ncand_ctr;
      const int nhot = *nhot_ctr;
      if (nhot > HOTCAP) {
        // no (tight) threshold yet: walk every candidate, as k_score_topk does
        int budget = p.cap - s_nkeys;
        tm.sync();
        for (int j0 = 0; j0 < ncand; j0 += NC) {
          if (budget < NC) {
            tm.sync();
            int n = s_nkeys;
            tm.sync();
            if (p.cap - n < NC) n = prune_topk(keys, &s_nkeys, &s_thr, p.k, tm);
            budget = p.cap - n;
          }
          budget -= NC;
          const int j = j0 + tid;
          bool push = false;
          unsigned long long key = 0ull;
          if (j < ncand) {
            const uint32_t slot = cand[j];
            const float sc = acc[slot];
            acc[slot] = 0.0f;
            bool match = true;
            if (!simple_or) { match = (cnt[slot] == (uint8_t)G); cnt[slot] = 0; }
            if (match) {
              key = make_key(sc, p.doc_base + m.t0 + slot);
              push = (key > s_thr) && (key < upper);
            }
          }
          const unsigned mk = __ballot_sync(0xFFFFFFFFu, push);
          if (mk) {
            int b = 0;
            if (lane == 0) b = atomicAdd(&s_nkeys, __popc(mk));
            b = __shfl_sync(0xFFFFFFFFu, b, 0);
            if (push) keys[b + __popc(mk & ((1u << lane) - 1u))] = key;
          }
        }
      } else {
        if (nhot > 0) {
          // the buffer always has room for HOTCAP more keys here (see the prune rule below)
          for (int j = tid; j < nhot; j += NC) {
            const uint32_t slot = hot[j];
            const unsigned long long key = make_key(acc[slot], p.doc_base + m.t0 + slot);
            if (key > s_thr && key < upper) keys[atomicAdd(&s_nkeys, 1)] = key;
          }
          tm.sync();                      // scores are read before the slots are cleared
        }
        if (simple_or) {
          for (int j = tid; j < ncand; j += NC) acc[cand[j]] = 0.0f;
        } else {
          for (int j = tid; j < ncand; j += NC) { const uint32_t slot = cand[j]; acc[slot] = 0.0f; cnt[slot] = 0; }
        }
      }
      tm.sync();                          // end of tile: slots are clean
      if (tid == 0) { *ncand_ctr = 0; *nhot_ctr = 0; }    // next used two tiles later
      // keep the threshold tight and the buffer small: sort + cut when enough keys piled up
      const int nk = s_nkeys;
      if (nk >= p.k && (nk >= (int)pp.prune_at || s_thr == 0ull)) {
        prune_topk(keys, &s_nkeys, &s_thr, p.k, tm);
        if (tid == 0) s_thr_score = key_score(s_thr);
        tm.sync();                        // one threshold per tile for everybody (no double "crossing")
        PROF_ADD(4);                      // [4] consumer: prune
      }
      ++seq;
      PROF_ADD(3);                        // [3] consumer: tile epilogue
    }
  }

  // ---- item epilogue (consumers only; the producer warp has exited) ---------------------------
  const int n = prune_topk(keys, &s_nkeys, &s_thr, p.k, tm);
  unsigned long long* out = p.part_keys + (size_t)item.part * p.k;
  for (int i = tid; i < p.k; i += NC) out[i] = (i < n) ? keys[i] : 0ull;
  for (int o = 16; o > 0; o >>= 1) my_total += __shfl_down_sync(0xFFFFFFFFu, my_total, o);
  if (lane == 0 && my_total) atomicAdd(&s_total, (unsigned long long)my_total);
  tm.sync();
  if (tid == 0 && s_total) atomicAdd(p.totals + item.q, s_total);
  PROF_ADD(5);                            // [5] consumer: item epilogue
  PROF_FLUSH(0, tid == 0);
}

// ------------------------------------------------------------------------------------------
// Warp-level helpers shared by the stream kernel
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t x, uint32_t y) {
  asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(addr), "r"(x), "r"(y) : "memory");
}
__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}

// insert `key` into the warp's sorted top list (lane i = i-th best); all lanes call this
__device__ __forceinline__ void warp_topk_insert(unsigned long long& mine, unsigned long long key, int lane) {
  const int pos = __popc(__ballot_sync(0xFFFFFFFFu, mine > key));
  const unsigned long long up = __shfl_up_sync(0xFFFFFFFFu, mine, 1);
  if (lane > pos) mine = up;
  if (lane == pos) mine = key;
}

// The same list with KR keys per lane (k <= 32 * KR): row j of lane i holds rank 32 * j + i.
template <int KR>
__device__ __forceinline__ void warp_topk_insert_rows(unsigned long long (&top)[KR], unsigned long long key, int lane) {
  bool inserted = false;
  unsigned long long carry = 0ull;
#pragma unroll
  for (int j = 0; j < KR; ++j) {
    const unsigned long long last = __shfl_sync(0xFFFFFFFFu, top[j], 31);
    const unsigned long long up = __shfl_up_sync(0xFFFFFFFFu, top[j], 1);
    if (!inserted) {
      const int pos = __popc(__ballot_sync(0xFFFFFFFFu, top[j] > key));
      if (pos < 32) {                       // the key belongs in this row; its last element moves on
        if (lane > pos) top[j] = up;
        if (lane == pos) top[j] = key;
        carry = last;
        inserted = true;
      }
    } else {                                // rows after it shift by one
      top[j] = (lane == 0) ? carry : up;
      carry = last;
    }
  }
}
template <int KR>
__device__ __forceinline__ unsigned long long warp_topk_kth(const unsigned long long (&top)[KR], int k) {
  unsigned long long v = 0ull;
#pragma unroll
  for (int j = 0; j < KR; ++j) {
    const unsigned long long t = __shfl_sync(0xFFFFFFFFu, top[j], (k - 1) & 31);
    if (j == ((k - 1) >> 5)) v = t;
  }
  return v;
}

#include "final.cuh"
#include "stream.cuh"
#include "team.cuh"
#include "isect.cuh"
#include "plan.cuh"

// ------------------------------------------------------------------------------------------
// Merge of sorted top-k lists.  List l of query q starts at keys + start(q) + l * stride.
// mode 0: lists are the partial lists of the query's work items (start = part_begin * k, stride k)
// mode 1: lists come from an all-gather over document shards  (start = q * k, stride = Q * k)
// ------------------------------------------------------------------------------------------
__global__ void k_merge_topk(const unsigned long long* __restrict__ keys_in, const QueryRec* __restrict__ queries,
                             int mode, int n_lists_fixed, unsigned long long stride_fixed, uint32_t Q, int k,
                             int kp /* pow2 >= k */, unsigned long long* __restrict__ keys_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(smem_raw);   // [2 * kp]
  const uint32_t q = blockIdx.x;
  if (q >= Q) return;
  unsigned long long start, stride;
  int n_lists;
  if (mode == 0) {
    const QueryRec qr = queries[q];
    start = (unsigned long long)qr.part_begin * k;
    stride = (unsigned long long)k;
    n_lists = (int)qr.n_parts;
  } else {
    start = (unsigned long long)q * k;
    stride = stride_fixed;
    n_lists = n_lists_fixed;
  }
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < 2 * kp; i += nt) buf[i] = 0ull;
  __syncthreads();
  if (n_lists > 0)
    for (int i = tid; i < k; i += nt) buf[i] = keys_in[start + i];
  __syncthreads();
  // Every list is sorted descending (the scoring kernels and this kernel write them that way) and so is buf[0, kp):
  // the next list goes into the upper half back to front, which makes buf bitonic, and one bitonic MERGE
  // (log2(2 kp) compare-exchange rounds instead of the ~log^2 of a sort) puts the 2 kp keys in descending order.
  for (int l = 1; l < n_lists; ++l) {
    for (int i = tid; i < kp; i += nt) buf[2 * kp - 1 - i] = (i < k) ? keys_in[start + l * stride + i] : 0ull;
    __syncthreads();
    for (int j = kp; j > 0; j >>= 1) {
      for (int i = tid; i < 2 * kp; i += nt) {
        const int x = i ^ j;
        if (x > i) {
          const unsigned long long ai = buf[i], ax = buf[x];
          if (ai < ax) { buf[i] = ax; buf[x] = ai; }
        }
      }
      __syncthreads();
    }
    for (int i = k + tid; i < kp; i += nt) buf[i] = 0ull;
    __syncthreads();
  }
  for (int i = tid; i < k; i += nt) keys_out[(size_t)q * k + i] = buf[i];
}

// Same merge for k <= 32: one warp per query, lane i keeps the i-th best key, candidates are inserted
// with shuffles (no shared memory, no barriers).
__global__ void k_merge_topk_warp(const unsigned long long* __restrict__ keys_in, const QueryRec* __restrict__ queries,
                                  int mode, int n_lists_fixed, unsigned long long stride_fixed, uint32_t Q, int k,
                                  unsigned long long* __restrict__ keys_out) {
  const int lane = threadIdx.x & 31;
  const uint32_t q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= Q) return;
  unsigned long long start, stride;
  int n_lists;
  if (mode == 0) {
    const QueryRec qr = queries[q];
    start = (unsigned long long)qr.part_begin * k;
    stride = (unsigned long long)k;
    n_lists = (int)qr.n_parts;
  } else {
    start = (unsigned long long)q * k;
    stride = stride_fixed;
    n_lists = n_lists_fixed;
  }
  unsigned long long best = (n_lists > 0 && lane < k) ? keys_in[start + lane] : 0ull;
  unsigned long long thr = __shfl_sync(0xFFFFFFFFu, best, k - 1);
  for (int l = 1; l < n_lists; ++l) {
    const unsigned long long key = (lane < k) ? keys_in[start + l * stride + lane] : 0ull;
    unsigned pm = __ballot_sync(0xFFFFFFFFu, key > thr);
    while (pm) {
      const int src = __ffs(pm) - 1;
      pm &= pm - 1u;
      const unsigned long long bk = __shfl_sync(0xFFFFFFFFu, key, src);
      if (bk > thr) {
        warp_topk_insert(best, bk, lane);
        thr = __shfl_sync(0xFFFFFFFFu, best, k - 1);
      }
    }
  }
  if (lane < k) keys_out[(size_t)q * k + lane] = best;
}

// Final mode: merge of a query's partial lists of 96-bit keys and decode in one pass, one warp per query,
// KR keys per lane (k <= 32 * KR).
template <int KR>
__global__ void k_merge_final(const unsigned long long* __restrict__ part_hi, const unsigned int* __restrict__ part_lo,
                              const QueryRec* __restrict__ queries, uint32_t Q, int k, double* __restrict__ out_final,
                              uint32_t* __restrict__ out_docids, uint32_t* __restrict__ out_counts) {
  const int lane = threadIdx.x & 31;
  const uint32_t q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= Q) return;
  const QueryRec qr = queries[q];
  const size_t start = (size_t)qr.part_begin * k;
  unsigned long long top[KR];
  uint32_t topl[KR];
#pragma unroll
  for (int j = 0; j < KR; ++j) { top[j] = 0ull; topl[j] = 0u; }
  unsigned long long thr_h = 0ull;
  uint32_t thr_l = 0u;
  for (uint32_t l = 0; l < qr.n_parts; ++l) {
#pragma unroll 1
    for (int j = 0; j < KR; ++j) {
      const int idx = 32 * j + lane;
      if (32 * j >= k) break;
      unsigned long long kh = 0ull;
      uint32_t kl = 0u;
      if (idx < k) {
        kh = part_hi[start + (size_t)l * k + idx];
        kl = part_lo[start + (size_t)l * k + idx];
      }
      unsigned pm = __ballot_sync(0xFFFFFFFFu, key2_gt(kh, kl, thr_h, thr_l));
      while (pm) {
        const int src = __ffs(pm) - 1;
        pm &= pm - 1u;
        const unsigned long long bh = __shfl_sync(0xFFFFFFFFu, kh, src);
        const uint32_t bl = __shfl_sync(0xFFFFFFFFu, kl, src);
        if (key2_gt(bh, bl, thr_h, thr_l)) {
          warp_topk2_insert_rows<KR>(top, topl, bh, bl, lane);
          warp_topk2_kth<KR>(top, topl, k, thr_h, thr_l);
        }
      }
    }
  }
  uint32_t n = 0;
#pragma unroll
  for (int j = 0; j < KR; ++j) {
    const int idx = 32 * j + lane;
    const bool ok = idx < k && top[j] != 0ull;
    if (idx < k) {
      out_final[(size_t)q * k + idx] = ok ? orderable_f64_value(top[j]) : -INFINITY;
      out_docids[(size_t)q * k + idx] = ok ? 0xFFFFFFFFu - topl[j] : 0xFFFFFFFFu;
    }
    n += (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, ok));
  }
  if (lane == 0) out_counts[q] = n;
}

// Final mode across document shards: merge of n_lists decoded result lists per query (layout
// [n_lists][Q][k], as an all-gather of the shards' (final value, docnum) results produces; an empty slot has
// docnum 0xFFFFFFFF), one warp per query, KR keys per lane (k <= 32 * KR).
template <int KR>
__global__ void k_merge_final_lists(const double* __restrict__ vals, const uint32_t* __restrict__ docids, int n_lists,
                                    uint32_t Q, int k, double* __restrict__ out_final, uint32_t* __restrict__ out_docids,
                                    uint32_t* __restrict__ out_counts) {
  const int lane = threadIdx.x & 31;
  const uint32_t q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= Q) return;
  unsigned long long top[KR];
  uint32_t topl[KR];
#pragma unroll
  for (int j = 0; j < KR; ++j) { top[j] = 0ull; topl[j] = 0u; }
  unsigned long long thr_h = 0ull;
  uint32_t thr_l = 0u;
  for (int l = 0; l < n_lists; ++l) {
    const size_t start = ((size_t)l * Q + q) * k;
#pragma unroll 1
    for (int j = 0; j < KR; ++j) {
      const int idx = 32 * j + lane;
      if (32 * j >= k) break;
      unsigned long long kh = 0ull;
      uint32_t kl = 0u;
      if (idx < k) {
        const uint32_t d = docids[start + idx];
        if (d != 0xFFFFFFFFu) {
          kh = orderable_f64(vals[start + idx]);
          kl = 0xFFFFFFFFu - d;
        }
      }
      unsigned pm = __ballot_sync(0xFFFFFFFFu, key2_gt(kh, kl, thr_h, thr_l));
      while (pm) {
        const int src = __ffs(pm) - 1;
        pm &= pm - 1u;
        const unsigned long long bh = __shfl_sync(0xFFFFFFFFu, kh, src);
        const uint32_t bl = __shfl_sync(0xFFFFFFFFu, kl, src);
        if (key2_gt(bh, bl, thr_h, thr_l)) {
          warp_topk2_insert_rows<KR>(top, topl, bh, bl, lane);
          warp_topk2_kth<KR>(top, topl, k, thr_h, thr_l);
        }
      }
    }
  }
  uint32_t n = 0;
#pragma unroll
  for (int j = 0; j < KR; ++j) {
    const int idx = 32 * j + lane;
    const bool ok = idx < k && top[j] != 0ull;
    if (idx < k) {
      out_final[(size_t)q * k + idx] = ok ? orderable_f64_value(top[j]) : -INFINITY;
      out_docids[(size_t)q * k + idx] = ok ? 0xFFFFFFFFu - topl[j] : 0xFFFFFFFFu;
    }
    n += (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, ok));
  }
  if (lane == 0) out_counts[q] = n;
}

__global__ void k_decode_keys(const unsigned long long* __restrict__ keys, uint32_t Q, int k,
                              float* __restrict__ scores, uint32_t* __restrict__ docids,
                              uint32_t* __restrict__ counts) {
  const uint32_t q = blockIdx.x;
  if (q >= Q) return;
  int n = 0;
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const unsigned long long key = keys[(size_t)q * k + i];
    const bool ok = key != 0ull;
    if (scores) scores[(size_t)q * k + i] = ok ? key_score(key) : -INFINITY;
    if (docids) docids[(size_t)q * k + i] = ok ? key_doc(key) : 0xFFFFFFFFu;
    n += ok;
  }
  if (counts) {
    __shared__ int s_n;
    if (threadIdx.x == 0) s_n = 0;
    __syncthreads();
    if (n) atomicAdd(&s_n, n);
    __syncthreads();
    if (threadIdx.x == 0) counts[q] = (uint32_t)s_n;
  }
}

// The exchange step of a document-sharded batch in one kernel after the merge: decode the merged keys and add up
// the shards' match counts.  `gathered` holds, per shard, `span` 64-bit words: its [Q * k] keys first, its [Q]
// totals at word `tot_off`.
__global__ void k_decode_keys_sum(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ gathered,
                                  int n_lists, unsigned long long span, unsigned long long tot_off, uint32_t Q, int k,
                                  float* __restrict__ scores, uint32_t* __restrict__ docids, uint32_t* __restrict__ counts,
                                  unsigned long long* __restrict__ totals) {
  const uint32_t q = blockIdx.x;
  if (q >= Q) return;
  int n = 0;
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    const unsigned long long key = keys[(size_t)q * k + i];
    const bool ok = key != 0ull;
    scores[(size_t)q * k + i] = ok ? key_score(key) : -INFINITY;
    docids[(size_t)q * k + i] = ok ? key_doc(key) : 0xFFFFFFFFu;
    n += ok;
  }
  __shared__ int s_n;
  if (threadIdx.x == 0) {
    s_n = 0;
    unsigned long long t = 0ull;
    for (int l = 0; l < n_lists; ++l) t += gathered[(size_t)l * span + tot_off + q];
    totals[q] = t;
  }
  __syncthreads();
  if (n) atomicAdd(&s_n, n);
  __syncthreads();
  if (threadIdx.x == 0) counts[q] = (uint32_t)s_n;
}

}  // namespace

// ==========================================================================================
// Host side

// ==========================================================================================

// A few persistent host threads for query planning (creating threads per call costs more than the work).
class PlanPool {
 public:
  explicit PlanPool(unsigned n) {
    for (unsigned i = 0; i < n; ++i) workers_.emplace_back([this, i] { run(i); });
  }
  ~PlanPool() {
    {
      std::lock_guard<std::mutex> g(m_);
      stop_ = true;
      ++gen_;
    }
    cv_.notify_all();
    for (auto& t : workers_) t.join();
  }
  unsigned size() const { return (unsigned)workers_.size(); }
  // run fn(i) for i in [0, n) on the workers (n <= size()) and wait
  void parallel(unsigned n, const std::function<void(unsigned)>& fn) {
    {
      std::lock_guard<std::mutex> g(m_);
      fn_ = &fn;
      n_ = n;
      pending_ = n;
      ++gen_;
    }
    cv_.notify_all();
    std::unique_lock<std::mutex> g(m_);
    done_.wait(g, [this] { return pending_ == 0; });
    fn_ = nullptr;
  }

 private:
  void run(unsigned i) {
    unsigned long long seen = 0;
    for (;;) {
      const std::function<void(unsigned)>* fn = nullptr;
      {
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [&] { return gen_ != seen; });
        seen = gen_;
        if (stop_) return;
        if (i < n_) fn = fn_;
      }
      if (fn) {
        (*fn)(i);
        std::lock_guard<std::mutex> g(m_);
        if (--pending_ == 0) done_.notify_one();
      }
    }
  }
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cv_, done_;
  const std::function<void(unsigned)>* fn_ = nullptr;
  unsigned n_ = 0, pending_ = 0;
  unsigned long long gen_ = 0;
  bool stop_ = false;
};

struct bm25f_handle {
  int device = 0;
  cudaStream_t stream = nullptr;      // stream in use
  cudaStream_t own_stream = nullptr;  // created by the library
  cudaStream_t aux_stream = nullptr;  // the candidate-driven / team kernels run here, beside the stream kernel
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  uint64_t n_docs = 0, n_terms = 0, n_postings = 0, doc_base = 0;
  uint32_t n_fields = 0;               // real fields; field index n_fields is the constant-score pseudo-field of Every()
  uint64_t n_real_terms = 0;           // posting lists of the caller; [n_real_terms, n_terms) are the Every(field) lists
  std::vector<uint64_t> term_offsets;
  std::vector<uint8_t> term_field;
  uint32_t* d_docids = nullptr;
  uint32_t* d_payload = nullptr;
  uint8_t* d_lb = nullptr;
  uint2* d_pairs = nullptr;           // {docid, tf / (tf + norm[lb]) under the current weighting}: the stream kernel's store
  float* d_norm = nullptr;
  double* d_final_add = nullptr;   // bm25f_set_final_date: per-document date term (NaN: no date); null = no final() step
  double* d_final_blk = nullptr;   // ... and the largest one of every aligned block of 32 documents
  bool packed = true;
  bool have_weighting = false;
  uint32_t S = 8192, NT = 256, split = 1u << 16;
  uint32_t variant = 0;               // 0 / 3: auto (stream kernel where eligible, else pipeline), 1: pipeline, 2: direct loads
  // stream kernel: warps per CTA, accumulator bytes per warp, target work per item, L2 prefetch distance
  uint32_t st_warps = 16, st_slot_bytes = 11776, wsplit = 1u << 17, st_pf = 2048;
  // team kernel (variant 4): warps per CTA, target work per item, slices ahead to prefetch
  uint32_t tl_warps = 8, tl_slot_bytes = 10240, tl_split = 1u << 18, tl_prefetch = 0;
  uint32_t chunk = 512, stages = 4;   // pipeline geometry
  int n_sms = 148;
  int ctas_per_sm = 0;
  int tl_ctas_per_sm = 0;
  int is_ctas_per_sm = 0;
  bool serial_streams = false;          // option: never run the second-stream kernels beside the first-stream ones
  bool host_plan = false;               // option: never plan a batch on the device (plan.cuh)
  // per-batch document lists (bm25f_put_lists): a region of `pairs` behind the index's postings; term ids
  // n_terms + 1 + i (term n_terms is the padding between the two regions and is never valid)
  uint64_t dyn_base = 0, dyn_cap = 0;
  uint32_t dyn_terms = 0;
  bool compact_store = false;           // option: release the raw postings after the first bm25f_set_weighting
  bool raw_dropped = false;             // ... done: 8 bytes a posting stay; no re-weighting, no CTA-kernel queries
  std::vector<float> norm_host;         // the weighting in force (compact_store: the only one this handle will ever serve)
  unsigned long long* d_term_offsets = nullptr;   // the device planner's copies of term_offsets / term_field
  uint8_t* d_term_field = nullptr;
  unsigned int* h_ctr = nullptr;        // pinned: the device planner's counters of the last executed plan (statistics)
  bool stats_from_ctr = false;          // ... which bm25f_get_stats folds in after a synchronize
  uint32_t is_ratio = 1, is_split = 2048, is_or_limit = 40000;   // candidate-driven AND: cost of a lookup in postings, candidates per item
  static constexpr int EV_RING = 32;   // executes whose timings may be pending at once
  cudaEvent_t ev[EV_RING][6] = {};     // [0..3] step phases; [4], [5] bracket the stream kernel alone
  int ev_head = 0;                     // next slot to use
  int ev_pending = 0;                  // slots recorded but not yet folded into the stats
  bm25f_stats stats{};
  uint64_t device_bytes = 0;
  unsigned long long* d_prof = nullptr;   // BM25F_PROFILE builds only
  // Grow-only workspaces reused by bm25f_search_batch / bm25f_submit (no cudaMalloc / cudaFree per call).
  // There are two, used alternately, so that the host can plan and upload batch i + 1 while the GPU
  // still runs batch i.
  struct Arena {
    unsigned char* d = nullptr;           // device: plan records, partial lists, results
    size_t d_cap = 0;
    unsigned char* h = nullptr;           // pinned staging of the plan records
    size_t h_cap = 0;
    unsigned char* h_out = nullptr;       // pinned landing zone of a submitted batch's results
    size_t h_out_cap = 0;
    cudaEvent_t ev_ready = nullptr;       // the plan's records are on the device (copy stream)
    cudaEvent_t ev_done = nullptr;        // a submitted batch's results are in h_out
    cudaEvent_t ev_scored = nullptr;      // ... are final on the device (the copy to h_out runs on d2h_stream)
    bm25f_plan* submitted = nullptr;      // submitted and not yet collected
  } arenas[2];
  int arena_next = 0;
  cudaStream_t copy_stream = nullptr;    // plan uploads, so that they do not queue behind the running batch
  cudaStream_t d2h_stream = nullptr;     // results of submitted batches, so that the next batch's kernels do not queue behind them
  PlanPool* pool = nullptr;              // created on the first large batch
};

struct bm25f_plan {
  bm25f_handle* h = nullptr;
  uint32_t Q = 0, n_leaves = 0, n_items = 0, n_parts = 0, T = 0;
  uint32_t n_w4 = 0, n_w8 = 0;            // stream-kernel items / team-kernel items; the rest are CTA items
  ItemRec* d_items_w4 = nullptr;
  ItemRec* d_items_w8 = nullptr;
  uint32_t n_is = 0;                      // candidate-driven items
  ItemRec* d_items_is = nullptr;
  int k = 0, kp = 1, cap = 1024;
  uint64_t postings = 0;
  uint64_t postings_cls[4] = {0, 0, 0, 0};   // per kernel class: stream, team, CTA, candidate-driven
  LeafRec* d_leaves = nullptr;
  QueryRec* d_queries = nullptr;
  ItemRec* d_items = nullptr;
  uint32_t* d_bounds = nullptr;
  unsigned long long* d_part_keys = nullptr;
  unsigned long long* d_keys = nullptr;
  unsigned long long* d_totals = nullptr;
  float* d_scores = nullptr;
  uint32_t* d_docids = nullptr;
  uint32_t* d_counts = nullptr;
  size_t smem_score = 0;
  bool owns_memory = true;      // false: buffers live in one of the handle's arenas (bm25f_search_batch)
  int arena = -1;               // which one
  bool final_mode = false;      // planned with a final() step: 96-bit keys, float64 results (bm25f_fetch_final)
  unsigned int* d_part_lo = nullptr;   // final mode: low halves of the partial lists' keys
  double* d_final = nullptr;           // final mode: [Q * k] final values
  bool submitted = false;       // bm25f_submit: bm25f_execute also brings the results to the arena's pinned h_out
  bool simple_kernel = false;   // k_score_topk instead of k_score_pipe (option, or a non-positive leaf weight)
  bool device_planned = false;  // plan.cuh: the items and their counts exist only on the device (d_ctr)
  unsigned int* d_ctr = nullptr;
};

namespace {

size_t score_smem_bytes(uint32_t S, int cap) { return (size_t)cap * 8 + (size_t)S * 7; }

size_t pipe_smem_bytes(const bm25f_handle* h, int cap);

int key_capacity(int k, int nt) {
  int need = k + 2 * nt;
  int cap = 1024;
  while (cap < need) cap <<= 1;
  return cap;
}

size_t pipe_smem_bytes(const bm25f_handle* h, int cap) {
  size_t b = (score_smem_bytes(h->S, cap) + 15) & ~(size_t)15;
  b += (size_t)h->stages * h->chunk * sizeof(uint2);
  b += (size_t)HOTCAP * sizeof(uint16_t);
  return b;
}

size_t team_smem_bytes(const bm25f_handle* h) { return (size_t)h->tl_warps * h->tl_slot_bytes + sizeof(TeamShared); }

size_t stream_smem_bytes(uint32_t warps, uint32_t slot_bytes) {
  // slots, tails, hot list, hot counter, and (16-byte aligned) the leaf records
  return (size_t)warps * (slot_bytes + ST_MAX_LEAVES * 256 + ST_HOT * 2 + 4) + 16 + (size_t)warps * ST_MAX_LEAVES * 32;
}

int pipe_prune_at(int k) { return std::max(2 * k, 256); }

// room for a full hot list on top of an unpruned buffer, and for the walk-all-candidates path
int pipe_key_capacity(int k, int nc) {
  int need = std::max(pipe_prune_at(k) + HOTCAP, k + 2 * nc);
  int cap = 1024;
  while (cap < need) cap <<= 1;
  return cap;
}

template <typename T>
int dev_alloc(T** p, size_t n, bm25f_handle* h = nullptr) {
  *p = nullptr;
  if (n == 0) n = 1;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), n * sizeof(T));
  if (e != cudaSuccess) return fail(BM25F_ENOMEM, "cudaMalloc(%zu bytes): %s", n * sizeof(T), cudaGetErrorString(e));
  if (h) h->device_bytes += n * sizeof(T);
  return 0;
}

// Fold the timings of the oldest `n` pending executes into the running sums (waits for them).
int fold_events(bm25f_handle* h, int n) {
  while (n-- > 0 && h->ev_pending > 0) {
    const int slot = (h->ev_head - h->ev_pending + 2 * bm25f_handle::EV_RING) % bm25f_handle::EV_RING;
    cudaEvent_t* e = h->ev[slot];
    CU(cudaEventSynchronize(e[3]));
    float a = 0, b = 0, c = 0, d = 0;
    CU(cudaEventElapsedTime(&a, e[0], e[1]));
    CU(cudaEventElapsedTime(&b, e[1], e[2]));
    CU(cudaEventElapsedTime(&c, e[2], e[3]));
    CU(cudaEventElapsedTime(&d, e[0], e[3]));
    float f = 0;
    CU(cudaEventElapsedTime(&f, e[4], e[5]));
    static const bool trace = getenv("BM25F_TRACE") != nullptr;
    if (trace && h->stats.n_executes > 0) {
      // idle time of the stream between the previous execute's last kernel and this one's first
      cudaEvent_t* prev = h->ev[(slot + bm25f_handle::EV_RING - 1) % bm25f_handle::EV_RING];
      float gap = 0;
      if (cudaEventElapsedTime(&gap, prev[3], e[0]) == cudaSuccess)
        fprintf(stderr, "[bm25f execute] gap %.3f ms, bounds %.3f, score %.3f (stream %.3f), merge %.3f\n", gap, a, b, f, c);
      else
        cudaGetLastError();
    }
    h->stats.ms_stream += f;
    h->stats.ms_bounds += a;
    h->stats.ms_score += b;
    h->stats.ms_merge += c;
    h->stats.ms_total += d;
    h->stats.n_executes += 1;
    --h->ev_pending;
  }
  return 0;
}

}  // namespace

extern "C" {

int bm25f_abi_version(void) { return BM25F_ABI_VERSION; }

const char* bm25f_last_error(void) { return g_err.c_str(); }

void bm25f_destroy(bm25f_handle* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaFree(h->d_docids);
  cudaFree(h->d_payload);
  cudaFree(h->d_lb);
  cudaFree(h->d_pairs);
  cudaFree(h->d_norm);
  cudaFree(h->d_final_add);
  cudaFree(h->d_final_blk);
  cudaFree(h->d_prof);
  cudaFree(h->d_term_offsets);
  cudaFree(h->d_term_field);
  if (h->h_ctr) cudaFreeHost(h->h_ctr);
  for (auto& A : h->arenas) {
    cudaFree(A.d);
    if (A.h) cudaFreeHost(A.h);
    if (A.h_out) cudaFreeHost(A.h_out);
    if (A.ev_ready) cudaEventDestroy(A.ev_ready);
    if (A.ev_done) cudaEventDestroy(A.ev_done);
    if (A.ev_scored) cudaEventDestroy(A.ev_scored);
  }
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  if (h->d2h_stream) cudaStreamDestroy(h->d2h_stream);
  for (auto& set : h->ev)
    for (auto& e : set)
      if (e) cudaEventDestroy(e);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h->pool;
  delete h;
}

int bm25f_create(const bm25f_index_desc* desc, int device, const bm25f_options* opts, bm25f_handle** out) {
  if (!desc || !out) return fail(BM25F_EINVAL, "null argument");
  *out = nullptr;
  if (desc->abi_version != BM25F_ABI_VERSION)
    return fail(BM25F_EABI, "ABI mismatch: caller %u, library %d", desc->abi_version, BM25F_ABI_VERSION);
  if (desc->n_fields == 0 || desc->n_fields > 255) return fail(BM25F_EINVAL, "n_fields must be 1..255");
  if (desc->n_docs_all >= 0xFFFFFFFFull || desc->doc_base + desc->n_docs_all >= 0xFFFFFFFFull)
    return fail(BM25F_EINVAL, "document numbers must fit 32 bits");
  if (!desc->term_offsets || !desc->term_field || !desc->len_bytes || (desc->n_postings && (!desc->docids || !desc->tfs)))
    return fail(BM25F_EINVAL, "null index array");
  if (desc->term_offsets[0] != 0 || desc->term_offsets[desc->n_terms] != desc->n_postings)
    return fail(BM25F_EINVAL, "term_offsets does not span n_postings");
  for (uint64_t t = 0; t < desc->n_terms; ++t) {
    if (desc->term_offsets[t + 1] < desc->term_offsets[t]) return fail(BM25F_EINVAL, "term_offsets not monotonic at %llu", (unsigned long long)t);
    if (desc->term_offsets[t + 1] - desc->term_offsets[t] > 0xFFFFFFFFull) return fail(BM25F_EINVAL, "posting list too long");
    if (desc->term_field[t] >= desc->n_fields) return fail(BM25F_EINVAL, "term_field out of range at %llu", (unsigned long long)t);
  }
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(BM25F_EINVAL, "device %d not present (%d visible)", device, ndev);
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) return fail(BM25F_ECUDA, "libbm25f is built for sm_100a; device is sm_%d%d", prop.major, prop.minor);

  bm25f_handle* h = new (std::nothrow) bm25f_handle();
  if (!h) return fail(BM25F_ENOMEM, "host allocation failed");
  h->device = device;
  h->n_sms = prop.multiProcessorCount;
  h->n_docs = desc->n_docs_all;
  h->n_terms = desc->n_terms;
  h->n_postings = desc->n_postings;
  h->doc_base = desc->doc_base;
  h->n_fields = desc->n_fields;
  if (opts) {
    if (opts->tile_docs) h->S = opts->tile_docs;
    if (opts->threads) h->NT = opts->threads;
    if (opts->split_postings) h->split = opts->split_postings;
    if (opts->variant) h->variant = opts->variant;
    if (opts->subtile_docs) h->st_slot_bytes = opts->subtile_docs * 4u;
    if (opts->warp_split) h->wsplit = opts->warp_split;
    if (opts->chunk_postings) h->chunk = opts->chunk_postings;
    if (opts->stages) h->stages = opts->stages;
    if (opts->stream_warps) h->st_warps = opts->stream_warps;
    if (opts->prefetch_postings) h->st_pf = opts->prefetch_postings == 0xFFFFFFFFu ? 0u : opts->prefetch_postings;
  }
  if (opts) {
    if (opts->cta_warps) h->tl_warps = opts->cta_warps;
    if (opts->cta_prefetch) h->tl_prefetch = opts->cta_prefetch == 0xFFFFFFFFu ? 0u : opts->cta_prefetch;
    if (opts->cta_split) h->tl_split = opts->cta_split;
    if (opts->cta_slice_docs) h->tl_slot_bytes = opts->cta_slice_docs * 4u;
  }
  if (h->tl_slot_bytes < 512 || (h->tl_slot_bytes & 511)) { delete h; return fail(BM25F_EINVAL, "cta_slice_docs must be a multiple of 128, at least 128"); }
  if (opts) {
    if (opts->isect_ratio) h->is_ratio = opts->isect_ratio;
    if (opts->isect_split) h->is_split = opts->isect_split;
    if (opts->isect_or_limit) h->is_or_limit = opts->isect_or_limit == 0xFFFFFFFFu ? 0u : opts->isect_or_limit;
  }
  if (!opts || !opts->isect_or_limit) {
    // The sweep a flat OR costs on the stream kernel grows with the shard's document space, the lookups of the
    // candidate-driven kernel do not: the break-even moves with n_docs.  (Measured on config 2: 40000 at 1M documents;
    // on a 125k-document shard 5000 runs the step in 0.40 ms, 40000 in 0.63 ms.)
    h->is_or_limit = (uint32_t)std::min<uint64_t>(40000, std::max<uint64_t>(2000, 40000ull * h->n_docs / 1000000ull));
  }
  if (opts) h->serial_streams = opts->serial_streams != 0;
  if (opts) h->host_plan = opts->host_plan != 0;
  if (opts) h->compact_store = opts->compact_store != 0;
  if (h->variant > 5) { delete h; return fail(BM25F_EINVAL, "variant must be 0 (auto), 1 (pipeline), 2 (direct loads), 3 (warp streams), 4 (warp teams) or 5 (candidate-driven)"); }
  if (h->tl_warps < 1 || h->tl_warps > (uint32_t)TM_MAX_WARPS) { delete h; return fail(BM25F_EINVAL, "cta_warps must be 1..%d", TM_MAX_WARPS); }
  if (h->st_slot_bytes < 512 || (h->st_slot_bytes & 511)) { delete h; return fail(BM25F_EINVAL, "subtile_docs must be a multiple of 128, at least 128"); }
  if (h->st_warps < 1 || h->st_warps > (uint32_t)ST_MAX_WARPS) { delete h; return fail(BM25F_EINVAL, "stream_warps must be 1..%d", ST_MAX_WARPS); }
  if (h->st_pf & (ST_PF_CHUNK - 1u)) { delete h; return fail(BM25F_EINVAL, "prefetch_postings must be a multiple of %u", ST_PF_CHUNK); }
  if (h->variant != 4 && h->variant != 1 && h->variant != 2 && stream_smem_bytes(h->st_warps, h->st_slot_bytes) > (size_t)prop.sharedMemPerBlockOptin) {
    const size_t need = stream_smem_bytes(h->st_warps, h->st_slot_bytes);
    delete h;
    return fail(BM25F_EINVAL, "stream_warps x subtile_docs needs %zu bytes of shared memory (> %zu)", need, (size_t)prop.sharedMemPerBlockOptin);
  }
  if ((h->variant == 4 || h->variant == 0) && team_smem_bytes(h) > (size_t)prop.sharedMemPerBlockOptin) {
    const size_t need = team_smem_bytes(h);
    delete h;
    return fail(BM25F_EINVAL, "cta_warps x subtile_docs needs %zu bytes of shared memory (> %zu)", need, (size_t)prop.sharedMemPerBlockOptin);
  }
  if (h->chunk < 64 || (h->chunk & 15) || h->chunk > 8192) { delete h; return fail(BM25F_EINVAL, "chunk_postings must be a multiple of 16 in 64..8192"); }
  if (h->stages < 2 || h->stages > (uint32_t)PIPE_MAX_STAGES) { delete h; return fail(BM25F_EINVAL, "stages must be 2..%d", PIPE_MAX_STAGES); }
  if (h->S < 256 || h->S > 65536 || (h->S & 3)) { delete h; return fail(BM25F_EINVAL, "tile_docs must be a multiple of 4 in 256..65536"); }
  if (h->NT < 64 || h->NT > 512 || (h->NT & 31)) { delete h; return fail(BM25F_EINVAL, "threads must be a multiple of 32 in 64..512"); }
  h->term_offsets.assign(desc->term_offsets, desc->term_offsets + desc->n_terms + 1);
  h->term_field.assign(desc->term_field, desc->term_field + desc->n_terms);

#define CUH(x)                                                          \
  do {                                                                  \
    cudaError_t e_ = (x);                                               \
    if (e_ != cudaSuccess) {                                            \
      int rc_ = fail(e_ == cudaErrorMemoryAllocation ? BM25F_ENOMEM : BM25F_ECUDA, "%s: %s", #x, cudaGetErrorString(e_)); \
      bm25f_destroy(h);                                                 \
      return rc_;                                                       \
    }                                                                   \
  } while (0)
#define RCH(x)                       \
  do {                               \
    int rc_ = (x);                   \
    if (rc_) { bm25f_destroy(h); return rc_; } \
  } while (0)

  CUH(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
  CUH(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
  CUH(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
  CUH(cudaStreamCreateWithFlags(&h->d2h_stream, cudaStreamNonBlocking));
  for (auto& A : h->arenas) {
    CUH(cudaEventCreateWithFlags(&A.ev_ready, cudaEventDisableTiming));
    CUH(cudaEventCreateWithFlags(&A.ev_done, cudaEventDisableTiming));
    CUH(cudaEventCreateWithFlags(&A.ev_scored, cudaEventDisableTiming));
  }
  CUH(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
  CUH(cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming));
  h->stream = h->own_stream;
  for (auto& set : h->ev)
    for (auto& e : set) CUH(cudaEventCreate(&e));

  uint64_t P = desc->n_postings;
  const size_t pad = 1024;   // rows / prefetch chunks may run past the last posting of the last list
  RCH(dev_alloc(&h->d_norm, (size_t)(h->n_fields + 1) * 256, h));
  CUH(cudaMemsetAsync(h->d_norm, 0, (size_t)(h->n_fields + 1) * 256 * sizeof(float), h->stream));   // the pseudo-field's row stays 0: impact = tf / (tf + 0) = 1
  // temporaries for compaction and packing
  uint32_t* d_raw_docids = nullptr;
  float* d_tfs = nullptr;
  uint8_t* d_len = nullptr;
  uint8_t* d_deleted = nullptr;
  unsigned long long* d_offs = nullptr;
  unsigned long long* d_new_offs = nullptr;
  uint32_t* d_counts = nullptr;
  int* d_flag = nullptr;
  auto free_tmp = [&]() {
    cudaFree(d_raw_docids); cudaFree(d_tfs); cudaFree(d_len); cudaFree(d_deleted); cudaFree(d_offs);
    cudaFree(d_new_offs); cudaFree(d_counts); cudaFree(d_flag);
  };
#define CUT(x)                                                          \
  do {                                                                  \
    cudaError_t e_ = (x);                                               \
    if (e_ != cudaSuccess) {                                            \
      int rc_ = fail(e_ == cudaErrorMemoryAllocation ? BM25F_ENOMEM : BM25F_ECUDA, "%s: %s", #x, cudaGetErrorString(e_)); \
      free_tmp();                                                       \
      bm25f_destroy(h);                                                 \
      return rc_;                                                       \
    }                                                                   \
  } while (0)
#define RCT(x)                       \
  do {                               \
    int rc_ = (x);                   \
    if (rc_) { free_tmp(); bm25f_destroy(h); return rc_; } \
  } while (0)
  // ---- Every(field) (reference cli.py:9): one more posting list per field with every document that has
  // the field (non-zero length byte), weight 1, on a pseudo-field whose norm row is 0, so that its score is
  // the constant w * 1 (Whoosh scores Every with the query boost).  Deleted documents leave it below.
  std::vector<uint32_t> every_docs;
  {
    std::vector<uint8_t> h_len((size_t)h->n_fields * h->n_docs);
    if (!h_len.empty()) CUT(cudaMemcpy(h_len.data(), desc->len_bytes, h_len.size(), cudaMemcpyDefault));
    h->n_real_terms = h->n_terms;
    for (uint32_t f = 0; f < h->n_fields; ++f) {
      const uint8_t* lb = h_len.data() + (size_t)f * h->n_docs;
      for (uint64_t d = 0; d < h->n_docs; ++d)
        if (lb[d]) every_docs.push_back((uint32_t)d);
      h->term_offsets.push_back(P + every_docs.size());
      h->term_field.push_back((uint8_t)h->n_fields);
    }
    h->n_terms += h->n_fields;
  }
  const uint64_t P_real = P;
  P += every_docs.size();
  h->n_postings = P;
  RCT(dev_alloc(&h->d_docids, P + pad, h));
  RCT(dev_alloc(&d_tfs, std::max<uint64_t>(P, 1)));
  RCT(dev_alloc(&d_len, (size_t)(h->n_fields + 1) * h->n_docs));
  RCT(dev_alloc(&d_flag, 1));
  if (P_real) {
    CUT(cudaMemcpyAsync(h->d_docids, desc->docids, P_real * 4, cudaMemcpyDefault, h->stream));
    CUT(cudaMemcpyAsync(d_tfs, desc->tfs, P_real * 4, cudaMemcpyDefault, h->stream));
  }
  std::vector<float> every_tfs(every_docs.size(), 1.0f);
  if (!every_docs.empty()) {
    CUT(cudaMemcpyAsync(h->d_docids + P_real, every_docs.data(), every_docs.size() * 4, cudaMemcpyHostToDevice, h->stream));
    CUT(cudaMemcpyAsync(d_tfs + P_real, every_tfs.data(), every_tfs.size() * 4, cudaMemcpyHostToDevice, h->stream));
  }
  CUT(cudaMemcpyAsync(d_len, desc->len_bytes, (size_t)h->n_fields * h->n_docs, cudaMemcpyDefault, h->stream));
  CUT(cudaMemsetAsync(d_len + (size_t)h->n_fields * h->n_docs, 0, h->n_docs, h->stream));
  CUT(cudaStreamSynchronize(h->stream));     // every_docs / every_tfs are pageable

  // ---- the lists must hold valid, ascending local docids -------------------------------------------
  if (P_real && h->n_real_terms) {
    unsigned long long* d_chk = nullptr;
    unsigned long long* d_offs_chk = nullptr;
    cudaError_t ec = cudaMalloc(reinterpret_cast<void**>(&d_chk), 8);
    if (ec == cudaSuccess) ec = cudaMalloc(reinterpret_cast<void**>(&d_offs_chk), (h->n_real_terms + 1) * 8);
    unsigned long long first_bad = ~0ull;
    if (ec == cudaSuccess) ec = cudaMemcpyAsync(d_chk, &first_bad, 8, cudaMemcpyHostToDevice, h->stream);
    if (ec == cudaSuccess) ec = cudaMemcpyAsync(d_offs_chk, h->term_offsets.data(), (h->n_real_terms + 1) * 8, cudaMemcpyHostToDevice, h->stream);
    if (ec == cudaSuccess) {
      const unsigned blocks = (unsigned)std::min<uint64_t>((h->n_real_terms + 7) / 8, (uint64_t)h->n_sms * 16);
      k_check_docids<<<blocks, 256, 0, h->stream>>>(h->d_docids, d_offs_chk, h->n_real_terms, (uint32_t)h->n_docs, d_chk);
      ec = cudaGetLastError();
    }
    if (ec == cudaSuccess) ec = cudaMemcpyAsync(&first_bad, d_chk, 8, cudaMemcpyDeviceToHost, h->stream);
    if (ec == cudaSuccess) ec = cudaStreamSynchronize(h->stream);
    cudaFree(d_chk);
    cudaFree(d_offs_chk);
    if (ec != cudaSuccess) { free_tmp(); bm25f_destroy(h); return fail(BM25F_ECUDA, "docid check: %s", cudaGetErrorString(ec)); }
    if (first_bad != ~0ull) {
      free_tmp();
      bm25f_destroy(h);
      return fail(BM25F_EINVAL, "posting list %llu: docids must be < n_docs_all (%llu) and strictly ascending inside a list",
                  (unsigned long long)(first_bad - 1), (unsigned long long)desc->n_docs_all);
    }
  }

  // ---- W9: drop the postings of deleted documents from the device store -----------------------
  if (desc->deleted && P && h->n_terms) {
    RCT(dev_alloc(&d_deleted, h->n_docs));
    RCT(dev_alloc(&d_offs, h->n_terms + 1));
    RCT(dev_alloc(&d_counts, h->n_terms));
    CUT(cudaMemcpyAsync(d_deleted, desc->deleted, h->n_docs, cudaMemcpyDefault, h->stream));
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "offset width");
    CUT(cudaMemcpyAsync(d_offs, h->term_offsets.data(), (h->n_terms + 1) * 8, cudaMemcpyHostToDevice, h->stream));
    const unsigned blocks = (unsigned)std::min<uint64_t>((h->n_terms + 7) / 8, (uint64_t)h->n_sms * 16);
    k_live_counts<<<blocks, 256, 0, h->stream>>>(h->d_docids, d_offs, h->n_terms, d_deleted, d_counts);
    CUT(cudaGetLastError());
    std::vector<uint32_t> counts(h->n_terms);
    CUT(cudaMemcpyAsync(counts.data(), d_counts, h->n_terms * 4, cudaMemcpyDeviceToHost, h->stream));
    CUT(cudaStreamSynchronize(h->stream));
    std::vector<uint64_t> new_offs(h->n_terms + 1);
    new_offs[0] = 0;
    for (uint64_t t = 0; t < h->n_terms; ++t) new_offs[t + 1] = new_offs[t] + counts[t];
    const uint64_t P_live = new_offs[h->n_terms];
    if (P_live != P) {
      float* d_tfs2 = nullptr;
      d_raw_docids = h->d_docids;
      h->d_docids = nullptr;
      h->device_bytes -= (P + pad) * 4;
      RCT(dev_alloc(&h->d_docids, P_live + pad, h));
      RCT(dev_alloc(&d_new_offs, h->n_terms + 1));
      cudaError_t e2 = cudaMalloc(reinterpret_cast<void**>(&d_tfs2), std::max<uint64_t>(P_live, 1) * 4);
      if (e2 != cudaSuccess) { free_tmp(); bm25f_destroy(h); return fail(BM25F_ENOMEM, "cudaMalloc: %s", cudaGetErrorString(e2)); }
      cudaError_t e3 = cudaMemcpyAsync(d_new_offs, new_offs.data(), (h->n_terms + 1) * 8, cudaMemcpyHostToDevice, h->stream);
      if (e3 == cudaSuccess) {
        k_compact_lists<<<blocks, 256, 0, h->stream>>>(d_raw_docids, d_tfs, d_offs, d_new_offs, h->n_terms, d_deleted, h->d_docids, d_tfs2);
        e3 = cudaGetLastError();
      }
      if (e3 == cudaSuccess) e3 = cudaStreamSynchronize(h->stream);
      cudaFree(d_tfs);
      d_tfs = d_tfs2;
      if (e3 != cudaSuccess) { free_tmp(); bm25f_destroy(h); return fail(BM25F_ECUDA, "compaction: %s", cudaGetErrorString(e3)); }
      h->term_offsets.swap(new_offs);
      P = P_live;
      h->n_postings = P;
    }
  }
  RCT(dev_alloc(&h->d_payload, P + pad, h));
  h->dyn_base = P + pad;
  h->dyn_cap = (opts && opts->filter_postings) ? opts->filter_postings : (1u << 20);
  RCT(dev_alloc(&h->d_pairs, P + pad + h->dyn_cap + pad, h));
  CUT(cudaMemsetAsync(h->d_docids + P, 0xFF, pad * 4, h->stream));
  CUT(cudaMemsetAsync(h->d_payload + P, 0, pad * 4, h->stream));
  CUT(cudaMemsetAsync(h->d_pairs + P, 0xFF, (pad + h->dyn_cap + pad) * 8, h->stream));

  CUT(cudaMemsetAsync(d_flag, 0, sizeof(int), h->stream));
  int flag = 0;
  if (P) {
    k_check_tf<<<h->n_sms * 8, 256, 0, h->stream>>>(d_tfs, P, d_flag);
    CUT(cudaGetLastError());
  }
  CUT(cudaMemcpyAsync(&flag, d_flag, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUT(cudaStreamSynchronize(h->stream));
  h->packed = (flag == 0);
  if (!h->packed) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&h->d_lb), P + pad);
    if (e != cudaSuccess) { free_tmp(); bm25f_destroy(h); return fail(BM25F_ENOMEM, "cudaMalloc: %s", cudaGetErrorString(e)); }
    h->device_bytes += P + pad;
    CUT(cudaMemsetAsync(h->d_lb + P, 0, pad, h->stream));
  }
  // runs of consecutive posting lists that belong to the same field
  uint64_t t = 0;
  while (t < h->n_terms) {
    uint64_t t2 = t;
    const uint8_t f = h->term_field[t];
    while (t2 < h->n_terms && h->term_field[t2] == f) ++t2;
    const uint64_t b = h->term_offsets[t], e = h->term_offsets[t2];
    if (e > b) {
      const uint64_t n = e - b;
      const unsigned blocks = (unsigned)std::min<uint64_t>((n + 255) / 256, (uint64_t)h->n_sms * 16);
      k_pack_postings<<<blocks, 256, 0, h->stream>>>(h->d_docids, d_tfs, d_len + (size_t)f * h->n_docs, nullptr, b, e,
                                                      h->packed ? 1 : 0, h->d_payload, h->d_lb);
      CUT(cudaGetLastError());
    }
    t = t2;
  }
  // the device planner's view of the posting lists (after the compaction above)
  RCT(dev_alloc(&h->d_term_offsets, h->n_terms + 2 + BM25F_MAX_FILTER_LISTS, h));
  RCT(dev_alloc(&h->d_term_field, h->n_terms + 2 + BM25F_MAX_FILTER_LISTS, h));
  CUT(cudaMemcpyAsync(h->d_term_offsets, h->term_offsets.data(), (h->n_terms + 1) * 8, cudaMemcpyHostToDevice, h->stream));
  if (h->n_terms) CUT(cudaMemcpyAsync(h->d_term_field, h->term_field.data(), h->n_terms, cudaMemcpyHostToDevice, h->stream));
  CUT(cudaHostAlloc(reinterpret_cast<void**>(&h->h_ctr), PL_CTR_BYTES, cudaHostAllocDefault));
  memset(h->h_ctr, 0, PL_CTR_BYTES);
  CUT(cudaStreamSynchronize(h->stream));
  free_tmp();
#undef RCT

  // kernel attributes: opt in to the large dynamic shared memory carve-out once
  const int cap_max = key_capacity(BM25F_MAX_K, (int)h->NT);
  const size_t smem_max = std::max(pipe_smem_bytes(h, pipe_key_capacity(BM25F_MAX_K, (int)h->NT)),
                                   score_smem_bytes(h->S, cap_max));
  if (smem_max > (size_t)prop.sharedMemPerBlockOptin) {
    bm25f_destroy(h);
    return fail(BM25F_EINVAL, "tile_docs=%u needs %zu bytes of shared memory (> %zu)", h->S, smem_max, (size_t)prop.sharedMemPerBlockOptin);
  }
  // The attribute is per-function state shared by every handle in the process: always opt in to
  // the device maximum so that engines with different tile sizes can coexist.
  const int optin = (int)prop.sharedMemPerBlockOptin;
  {
    const void* wfns[7] = {(const void*)k_score_stream<1, false>, (const void*)k_score_stream<4, false>, (const void*)k_score_team,
                           (const void*)k_score_stream<1, true>, (const void*)k_score_stream<4, true>,
                           (const void*)k_score_stream<8, false>, (const void*)k_score_stream<8, true>};
    for (const void* fn : wfns) {
      cudaFuncAttributes fa;
      CUH(cudaFuncGetAttributes(&fa, fn));
      CUH(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes));
    }
    const void* fns[2] = {(const void*)k_score_topk, (const void*)k_score_pipe};
    for (const void* fn : fns) {
      cudaFuncAttributes fa;
      CUH(cudaFuncGetAttributes(&fa, fn));
      CUH(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - (int)fa.sharedSizeBytes));
      if (smem_max + fa.sharedSizeBytes > (size_t)optin) {
        bm25f_destroy(h);
        return fail(BM25F_EINVAL, "tile_docs=%u needs %zu bytes of shared memory (> %d)", h->S,
                    smem_max + fa.sharedSizeBytes, optin);
      }
    }
  }
#ifdef BM25F_PROFILE
  CUH(cudaMalloc(reinterpret_cast<void**>(&h->d_prof), 16 * sizeof(unsigned long long)));
  CUH(cudaMemset(h->d_prof, 0, 16 * sizeof(unsigned long long)));
#endif
  h->stats.tile_docs = h->S;
  h->stats.threads = h->NT;
  h->stats.packed_payload = h->packed ? 1u : 0u;
  h->stats.device_bytes = h->device_bytes;
  *out = h;
  return 0;
#undef CUH
#undef RCH
#undef CUT
}

int bm25f_set_weighting(bm25f_handle* h, const float* norm) {
  if (!h || !norm) return fail(BM25F_EINVAL, "null argument");
  CU(cudaSetDevice(h->device));
  std::vector<int> weight_only(h->n_fields + 1, 0);
  for (uint32_t f = 0; f < h->n_fields; ++f) {
    // a row of -1: the field is not scorable, its postings score their weight (Whoosh's WeightScorer)
    bool all_neg1 = true;
    for (uint32_t i = 0; i < 256; ++i) all_neg1 = all_neg1 && norm[f * 256 + i] == -1.0f;
    weight_only[f] = all_neg1 ? 1 : 0;
    if (all_neg1) continue;
    for (uint32_t i = f * 256; i < (f + 1) * 256; ++i)
      if (!(norm[i] > 0.0f) || !std::isfinite(norm[i])) return fail(BM25F_EINVAL, "norm table entry %u is not a positive finite number (or the whole row -1: field not scorable)", i);
  }
  if (h->raw_dropped) {
    if (memcmp(h->norm_host.data(), norm, (size_t)h->n_fields * 256 * sizeof(float)) == 0) return 0;   // the same weighting again
    return fail(BM25F_EINVAL, "compact_store: the raw postings were released after the first bm25f_set_weighting; "
                              "create another engine to score with a different weighting");
  }
  CU(cudaMemcpyAsync(h->d_norm, norm, (size_t)h->n_fields * 256 * sizeof(float), cudaMemcpyHostToDevice, h->stream));
  // refresh the per-posting impacts (one streaming pass over the store per field run)
  uint64_t t = 0;
  while (t < h->n_terms) {
    uint64_t t2 = t;
    const uint8_t f = h->term_field[t];
    while (t2 < h->n_terms && h->term_field[t2] == f) ++t2;
    const uint64_t b = h->term_offsets[t], e = h->term_offsets[t2];
    if (e > b) {
      const unsigned blocks = (unsigned)std::min<uint64_t>((e - b + 255) / 256, (uint64_t)h->n_sms * 16);
      k_impacts<<<blocks, 256, 0, h->stream>>>(h->d_docids, h->d_payload, h->d_lb, h->d_norm + (size_t)f * 256, b, e, h->packed ? 1 : 0, weight_only[f], h->d_pairs);
      CU(cudaGetLastError());
    }
    t = t2;
  }
  CU(cudaStreamSynchronize(h->stream));
  h->have_weighting = true;
  h->norm_host.assign(norm, norm + (size_t)h->n_fields * 256);
  if (h->compact_store) {
    // the scoring kernels read only the {docid, impact} pairs: 8 of the 16 bytes a posting can go
    const uint64_t n = h->n_postings + 1024;        // (the padded length of the arrays)
    uint64_t freed = 0;
    if (h->d_docids) freed += n * 4;
    if (h->d_payload) freed += n * 4;
    if (h->d_lb) freed += n;
    cudaFree(h->d_docids);
    cudaFree(h->d_payload);
    cudaFree(h->d_lb);
    h->d_docids = nullptr;
    h->d_payload = nullptr;
    h->d_lb = nullptr;
    h->raw_dropped = true;
    h->device_bytes = h->device_bytes > freed ? h->device_bytes - freed : 0;
    h->stats.device_bytes = h->device_bytes;
  }
  return 0;
}

void bm25f_plan_destroy(bm25f_plan* p) {
  if (!p) return;
  if (!p->owns_memory) { delete p; return; }
  if (p->h) cudaSetDevice(p->h->device);
  cudaFree(p->d_leaves);
  cudaFree(p->d_queries);
  cudaFree(p->d_items);
  cudaFree(p->d_bounds);
  cudaFree(p->d_part_keys);
  cudaFree(p->d_keys);          // the totals live behind the keys
  cudaFree(p->d_scores);
  cudaFree(p->d_docids);
  cudaFree(p->d_counts);
  cudaFree(p->d_part_lo);
  cudaFree(p->d_final);
  delete p;
}

}  // extern "C" (reopened below)

namespace {

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) & ~(a - 1); }

// BM25F_TERM_EVERY(field) -> the field's pseudo posting list; an unknown field matches nothing
// a resolved leaf_term names a posting list of the index, an Every(field) list, or a list of the last bm25f_put_lists
inline bool valid_term(const bm25f_handle* h, uint32_t term) {
  return term < h->n_terms || (term > h->n_terms && term <= h->n_terms + h->dyn_terms);
}

inline uint32_t resolve_term(const bm25f_handle* h, uint32_t term) {
  if (term >= BM25F_TERM_EVERY_BASE && term != BM25F_TERM_UNKNOWN) {
    const uint32_t f = term - BM25F_TERM_EVERY_BASE;
    return f < h->n_fields ? (uint32_t)h->n_real_terms + f : BM25F_TERM_UNKNOWN;
  }
  return term;
}

// order items heaviest-first (longest-processing-time order for the block scheduler) with an O(n)
// bucket pass: exact order inside a quarter-octave of weight does not matter
void order_items(const std::vector<ItemRec>& items, const std::vector<uint64_t>& w, ItemRec* out) {
  constexpr int NB = 256;
  uint32_t count[NB + 1] = {0};
  auto bucket = [](uint64_t x) {
    if (x < 4) return (int)x;
    const int lg = 63 - __builtin_clzll(x);
    return std::min(NB - 1, lg * 4 + (int)((x >> (lg - 2)) & 3));
  };
  for (uint64_t x : w) ++count[NB - 1 - bucket(x)];
  uint32_t sum = 0;
  for (int i = 0; i < NB; ++i) { const uint32_t c = count[i]; count[i] = sum; sum += c; }
  for (size_t i = 0; i < items.size(); ++i) out[count[NB - 1 - bucket(w[i])]++] = items[i];
}

// Work items are cut so that the batch spreads over every warp of the GPU: a single interactive query (the
// reference's use) as well as a 10k-query batch on a 1/8 document shard, where no query alone reaches the
// default item size and the heaviest one would otherwise pin one warp for the whole step.
void item_sizes(const bm25f_handle* h, uint32_t Q, uint64_t total, uint32_t* wsplit_out, uint32_t* is_split_out, uint32_t* tl_split_out) {
  uint32_t wsplit = h->wsplit, is_split = h->is_split, tl_split = h->tl_split;
  // ~2 items per stream-kernel warp; a large batch is not cut finer than 32k postings an item (every item costs the
  // planner and the merge: at 8 shards x 10k queries finer items made the step host-bound)
  const uint64_t per_item = std::max<uint64_t>(Q <= 1024 ? 4096 : 32768, total / ((uint64_t)h->n_sms * 32));
  if (per_item < wsplit) {
    is_split = (uint32_t)std::max<uint64_t>(Q <= 1024 ? 128 : 1024, (uint64_t)is_split * per_item / wsplit);
    tl_split = (uint32_t)std::max<uint64_t>(16384, (uint64_t)tl_split * per_item / wsplit);
    wsplit = (uint32_t)per_item;
  }
  *wsplit_out = wsplit;
  *is_split_out = is_split;
  *tl_split_out = tl_split;
}

// Planner threads of this process: BM25F_PLAN_THREADS, else the host's cores shared out between the ranks of
// the box (torchrun exports LOCAL_WORLD_SIZE; one process per GPU, and all of them plan at the same time
// because the collectives keep them in step), at most 8.
unsigned plan_thread_budget() {
  static const unsigned budget = [] {
    if (const char* e = getenv("BM25F_PLAN_THREADS")) {
      const int v = atoi(e);
      if (v >= 1) return (unsigned)std::min(v, 8);
    }
    unsigned hw = std::max(1u, std::thread::hardware_concurrency());
    unsigned local = 1;
    if (const char* e = getenv("LOCAL_WORLD_SIZE")) local = (unsigned)std::max(1, atoi(e));
    return std::min(8u, std::max(1u, hw / local));
  }();
  return budget;
}

// Batches the warp kernels serve alone are planned on the device (plan.cuh): the host checks eligibility, stages the
// caller's arrays in the arena's pinned memory and enqueues one copy and three small kernels on the copy stream.
// *done stays false when the batch is not eligible (the host planner then runs, and reports malformed input).
constexpr uint32_t DEVICE_PLAN_MIN_Q = 256;   // below this the host plans faster than three launches and full grids cost

int prepare_on_device(bm25f_handle* h, const bm25f_query_batch* b, int k, bm25f_plan** out, bool* done) {
  *done = false;
  const uint32_t Q = b->n_queries, NL = b->n_leaves;
  static const bool trace = getenv("BM25F_TRACE") != nullptr;
#define DECLINE(why)                                                                \
  do {                                                                              \
    if (trace) fprintf(stderr, "[bm25f prepare] host planner: a query %s\n", why);  \
    return 0;                                                                       \
  } while (0)
  // Eligibility in two branch-free passes (this runs once a batch on the submitting thread: at 8 ranks x 10k queries
  // it was a third of the host's step).  The batch's postings only size the work items: in a large batch every 8th
  // leaf is looked up (the random reads of term_offsets were most of the time).
  const auto t_a = std::chrono::steady_clock::now();
  const uint32_t* qoff = b->query_leaf_offsets;
  const uint8_t* qng = b->query_n_groups;
  const uint8_t* lgrp = b->leaf_group;
  const uint32_t* lterm = b->leaf_term;
  const float* lw = b->leaf_weight;
  // (1) per query: leaf range, at most 8 leaves and groups, groups non-decreasing and below n_groups (a NOT leaf is 0xFF)
  uint32_t bad_q = 0;
  for (uint32_t qi = 0; qi < Q; ++qi) {
    const uint32_t a = qoff[qi], e = qoff[qi + 1], G = qng[qi];
    if (e < a || e > NL) DECLINE("has a bad leaf range");
    bad_q |= (e - a > (uint32_t)PL_MAX_LEAVES) | (G > (uint32_t)PL_MAX_LEAVES);
    uint32_t prev_g = 0, bad = 0;
    for (uint32_t i = a; i < e; ++i) {
      const uint32_t g = lgrp[i];
      bad |= (g >= G) | (g < prev_g);
      prev_g = g;
    }
    bad_q |= bad;
  }
  if (bad_q) DECLINE("has more than 8 leaves or groups, a NOT clause or malformed groups");
  // (2) per leaf: finite weight; a known term must be in range and carry a positive weight (an unknown term's leaf is
  // dropped: its weight - 0 for a term no shard knows - does not matter)
  const uint32_t n_lists = (uint32_t)h->n_terms;                   // (n_real_terms + the Every lists)
  const uint32_t dyn_lo = (uint32_t)h->n_terms + 1u, dyn_hi = (uint32_t)h->n_terms + h->dyn_terms;   // bm25f_put_lists
  const uint32_t n_fields = h->n_fields;
  uint32_t bad_l = 0;
  for (uint32_t i = 0; i < NL; ++i) {
    const uint32_t t = lterm[i];
    const float w = lw[i];
    const uint32_t unknown = (t == BM25F_TERM_UNKNOWN) | ((t >= BM25F_TERM_EVERY_BASE) & (t - BM25F_TERM_EVERY_BASE >= n_fields));
    const uint32_t every = (t >= BM25F_TERM_EVERY_BASE) & (unknown ^ 1u);
    const uint32_t finite = (std::fabs(w) <= 3.402823466e+38f);               // false for NaN and infinities
    const uint32_t in_range = (t < n_lists) | ((t >= dyn_lo) & (t <= dyn_hi));
    bad_l |= (finite ^ 1u) | ((unknown ^ 1u) & (((every ^ 1u) & (in_range ^ 1u)) | (uint32_t)!(w > 1e-30f)));
  }
  if (bad_l) DECLINE("has a non-finite or non-positive weight, or names a posting list out of range");
  const uint32_t sample = NL >= 8192 ? 8u : 1u;
  uint64_t total = 0;
  for (uint32_t i = 0; i < NL; i += sample) {
    const uint32_t term = resolve_term(h, lterm[i]);
    if (term != BM25F_TERM_UNKNOWN && term < h->n_terms) total += h->term_offsets[term + 1] - h->term_offsets[term];
  }
  total *= sample;
#undef DECLINE
  const auto t_b = std::chrono::steady_clock::now();
  uint32_t wsplit, is_split, tl_split;
  item_sizes(h, Q, total, &wsplit, &is_split, &tl_split);

  const int slot = h->arena_next;
  bm25f_handle::Arena& A = h->arenas[slot];
  if (A.submitted) return fail(BM25F_EINVAL, "two submitted batches are in flight: bm25f_collect the oldest one first");
  h->arena_next ^= 1;

  // pinned staging: the caller's arrays, back to back
  size_t hoff = 0;
  auto htake = [&](size_t bytes) { const size_t o = hoff; hoff += align_up(bytes); return o; };
  const size_t i_qoff = htake((size_t)(Q + 1) * 4), i_ng = htake(Q), i_term = htake((size_t)NL * 4), i_w = htake((size_t)NL * 4),
               i_g = htake(NL);
  const size_t in_bytes = hoff;
  if (A.h_cap < in_bytes) {
    if (A.h) cudaFreeHost(A.h);
    A.h = nullptr;
    A.h_cap = 0;
    const size_t cap = align_up(in_bytes * 2 + (1u << 20), 1u << 20);
    cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&A.h), cap, cudaHostAllocDefault);
    if (e != cudaSuccess) return fail(BM25F_ENOMEM, "cudaHostAlloc(%zu): %s", cap, cudaGetErrorString(e));
    A.h_cap = cap;
  }
  memcpy(A.h + i_qoff, b->query_leaf_offsets, (size_t)(Q + 1) * 4);
  memcpy(A.h + i_ng, b->query_n_groups, Q);
  memcpy(A.h + i_term, b->leaf_term, (size_t)NL * 4);
  memcpy(A.h + i_w, b->leaf_weight, (size_t)NL * 4);
  memcpy(A.h + i_g, b->leaf_group, NL);

  // every query may be cut into max_split items at most, so the item array cannot overflow
  // (the slack shrinks with k: the partial lists, k keys an item, stay below ~1 GB)
  const uint32_t slack = (uint32_t)std::min<size_t>(1u << 20, std::max<size_t>(65536, ((size_t)1 << 30) / ((size_t)k * 8)));
  const uint32_t max_split = 4u + slack / Q;
  const size_t item_cap = (size_t)Q * max_split;
  size_t off = 0;
  auto take = [&](size_t bytes) { const size_t o = off; off += align_up(bytes); return o; };
  const size_t o_in = take(in_bytes), o_leaves = take((size_t)NL * sizeof(LeafRec)), o_queries = take((size_t)Q * sizeof(QueryRec)),
               o_items = take(item_cap * sizeof(ItemRec)), o_tmp = take((size_t)Q * sizeof(uint4)), o_ctr = take(PL_CTR_BYTES),
               o_part = take(item_cap * k * 8), o_keys = take((size_t)Q * k * 8), o_tot = take((size_t)(Q + 8) * 8),
               o_sc = take((size_t)Q * k * 4), o_doc = take((size_t)Q * k * 4), o_cnt = take((size_t)Q * 4);
  if (off > A.d_cap) {
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaStreamSynchronize(h->copy_stream));
    cudaFree(A.d);
    A.d = nullptr;
    A.d_cap = 0;
    const size_t cap = align_up(off + off / 2, 1u << 20);
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&A.d), cap);
    if (e != cudaSuccess) return fail(BM25F_ENOMEM, "cudaMalloc(%zu): %s", cap, cudaGetErrorString(e));
    A.d_cap = cap;
  }
  bm25f_plan* p = new (std::nothrow) bm25f_plan();
  if (!p) return fail(BM25F_ENOMEM, "host allocation failed");
  unsigned char* d = A.d;
  p->h = h;
  p->Q = Q;
  p->k = k;
  p->kp = 1;
  while (p->kp < k) p->kp <<= 1;
  p->cap = pipe_key_capacity(k, (int)h->NT);
  p->n_leaves = NL;
  p->T = 1;
  p->owns_memory = false;
  p->arena = slot;
  p->device_planned = true;
  p->n_w4 = 1;                       // "maybe": the kernels read the counts from d_ctr
  p->n_is = 1;
  p->n_w8 = k <= 32 ? 1 : 0;
  p->n_parts = (uint32_t)item_cap;
  p->d_leaves = reinterpret_cast<LeafRec*>(d + o_leaves);
  p->d_queries = reinterpret_cast<QueryRec*>(d + o_queries);
  p->d_items = reinterpret_cast<ItemRec*>(d + o_items);
  p->d_items_w4 = p->d_items_w8 = p->d_items_is = p->d_items;
  p->d_ctr = reinterpret_cast<unsigned int*>(d + o_ctr);
  p->d_part_keys = reinterpret_cast<unsigned long long*>(d + o_part);
  p->d_keys = reinterpret_cast<unsigned long long*>(d + o_keys);
  p->d_totals = reinterpret_cast<unsigned long long*>(d + o_tot);
  p->d_scores = reinterpret_cast<float*>(d + o_sc);
  p->d_docids = reinterpret_cast<uint32_t*>(d + o_doc);
  p->d_counts = reinterpret_cast<uint32_t*>(d + o_cnt);

  PlanParams pp;
  pp.term_offsets = h->d_term_offsets;
  pp.term_field = h->d_term_field;
  pp.q_off = reinterpret_cast<const uint32_t*>(d + o_in + i_qoff);
  pp.q_ng = d + o_in + i_ng;
  pp.leaf_term = reinterpret_cast<const uint32_t*>(d + o_in + i_term);
  pp.leaf_w = reinterpret_cast<const float*>(d + o_in + i_w);
  pp.leaf_g = d + o_in + i_g;
  pp.leaves = p->d_leaves;
  pp.queries = p->d_queries;
  pp.items = p->d_items;
  pp.tmp = reinterpret_cast<uint4*>(d + o_tmp);
  pp.ctr = p->d_ctr;
  pp.Q = Q;
  pp.n_docs = (uint32_t)h->n_docs;
  pp.n_fields = h->n_fields;
  pp.n_real_terms = (uint32_t)h->n_real_terms;
  pp.max_split = max_split;
  pp.wsplit = wsplit;
  pp.is_split = is_split;
  pp.tl_split = tl_split;
  pp.is_or_limit = h->is_or_limit;
  pp.is_ratio = h->is_ratio;
  pp.st_slot_bytes = h->st_slot_bytes;
  pp.tl_slot_bytes = h->tl_slot_bytes;
  pp.k = k;
  cudaStream_t up = h->copy_stream;
  cudaError_t ce = cudaMemcpyAsync(d + o_in, A.h, in_bytes, cudaMemcpyHostToDevice, up);
  if (ce == cudaSuccess) ce = cudaMemsetAsync(p->d_ctr, 0, PL_CTR_BYTES, up);
  if (ce == cudaSuccess) {
    k_plan_queries<<<(Q + 127) / 128, 128, 0, up>>>(pp);
    k_plan_scan<<<1, 1024, 0, up>>>(pp);
    k_plan_items<<<(Q + 127) / 128, 128, 0, up>>>(pp);
    ce = cudaGetLastError();
  }
  if (ce == cudaSuccess) ce = cudaEventRecord(A.ev_ready, up);
  if (ce != cudaSuccess) {
    delete p;
    return fail(BM25F_ECUDA, "device planner: %s", cudaGetErrorString(ce));
  }
  if (trace) {
    auto us = [](auto x, auto y) { return (double)std::chrono::duration_cast<std::chrono::nanoseconds>(y - x).count() / 1e3; };
    fprintf(stderr, "[bm25f prepare] device planner: check %.0f us, stage + enqueue %.0f us\n", us(t_a, t_b), us(t_b, std::chrono::steady_clock::now()));
  }
  *out = p;
  *done = true;
  return 0;
}

// Host planning + upload.  With use_arena the plan's buffers live in the handle's grow-only
// workspaces (pinned host staging, one device arena): no allocation on the hot path.
int prepare_impl(bm25f_handle* h, const bm25f_query_batch* b, int k, bm25f_plan** out, bool use_arena) {
  if (!h || !b || !out) return fail(BM25F_EINVAL, "null argument");
  *out = nullptr;
  if (k < 1 || k > BM25F_MAX_K) return fail(BM25F_EINVAL, "k must be 1..%d", BM25F_MAX_K);
  if (!h->have_weighting) return fail(BM25F_EINVAL, "bm25f_set_weighting has not been called");
  const uint32_t Q = b->n_queries, NL = b->n_leaves;
  if (Q && (!b->query_leaf_offsets || !b->query_n_groups)) return fail(BM25F_EINVAL, "null query arrays");
  if (NL && (!b->leaf_term || !b->leaf_weight || !b->leaf_group)) return fail(BM25F_EINVAL, "null leaf arrays");
  if (Q && (b->query_leaf_offsets[0] != 0 || b->query_leaf_offsets[Q] != NL)) return fail(BM25F_EINVAL, "query_leaf_offsets does not span n_leaves");
  CU(cudaSetDevice(h->device));
  if (use_arena && !h->host_plan && h->variant == 0 && !h->d_final_add && !b->after_keys && k <= FAST_MAX_K && Q >= DEVICE_PLAN_MIN_Q) {
    bool done = false;
    const int rc = prepare_on_device(h, b, k, out, &done);
    if (rc || done) return rc;
  }

  const uint32_t S = h->S;
  const uint32_t T = (uint32_t)std::max<uint64_t>(1, (h->n_docs + S - 1) / S);

  // pinned staging for the leaf and query records (upper bounds known up front)
  const size_t hl_bytes = align_up((size_t)NL * sizeof(LeafRec)), hq_bytes = align_up((size_t)Q * sizeof(QueryRec));
  std::vector<LeafRec> own_leaves;
  std::vector<QueryRec> own_queries;
  LeafRec* leaves;
  QueryRec* queries;
  const int slot = use_arena ? h->arena_next : 0;
  bm25f_handle::Arena& A = h->arenas[slot];
  if (use_arena) {
    if (A.submitted) return fail(BM25F_EINVAL, "two submitted batches are in flight: bm25f_collect the oldest one first");
    h->arena_next ^= 1;
    // items are appended after planning; reserve generously (grown below if needed)
    const size_t want = hl_bytes + hq_bytes;
    if (A.h_cap < want + (1u << 20)) {
      if (A.h) cudaFreeHost(A.h);
      A.h = nullptr;
      A.h_cap = 0;
      const size_t cap = align_up((want + (1u << 20)) * 2, 1u << 20);
      cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&A.h), cap, cudaHostAllocDefault);
      if (e != cudaSuccess) return fail(BM25F_ENOMEM, "cudaHostAlloc(%zu): %s", cap, cudaGetErrorString(e));
      A.h_cap = cap;
    }
    leaves = reinterpret_cast<LeafRec*>(A.h);
    queries = reinterpret_cast<QueryRec*>(A.h + hl_bytes);
  } else {
    own_leaves.resize(NL);
    own_queries.resize(Q);
    leaves = own_leaves.data();
    queries = own_queries.data();
  }

  uint32_t wsplit, is_split, tl_split;
  {
    uint64_t total = 0;
    for (uint32_t i = 0; i < NL; ++i) {
      const uint32_t term = resolve_term(h, b->leaf_term[i]);
      if (term != BM25F_TERM_UNKNOWN && term < h->n_terms) total += h->term_offsets[term + 1] - h->term_offsets[term];
    }
    item_sizes(h, Q, total, &wsplit, &is_split, &tl_split);
  }
  // Planning is per query and independent: ranges of queries are planned by a few host threads (each
  // into its own item lists and counters), then stitched together.  A query's leaf records live at
  // the positions of its input leaves, so no thread needs another's running totals.
  struct PlanLocal {
    std::vector<ItemRec> items[4];     // 0: warp streams; 1: warp teams; 2: CTA kernels; 3: candidate-driven
    std::vector<uint64_t> item_w[4];
    uint64_t postings = 0, cls_postings[4] = {0, 0, 0, 0};
    uint32_t n_parts = 0;
    bool any_nonpos = false;
    int rc = 0;
    char err[256] = {0};
  };
#define PFAIL(code, ...)                                   \
  do {                                                     \
    L.rc = (code);                                         \
    snprintf(L.err, sizeof L.err, __VA_ARGS__);            \
    return;                                                \
  } while (0)
  auto dummy_leaves = [&](uint32_t a, uint32_t e) {
    for (uint32_t i = a; i < e; ++i) { leaves[i] = LeafRec{}; leaves[i].qleaf0 = i; leaves[i].qnl = 1; }
  };
  const bool final_mode = h->d_final_add != nullptr;
  auto plan_range = [&](uint32_t q_begin, uint32_t q_end, PlanLocal& L) {
    for (uint32_t qi = q_begin; qi < q_end; ++qi) {
    const uint32_t a = b->query_leaf_offsets[qi], e = b->query_leaf_offsets[qi + 1];
    if (e < a || e > NL) PFAIL(BM25F_EINVAL, "query %u: bad leaf range", qi);
    const uint32_t nl = e - a;
    const uint32_t G = b->query_n_groups[qi];
    QueryRec& qr = queries[qi];
    qr = QueryRec{};
    qr.after_key = b->after_keys ? b->after_keys[qi] : 0ull;
    qr.after_lo = (b->after_keys && b->after_lo) ? b->after_lo[qi] : 0u;
    qr.leaf_begin = a;
    qr.part_begin = L.n_parts;
    if (nl > (uint32_t)MAXL) PFAIL(BM25F_EINVAL, "query %u has %u leaves (max %d)", qi, nl, MAXL);
    if (G > 32) PFAIL(BM25F_EINVAL, "query %u has %u groups (max 32)", qi, G);
    if (G == 0 || nl == 0) { dummy_leaves(a, e); continue; }   // null query

    // per-group size; validates group ordering
    uint64_t gsize[32];
    bool gseen[32];
    for (uint32_t g = 0; g < G; ++g) { gsize[g] = 0; gseen[g] = false; }
    uint32_t prev_g = 0, n_neg_in = 0;
    bool all_pos = true, has_dyn = false;
    for (uint32_t i = a; i < e; ++i) {
      const uint32_t g = b->leaf_group[i];
      const bool neg = (g == BM25F_GROUP_NOT);             // a leaf of a NOT clause: excludes, never scores
      if ((!neg && g >= G) || g < prev_g) PFAIL(BM25F_EINVAL, "query %u: leaf_group must be non-decreasing and < n_groups", qi);
      prev_g = g;
      if (!neg) gseen[g] = true;
      const uint32_t term = resolve_term(h, b->leaf_term[i]);
      if (term != BM25F_TERM_UNKNOWN) {
        if (!valid_term(h, term)) PFAIL(BM25F_EINVAL, "query %u: leaf_term %u out of range", qi, b->leaf_term[i]);
        if (term > h->n_terms) has_dyn = true;
        if (!neg) gsize[g] += h->term_offsets[term + 1] - h->term_offsets[term];
      }
      if (neg) { ++n_neg_in; continue; }
      if (term != BM25F_TERM_UNKNOWN && !(b->leaf_weight[i] > 1e-30f)) all_pos = false;   // (an unknown term's leaf is dropped)
      if (!std::isfinite(b->leaf_weight[i])) PFAIL(BM25F_EINVAL, "query %u: leaf weight is not finite", qi);
    }
    bool dead = false;
    for (uint32_t g = 0; g < G; ++g)
      if (!gseen[g] || gsize[g] == 0) dead = true;   // an empty group: the AND matches nothing (W10)
    if (dead) { dummy_leaves(a, e); continue; }

    // smallest group first: it defines the candidate set, later groups only filter it
    uint32_t order[32], rank[32];
    for (uint32_t g = 0; g < G; ++g) order[g] = g;
    if (G > 1) std::stable_sort(order, order + G, [&](uint32_t x, uint32_t y) { return gsize[x] < gsize[y]; });
    for (uint32_t r = 0; r < G; ++r) rank[order[r]] = r;
    uint64_t P = 0;
    uint32_t nlq = 0;
    // the leaves of NOT clauses go first: the accumulating kernels visit leaves in this order and a
    // poisoned slot must be poisoned before a positive posting looks at it
    uint32_t n_neg = 0;
    for (uint32_t i = a; n_neg_in && i < e; ++i) {
      if (b->leaf_group[i] != BM25F_GROUP_NOT) continue;
      const uint32_t term = resolve_term(h, b->leaf_term[i]);
      if (term == BM25F_TERM_UNKNOWN) continue;
      const uint64_t off = h->term_offsets[term], df = h->term_offsets[term + 1] - off;
      if (df == 0) continue;
      LeafRec& lf = leaves[a + nlq];
      lf.off = off;
      lf.df = (uint32_t)df;
      lf.w = 1.0f;
      lf.norm_off = (uint32_t)h->term_field[term] * 256u;
      lf.group = NEG_GROUP;
      lf.qleaf0 = a;
      P += df;
      ++nlq;
      ++n_neg;
    }
    for (uint32_t r = 0; r < G; ++r) {
      for (uint32_t i = a; i < e; ++i) {
        if (b->leaf_group[i] != order[r]) continue;
        const uint32_t term = resolve_term(h, b->leaf_term[i]);
        if (term == BM25F_TERM_UNKNOWN) continue;
        const uint64_t off = h->term_offsets[term], df = h->term_offsets[term + 1] - off;
        if (df == 0) continue;
        LeafRec& lf = leaves[a + nlq];
        lf.off = off;
        lf.df = (uint32_t)df;
        lf.w = b->leaf_weight[i];
        lf.norm_off = (uint32_t)h->term_field[term] * 256u;
        lf.group = rank[b->leaf_group[i]];
        lf.qleaf0 = a;
        P += df;
        ++nlq;
      }
    }
    for (uint32_t i = 0; i < nlq; ++i) leaves[a + i].qnl = nlq;
    for (uint32_t i = a + nlq; i < e; ++i) { leaves[i] = LeafRec{}; leaves[i].qleaf0 = i; leaves[i].qnl = 1; }   // unused slots stay harmless
    qr.n_leaves = (uint16_t)nlq;
    qr.n_groups = (uint16_t)G;
    qr.flags = (G == 1 && all_pos && n_neg == 0) ? QF_SIMPLE_OR : 0u;
    if (!all_pos) L.any_nonpos = true;
    L.postings += P;

    // Route the query: stream kernel when it is eligible (top list fits one warp, few enough leaves
    // for register-resident rings, positive weights, no paging bound), else the CTA-per-item kernels.
    // (a paging bound is served by the warp kernels only in their final() instantiations, by the CTA kernels otherwise)
    const bool no_bound = qr.after_key == 0ull || final_mode;
    const bool stream_ok = (h->variant == 0 || h->variant >= 3) && k <= FAST_MAX_K && nlq <= 8 && all_pos && no_bound;
    // auto: a flat OR sweeps every sub-range anyway and runs best on independent warps (stream
    // kernel); an AND skips the slices in which a group is absent and runs best on warp teams
    // ... unless its smallest group is so much sparser than the rest that looking its documents up in
    // the other lists (Whoosh's IntersectionMatcher + skip_to) beats streaming every list
    const uint64_t g0 = gsize[order[0]];
    if (n_neg && !(k <= FAST_MAX_K && nlq <= 32 && G < NEG_GROUP && all_pos && no_bound))
      PFAIL(BM25F_EINVAL, "query %u: NOT clauses are served for k <= 256, at most 32 leaves and 30 groups, positive weights and no paging bound", qi);
    const bool isect_ok = k <= FAST_MAX_K && nlq <= 32 && all_pos && no_bound;
    if (final_mode && !isect_ok && !stream_ok)
      PFAIL(BM25F_EINVAL, "query %u: a final() weighting is served for k <= 256, at most 32 leaves and positive weights", qi);
    const uint64_t n_cand = (qr.flags & QF_SIMPLE_OR) ? P * (uint64_t)(nlq > 1 ? nlq - 1 : 1) : g0 * (uint64_t)(nlq - 1);   // lookups
    // A flat OR with few L.postings is also cheaper the candidate-driven way (every posting is a candidate
    // and is still read exactly once; sweeping every sub-range of the document space is what costs).
    const bool use_isect = isect_ok && ((final_mode && !stream_ok) || h->variant == 5 || (n_neg && !stream_ok) || (h->variant == 0 &&
        ((qr.flags & QF_SIMPLE_OR) ? n_cand < (uint64_t)h->is_or_limit
                                   : g0 * (uint64_t)(nlq - 1) * h->is_ratio < P)));
    const bool use_team = !use_isect && stream_ok && qr.after_key == 0ull && n_neg == 0 && !final_mode && k <= 32 && (h->variant == 4 || (h->variant == 0 && !(qr.flags & QF_SIMPLE_OR)));
    const int cls = use_isect ? 3 : stream_ok ? (use_team ? 1 : 0) : 2;
    if (cls == 2 && has_dyn)
      PFAIL(BM25F_EINVAL, "query %u uses a bm25f_put_lists list and needs the CTA kernels (k > 256, more than 32 leaves, a non-positive "
                          "weight or a paging bound): per-batch lists are served by the warp kernels only", qi);
    if (cls == 2 && h->raw_dropped)
      PFAIL(BM25F_EINVAL, "query %u needs the kernels that read the raw postings (k > 256, more than 32 leaves, a non-positive weight or a "
                          "paging bound) and the engine was created with compact_store", qi);
    uint32_t nsplit;
    if (use_isect) {
      nsplit = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, h->n_docs / 256), std::max<uint64_t>(1, (n_cand + is_split) / (2ull * is_split)));
      qr.n_parts = nsplit;
      for (uint32_t s = 0; s < nsplit; ++s) {
        ItemRec it;
        it.q = qi;
        it.tile_begin = (uint32_t)(h->n_docs * s / nsplit);          // document range [lo, hi)
        it.tile_end = (uint32_t)(h->n_docs * (s + 1) / nsplit);
        it.part = L.n_parts + s;
        L.items[cls].push_back(it);
        L.item_w[cls].push_back(n_cand / nsplit + 64);
      }
    } else if (use_team) {
      // warp teams: an item is a document range; its slices are handed out inside the CTA
      const uint64_t sw = h->tl_slot_bytes / ((qr.flags & QF_SIMPLE_OR) ? 4u : 8u);
      const uint64_t nsl = (h->n_docs + sw - 1) / sw;
      const uint64_t work = P + nsl * (16ull * nlq + 24ull);
      nsplit = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, nsl / 32), std::max<uint64_t>(1, (work + tl_split / 2) / tl_split));
      qr.n_parts = nsplit;
      for (uint32_t s = 0; s < nsplit; ++s) {
        ItemRec it;
        it.q = qi;
        it.tile_begin = (uint32_t)((nsl * s / nsplit) * sw);                    // document range [lo, hi), slice-aligned
        it.tile_end = (uint32_t)std::min<uint64_t>(h->n_docs, (nsl * (s + 1) / nsplit) * sw);
        it.part = L.n_parts + s;
        L.items[cls].push_back(it);
        L.item_w[cls].push_back(work / nsplit);
      }
    } else if (stream_ok) {
      // cost model in posting-equivalents: every (sub-range, leaf) visit costs a fixed amount
      const uint64_t sw = h->st_slot_bytes / ((qr.flags & QF_SIMPLE_OR) ? 4u : 8u);
      const uint64_t nsub = (h->n_docs + sw - 1) / sw;
      const uint64_t work = P + nsub * (16ull * nlq + 24ull);
      nsplit = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(1, h->n_docs / 1024), std::max<uint64_t>(1, (work + wsplit / 2) / wsplit));
      qr.n_parts = nsplit;
      for (uint32_t s = 0; s < nsplit; ++s) {
        ItemRec it;
        it.q = qi;
        it.tile_begin = (uint32_t)(h->n_docs * s / nsplit);          // document range [lo, hi)
        it.tile_end = (uint32_t)(h->n_docs * (s + 1) / nsplit);
        it.part = L.n_parts + s;
        L.items[cls].push_back(it);
        L.item_w[cls].push_back(work / nsplit);
      }
    } else {
      nsplit = (uint32_t)std::min<uint64_t>(T, std::max<uint64_t>(1, (P + h->split / 2) / h->split));
      qr.n_parts = nsplit;
      for (uint32_t s = 0; s < nsplit; ++s) {
        ItemRec it;
        it.q = qi;
        it.tile_begin = (uint32_t)((uint64_t)T * s / nsplit);
        it.tile_end = (uint32_t)((uint64_t)T * (s + 1) / nsplit);
        it.part = L.n_parts + s;
        L.items[cls].push_back(it);
        L.item_w[cls].push_back(P / nsplit + (uint64_t)(it.tile_end - it.tile_begin) * 64);
      }
    }
    L.cls_postings[cls] += P;
    L.n_parts += nsplit;
    }
  };
#undef PFAIL
  const bool trace = getenv("BM25F_TRACE") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto t_a = now();
  unsigned n_thr = 1;
  if (Q >= 2048) n_thr = std::min<unsigned>(plan_thread_budget(), Q / 1024);
  std::vector<PlanLocal> locals(n_thr);
  if (n_thr == 1) {
    plan_range(0, Q, locals[0]);
  } else {
    if (!h->pool) h->pool = new PlanPool(8);
    n_thr = std::min(n_thr, h->pool->size());
    locals.resize(n_thr);
    const std::function<void(unsigned)> job = [&](unsigned t) {
      plan_range((uint32_t)((uint64_t)Q * t / n_thr), (uint32_t)((uint64_t)Q * (t + 1) / n_thr), locals[t]);
    };
    h->pool->parallel(n_thr, job);
  }
  for (auto& L : locals)
    if (L.rc) return fail(L.rc, "%s", L.err);
  // stitch: partial-list indices and bitmap offsets become global
  std::vector<ItemRec> items[4];
  std::vector<uint64_t> item_w[4];
  uint64_t postings = 0, cls_postings[4] = {0, 0, 0, 0};
  uint32_t n_parts = 0;
  bool any_nonpos = false;
  for (unsigned t = 0; t < n_thr; ++t) {
    PlanLocal& L = locals[t];
    if (t > 0 && n_parts) {
      const uint32_t q0 = (uint32_t)((uint64_t)Q * t / n_thr), q1 = (uint32_t)((uint64_t)Q * (t + 1) / n_thr);
      for (uint32_t qi = q0; qi < q1; ++qi) queries[qi].part_begin += n_parts;
      for (int c = 0; c < 4; ++c)
        for (auto& it : L.items[c]) it.part += n_parts;
    }
    for (int c = 0; c < 4; ++c) {
      items[c].insert(items[c].end(), L.items[c].begin(), L.items[c].end());
      item_w[c].insert(item_w[c].end(), L.item_w[c].begin(), L.item_w[c].end());
      cls_postings[c] += L.cls_postings[c];
    }
    postings += L.postings;
    n_parts += L.n_parts;
    any_nonpos = any_nonpos || L.any_nonpos;
  }
  const uint32_t out_leaf = NL;            // leaf records sit at their input positions
  auto t_b = now();

  bm25f_plan* p = new (std::nothrow) bm25f_plan();
  if (!p) return fail(BM25F_ENOMEM, "host allocation failed");
  p->h = h;
  p->Q = Q;
  p->k = k;
  p->kp = 1;
  while (p->kp < k) p->kp <<= 1;
  p->simple_kernel = (h->variant == 2) || any_nonpos;
  p->cap = p->simple_kernel ? key_capacity(k, (int)h->NT) : pipe_key_capacity(k, (int)h->NT);
  p->n_leaves = out_leaf;
  p->n_items = (uint32_t)items[2].size();
  p->n_w4 = (uint32_t)items[0].size();
  p->n_w8 = (uint32_t)items[1].size();
  p->n_is = (uint32_t)items[3].size();
  p->n_parts = n_parts;
  p->T = T;
  p->postings = postings;
  for (int c = 0; c < 4; ++c) p->postings_cls[c] = cls_postings[c];
  p->smem_score = p->simple_kernel ? score_smem_bytes(S, p->cap) : pipe_smem_bytes(h, p->cap);
  p->owns_memory = !use_arena;
  p->arena = use_arena ? slot : -1;
  p->final_mode = final_mode;

#define RCP(x)                                    \
  do {                                            \
    int rc_ = (x);                                \
    if (rc_) { bm25f_plan_destroy(p); return rc_; } \
  } while (0)
#define CUP(x)                                                          \
  do {                                                                  \
    cudaError_t e_ = (x);                                               \
    if (e_ != cudaSuccess) {                                            \
      int rc_ = fail(BM25F_ECUDA, "%s: %s", #x, cudaGetErrorString(e_)); \
      bm25f_plan_destroy(p);                                            \
      return rc_;                                                       \
    }                                                                   \
  } while (0)
  const size_t n_bounds = p->n_items ? (size_t)out_leaf * (T + 1) : 0;   // only the CTA kernels use the boundary table
  const size_t n_it = (size_t)p->n_items + p->n_w4 + p->n_w8 + p->n_is;
  std::vector<ItemRec> own_items;
  ItemRec* h_items;
  if (use_arena) {
    // the sorted item records follow the leaf / query records in the pinned arena
    const size_t need = hl_bytes + hq_bytes + align_up(n_it * sizeof(ItemRec));
    if (need > A.h_cap) {
      unsigned char* bigger = nullptr;
      const size_t cap = align_up(need * 2, 1u << 20);
      cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&bigger), cap, cudaHostAllocDefault);
      if (e != cudaSuccess) { delete p; return fail(BM25F_ENOMEM, "cudaHostAlloc(%zu): %s", cap, cudaGetErrorString(e)); }
      memcpy(bigger, A.h, hl_bytes + hq_bytes);
      cudaFreeHost(A.h);
      A.h = bigger;
      A.h_cap = cap;
      leaves = reinterpret_cast<LeafRec*>(A.h);
      queries = reinterpret_cast<QueryRec*>(A.h + hl_bytes);
    }
    h_items = reinterpret_cast<ItemRec*>(A.h + hl_bytes + hq_bytes);
  } else {
    own_items.resize(n_it);
    h_items = own_items.data();
  }
  // layout of the item array: [CTA items][warp streams][warp teams][candidate-driven AND]
  order_items(items[2], item_w[2], h_items);
  order_items(items[0], item_w[0], h_items + p->n_items);
  order_items(items[1], item_w[1], h_items + p->n_items + p->n_w4);
  order_items(items[3], item_w[3], h_items + p->n_items + p->n_w4 + p->n_w8);
  if (use_arena) {
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += align_up(bytes); return o; };
    const size_t o_leaves = take((size_t)out_leaf * sizeof(LeafRec)), o_queries = take((size_t)Q * sizeof(QueryRec)),
                 o_items = take(n_it * sizeof(ItemRec)), o_bounds = take(n_bounds * 4),
                 o_part = take((size_t)n_parts * k * 8), o_keys = take((size_t)Q * k * 8), o_tot = take((size_t)(Q + 8) * 8),
                 o_sc = take((size_t)Q * k * 4), o_doc = take((size_t)Q * k * 4), o_cnt = take((size_t)Q * 4),
                 o_plo = take(final_mode ? (size_t)n_parts * k * 4 : 0), o_fin = take(final_mode ? (size_t)Q * k * 8 : 0);
    if (off > A.d_cap) {
      CUP(cudaStreamSynchronize(h->stream));
      CUP(cudaStreamSynchronize(h->copy_stream));
      cudaFree(A.d);
      A.d = nullptr;
      A.d_cap = 0;
      const size_t cap = align_up(off + off / 2, 1u << 20);
      cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&A.d), cap);
      if (e != cudaSuccess) { delete p; return fail(BM25F_ENOMEM, "cudaMalloc(%zu): %s", cap, cudaGetErrorString(e)); }
      A.d_cap = cap;
    }
    unsigned char* d = A.d;
    p->d_leaves = reinterpret_cast<LeafRec*>(d + o_leaves);
    p->d_queries = reinterpret_cast<QueryRec*>(d + o_queries);
    p->d_items = reinterpret_cast<ItemRec*>(d + o_items);
    p->d_bounds = reinterpret_cast<uint32_t*>(d + o_bounds);
    p->d_part_keys = reinterpret_cast<unsigned long long*>(d + o_part);
    p->d_keys = reinterpret_cast<unsigned long long*>(d + o_keys);
    p->d_totals = reinterpret_cast<unsigned long long*>(d + o_tot);
    p->d_scores = reinterpret_cast<float*>(d + o_sc);
    p->d_docids = reinterpret_cast<uint32_t*>(d + o_doc);
    p->d_counts = reinterpret_cast<uint32_t*>(d + o_cnt);
    if (final_mode) {
      p->d_part_lo = reinterpret_cast<unsigned int*>(d + o_plo);
      p->d_final = reinterpret_cast<double*>(d + o_fin);
    }
  } else {
    RCP(dev_alloc(&p->d_leaves, out_leaf));
    RCP(dev_alloc(&p->d_queries, Q));
    RCP(dev_alloc(&p->d_items, n_it));
    RCP(dev_alloc(&p->d_bounds, n_bounds));
    RCP(dev_alloc(&p->d_part_keys, (size_t)n_parts * k));
    // keys and totals in one allocation: one span for the sharded exchange (bm25f_plan_gather_span)
    RCP(dev_alloc(&p->d_keys, align_up((size_t)Q * k * 8) / 8 + (size_t)Q + 8));
    p->d_totals = p->d_keys + align_up((size_t)Q * k * 8) / 8;
    RCP(dev_alloc(&p->d_scores, (size_t)Q * k));
    RCP(dev_alloc(&p->d_docids, (size_t)Q * k));
    RCP(dev_alloc(&p->d_counts, Q));
    if (final_mode) {
      RCP(dev_alloc(&p->d_part_lo, (size_t)n_parts * k + 1));
      RCP(dev_alloc(&p->d_final, (size_t)Q * k + 1));
    }
  }
  p->d_items_w4 = p->d_items + p->n_items;
  p->d_items_w8 = p->d_items + p->n_items + p->n_w4;
  p->d_items_is = p->d_items + p->n_items + p->n_w4 + p->n_w8;
  auto t_c = now();
  // Arena plans upload on the copy stream (bm25f_execute waits for ev_ready): the records of the next batch
  // travel while the current one is still being scored.  Nothing else touches this arena: its previous
  // batch was fetched / collected before it was handed out again.
  cudaStream_t up = use_arena ? h->copy_stream : h->stream;
  if (out_leaf) CUP(cudaMemcpyAsync(p->d_leaves, leaves, (size_t)out_leaf * sizeof(LeafRec), cudaMemcpyHostToDevice, up));
  if (Q) CUP(cudaMemcpyAsync(p->d_queries, queries, (size_t)Q * sizeof(QueryRec), cudaMemcpyHostToDevice, up));
  if (n_it) CUP(cudaMemcpyAsync(p->d_items, h_items, n_it * sizeof(ItemRec), cudaMemcpyHostToDevice, up));
  if (use_arena) CUP(cudaEventRecord(A.ev_ready, up));
  // pageable sources must outlive the copy; a pinned arena is only rewritten two batches later
  if (!use_arena) CUP(cudaStreamSynchronize(h->stream));
  if (trace) {
    auto us = [](auto x, auto y) { return (double)std::chrono::duration_cast<std::chrono::nanoseconds>(y - x).count() / 1e3; };
    fprintf(stderr, "[bm25f prepare] plan %.0f us (%u threads), order+alloc %.0f us, enqueue copies %.0f us\n", us(t_a, t_b), n_thr, us(t_b, t_c), us(t_c, now()));
  }
  *out = p;
  return 0;
#undef RCP
#undef CUP
}

}  // namespace

extern "C" {

int bm25f_prepare(bm25f_handle* h, const bm25f_query_batch* b, int k, bm25f_plan** out) {
  return prepare_impl(h, b, k, out, false);
}

int bm25f_prepare_arena(bm25f_handle* h, const bm25f_query_batch* b, int k, bm25f_plan** out) {
  return prepare_impl(h, b, k, out, true);
}

int bm25f_execute(bm25f_handle* h, bm25f_plan* p) {
  if (!h || !p || p->h != h) return fail(BM25F_EINVAL, "plan does not belong to this handle");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  uint64_t launches = 0;
  if (h->ev_pending == bm25f_handle::EV_RING) {
    int rc = fold_events(h, 1);
    if (rc) return rc;
  }
  if (p->final_mode && !h->d_final_add) return fail(BM25F_EINVAL, "the plan was prepared with a final() step that has since been switched off");
  cudaEvent_t* ev = h->ev[h->ev_head];
  if (p->arena >= 0) CU(cudaStreamWaitEvent(st, h->arenas[p->arena].ev_ready, 0));
  CU(cudaEventRecord(ev[0], st));
  CU(cudaMemsetAsync(p->d_totals, 0, ((size_t)p->Q + 8) * 8, st));   // totals + the work counters
  const unsigned long long nb = p->n_items ? (unsigned long long)p->n_leaves * (p->T + 1) : 0ull;
  if (nb) {
    k_tile_bounds<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(p->d_leaves, p->n_leaves, p->T, h->S, h->d_docids, p->d_bounds);
    CU(cudaGetLastError());
    ++launches;
  }
  CU(cudaEventRecord(ev[1], st));
  if (p->n_items || p->n_w4 || p->n_w8 || p->n_is) {
    ScoreParams sp;
    sp.pairs = h->d_pairs;
    sp.leaves = p->d_leaves;
    sp.queries = p->d_queries;
    sp.items = p->d_items;
    sp.bounds = p->d_bounds;
    sp.part_keys = p->d_part_keys;
    sp.totals = p->d_totals;
    sp.S = h->S;
    sp.T = p->T;
    sp.n_docs = (uint32_t)h->n_docs;
    sp.doc_base = (uint32_t)h->doc_base;
    sp.k = p->k;
    sp.cap = p->cap;
    sp.prof = h->d_prof;
    // The stream kernel (one fat CTA per SM) and the candidate-driven kernel (no shared memory, few
    // registers) fit on an SM together and stall on different things: launch them side by side.
    // (a final() step with more than one key a lane: the FINAL instantiations need too many registers to share an
    // SM, the second kernel would trickle in behind the first one's CTAs - run them one after the other)
    const bool side = p->n_w4 && (p->n_is || p->n_w8) && !h->serial_streams && (!p->final_mode || p->k <= 32);
    cudaStream_t ax = side ? h->aux_stream : st;
    if (side) {
      CU(cudaEventRecord(h->ev_fork, st));
      CU(cudaStreamWaitEvent(ax, h->ev_fork, 0));
    }
    if (p->n_w4) {
      StreamParams stp;
      stp.pairs = h->d_pairs;
      stp.leaves = p->d_leaves;
      stp.queries = p->d_queries;
      stp.part_keys = p->d_part_keys;
      stp.totals = p->d_totals;
      stp.doc_base = (uint32_t)h->doc_base;
      stp.pf_dist = h->st_pf;
      stp.k = p->k;
      stp.items = p->d_items_w4;
      stp.n_items = p->n_w4;
      stp.n_items_dev = p->device_planned ? p->d_ctr + PL_CTR_ITEMS + 0 : nullptr;
      stp.items_off_dev = p->device_planned ? p->d_ctr + PL_CTR_OFF + 0 : nullptr;
      stp.slot_bytes = h->st_slot_bytes;
      stp.final_add = h->d_final_add;
      stp.final_blk = h->d_final_blk;
      stp.part_lo = p->d_part_lo;
      stp.queue = reinterpret_cast<unsigned int*>(p->d_totals + p->Q);
      const unsigned grid = p->device_planned ? (unsigned)h->n_sms : std::min<unsigned>((unsigned)h->n_sms, (p->n_w4 + h->st_warps - 1) / h->st_warps);
      CU(cudaEventRecord(ev[4], st));
      const size_t smem = stream_smem_bytes(h->st_warps, h->st_slot_bytes);
      if (p->final_mode) {
        if (p->k <= 32) k_score_stream<1, true><<<grid, h->st_warps * 32u, smem, st>>>(stp);
        else if (p->k <= 128) k_score_stream<4, true><<<grid, h->st_warps * 32u, smem, st>>>(stp);
        else k_score_stream<8, true><<<grid, h->st_warps * 32u, smem, st>>>(stp);
      } else if (p->k <= 32) k_score_stream<1, false><<<grid, h->st_warps * 32u, smem, st>>>(stp);
      else if (p->k <= 128) k_score_stream<4, false><<<grid, h->st_warps * 32u, smem, st>>>(stp);
      else k_score_stream<8, false><<<grid, h->st_warps * 32u, smem, st>>>(stp);
      CU(cudaEventRecord(ev[5], st));
      CU(cudaGetLastError());
      ++launches;
    }
    if (p->n_is) {
      IsectParams ip;
      ip.pairs = h->d_pairs;
      ip.leaves = p->d_leaves;
      ip.queries = p->d_queries;
      ip.items = p->d_items_is;
      ip.part_keys = p->d_part_keys;
      ip.totals = p->d_totals;
      ip.queue = reinterpret_cast<unsigned int*>(p->d_totals + p->Q + 2);
      ip.n_items = p->n_is;
      ip.n_items_dev = p->device_planned ? p->d_ctr + PL_CTR_ITEMS + 2 : nullptr;
      ip.items_off_dev = p->device_planned ? p->d_ctr + PL_CTR_OFF + 2 : nullptr;
      ip.doc_base = (uint32_t)h->doc_base;
      ip.k = p->k;
      ip.final_add = h->d_final_add;
      ip.part_lo = p->d_part_lo;
      if (h->is_ctas_per_sm == 0) {
        int nb_ = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_, k_score_isect<1, false>, IS_WARPS * 32, 0));
        h->is_ctas_per_sm = std::max(1, nb_);
      }
      const unsigned grid = p->device_planned ? (unsigned)(h->n_sms * h->is_ctas_per_sm)
                                              : std::min<unsigned>((unsigned)(h->n_sms * h->is_ctas_per_sm), (p->n_is + IS_WARPS - 1) / IS_WARPS);
      if (p->final_mode) {
        // final() of every match before the top-k: 96-bit keys, more registers, 2 CTAs per SM at least
        const unsigned gridf = std::min<unsigned>((unsigned)(h->n_sms * 2), (p->n_is + IS_WARPS - 1) / IS_WARPS);
        if (p->k <= 32) k_score_isect<1, true><<<gridf, IS_WARPS * 32, 0, ax>>>(ip);
        else if (p->k <= 128) k_score_isect<4, true><<<gridf, IS_WARPS * 32, 0, ax>>>(ip);
        else k_score_isect<8, true><<<gridf, IS_WARPS * 32, 0, ax>>>(ip);
      } else if (p->k <= 32) k_score_isect<1, false><<<grid, IS_WARPS * 32, 0, ax>>>(ip);
      else if (p->k <= 128) k_score_isect<4, false><<<grid, IS_WARPS * 32, 0, ax>>>(ip);
      else k_score_isect<8, false><<<std::min<unsigned>(grid, (unsigned)(h->n_sms * 2)), IS_WARPS * 32, 0, ax>>>(ip);
      CU(cudaGetLastError());
      ++launches;
    }
    if (p->n_w8) {
      TeamParams tp;
      tp.pairs = h->d_pairs;
      tp.leaves = p->d_leaves;
      tp.queries = p->d_queries;
      tp.items = p->d_items_w8;
      tp.part_keys = p->d_part_keys;
      tp.totals = p->d_totals;
      tp.queue = reinterpret_cast<unsigned int*>(p->d_totals + p->Q + 1);
      tp.n_items = p->n_w8;
      tp.n_items_dev = p->device_planned ? p->d_ctr + PL_CTR_ITEMS + 1 : nullptr;
      tp.items_off_dev = p->device_planned ? p->d_ctr + PL_CTR_OFF + 1 : nullptr;
      tp.slot_bytes = h->tl_slot_bytes;
      tp.doc_base = (uint32_t)h->doc_base;
      tp.prefetch = h->tl_prefetch;
      tp.k = p->k;
      if (h->tl_ctas_per_sm == 0) {
        int nb_ = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_, k_score_team, (int)h->tl_warps * 32, team_smem_bytes(h)));
        h->tl_ctas_per_sm = std::max(1, nb_);
      }
      const unsigned grid = p->device_planned ? (unsigned)(h->n_sms * h->tl_ctas_per_sm) : std::min<unsigned>((unsigned)(h->n_sms * h->tl_ctas_per_sm), p->n_w8);
      k_score_team<<<grid, h->tl_warps * 32u, team_smem_bytes(h), ax>>>(tp);
      CU(cudaGetLastError());
      ++launches;
    }
    if (side) {
      CU(cudaEventRecord(h->ev_join, ax));
      CU(cudaStreamWaitEvent(st, h->ev_join, 0));
    }
    if (!p->n_items) {
      // nothing for the CTA kernels
    } else if (!p->simple_kernel) {
      PipeParams pp;
      pp.sp = sp;
      pp.chunk = h->chunk;
      pp.stages = h->stages;
      pp.prune_at = (uint32_t)pipe_prune_at(p->k);
      k_score_pipe<<<p->n_items, h->NT + 32, p->smem_score, st>>>(pp);
    } else {
      k_score_topk<<<p->n_items, h->NT, p->smem_score, st>>>(sp);
    }
    if (p->n_items) {
      CU(cudaGetLastError());
      ++launches;
    }
  }
  if (!p->n_w4) { CU(cudaEventRecord(ev[4], st)); CU(cudaEventRecord(ev[5], st)); }
  CU(cudaEventRecord(ev[2], st));
  if (p->Q && p->final_mode) {
    if (p->k <= 128) k_merge_final<4><<<(p->Q + 7) / 8, 256, 0, st>>>(p->d_part_keys, p->d_part_lo, p->d_queries, p->Q, p->k, p->d_final, p->d_docids, p->d_counts);
    else k_merge_final<8><<<(p->Q + 7) / 8, 256, 0, st>>>(p->d_part_keys, p->d_part_lo, p->d_queries, p->Q, p->k, p->d_final, p->d_docids, p->d_counts);
    CU(cudaGetLastError());
    ++launches;
  } else if (p->Q) {
    if (p->k <= 32) k_merge_topk_warp<<<(p->Q + 7) / 8, 256, 0, st>>>(p->d_part_keys, p->d_queries, 0, 0, 0ull, p->Q, p->k, p->d_keys);
    else k_merge_topk<<<p->Q, 128, (size_t)2 * p->kp * 8, st>>>(p->d_part_keys, p->d_queries, 0, 0, 0ull, p->Q, p->k, p->kp, p->d_keys);
    CU(cudaGetLastError());
    k_decode_keys<<<p->Q, 64, 0, st>>>(p->d_keys, p->Q, p->k, p->d_scores, p->d_docids, p->d_counts);
    CU(cudaGetLastError());
    launches += 2;
  }
  CU(cudaEventRecord(ev[3], st));
  h->ev_head = (h->ev_head + 1) % bm25f_handle::EV_RING;
  ++h->ev_pending;
  if (p->submitted) {
    // results -> the arena's pinned landing zone: totals, scores, docids and counts are neighbours in the arena, so one
    // copy, on its own stream (the next batch's kernels start while it travels)
    bm25f_handle::Arena& A = h->arenas[p->arena];
    const unsigned char* base = reinterpret_cast<const unsigned char*>(p->d_totals);
    const size_t need = (size_t)(reinterpret_cast<const unsigned char*>(p->d_counts + p->Q) - base);
    if (need > A.h_out_cap) {
      if (A.h_out) cudaFreeHost(A.h_out);
      A.h_out = nullptr;
      A.h_out_cap = 0;
      const size_t cap = align_up(need + need / 2, 1u << 20);
      cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&A.h_out), cap, cudaHostAllocDefault);
      if (e != cudaSuccess) return fail(BM25F_ENOMEM, "cudaHostAlloc(%zu): %s", cap, cudaGetErrorString(e));
      A.h_out_cap = cap;
    }
    CU(cudaEventRecord(A.ev_scored, st));
    CU(cudaStreamWaitEvent(h->d2h_stream, A.ev_scored, 0));
    if (p->Q) CU(cudaMemcpyAsync(A.h_out, base, need, cudaMemcpyDeviceToHost, h->d2h_stream));
    CU(cudaEventRecord(A.ev_done, h->d2h_stream));
  }
  h->stats_from_ctr = p->device_planned;
  if (p->device_planned) {
    // the planner's counters follow the results; bm25f_get_stats reads them after a synchronize
    CU(cudaMemcpyAsync(h->h_ctr, p->d_ctr, PL_CTR_BYTES, cudaMemcpyDeviceToHost, st));
    launches += 3;                   // k_plan_queries, k_plan_scan, k_plan_items (bm25f_prepare_arena enqueued them)
  }
  h->stats.postings_touched = p->postings;
  h->stats.postings_stream = p->postings_cls[0];
  h->stats.postings_team = p->postings_cls[1];
  h->stats.postings_cta = p->postings_cls[2];
  h->stats.postings_lookup = p->postings_cls[3];
  h->stats.n_items = (uint64_t)p->n_items + p->n_w4 + p->n_w8 + p->n_is;
  h->stats.n_launches = launches;
  if (h->ctas_per_sm == 0) {
    int nb_ = 0;
    if (p->n_w8 && !p->n_w4) {
      nb_ = h->tl_ctas_per_sm;
    } else if (p->n_w4) {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_, k_score_stream<1, false>, (int)h->st_warps * 32, stream_smem_bytes(h->st_warps, h->st_slot_bytes));
    } else if (!p->simple_kernel) {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_, k_score_pipe, (int)h->NT + 32, p->smem_score);
    } else {
      cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb_, k_score_topk, (int)h->NT, p->smem_score);
    }
    h->ctas_per_sm = nb_;
    h->stats.ctas_per_sm = (uint32_t)nb_;
  }
  return 0;
}

int bm25f_set_stream(bm25f_handle* h, void* stream, int use_own) {
  if (!h) return fail(BM25F_EINVAL, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  // a NULL `stream` is a valid handle: the legacy default stream
  h->stream = use_own ? h->own_stream : static_cast<cudaStream_t>(stream);
  return 0;
}

int bm25f_synchronize(bm25f_handle* h) {
  if (!h) return fail(BM25F_EINVAL, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  CU(cudaStreamSynchronize(h->d2h_stream));
  return fold_events(h, h->ev_pending);
}

int bm25f_fetch(bm25f_handle* h, bm25f_plan* p, float* out_scores, uint32_t* out_docids, uint32_t* out_counts,
                uint64_t* out_totals) {
  if (!h || !p || p->h != h) return fail(BM25F_EINVAL, "plan does not belong to this handle");
  CU(cudaSetDevice(h->device));
  if (p->final_mode) return fail(BM25F_EINVAL, "the plan was prepared with a final() step: use bm25f_fetch_final");
  const size_t n = (size_t)p->Q * p->k;
  if (out_scores && n) CU(cudaMemcpyAsync(out_scores, p->d_scores, n * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out_docids && n) CU(cudaMemcpyAsync(out_docids, p->d_docids, n * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out_counts && p->Q) CU(cudaMemcpyAsync(out_counts, p->d_counts, (size_t)p->Q * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out_totals && p->Q) CU(cudaMemcpyAsync(out_totals, p->d_totals, (size_t)p->Q * 8, cudaMemcpyDeviceToHost, h->stream));
  return bm25f_synchronize(h);
}

int bm25f_fetch_final(bm25f_handle* h, bm25f_plan* p, double* out_final, uint32_t* out_docids, uint32_t* out_counts,
                      uint64_t* out_totals) {
  if (!h || !p || p->h != h) return fail(BM25F_EINVAL, "plan does not belong to this handle");
  if (!p->final_mode) return fail(BM25F_EINVAL, "the plan was prepared without a final() step: use bm25f_fetch");
  CU(cudaSetDevice(h->device));
  const size_t n = (size_t)p->Q * p->k;
  if (out_final && n) CU(cudaMemcpyAsync(out_final, p->d_final, n * 8, cudaMemcpyDeviceToHost, h->stream));
  if (out_docids && n) CU(cudaMemcpyAsync(out_docids, p->d_docids, n * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out_counts && p->Q) CU(cudaMemcpyAsync(out_counts, p->d_counts, (size_t)p->Q * 4, cudaMemcpyDeviceToHost, h->stream));
  if (out_totals && p->Q) CU(cudaMemcpyAsync(out_totals, p->d_totals, (size_t)p->Q * 8, cudaMemcpyDeviceToHost, h->stream));
  return bm25f_synchronize(h);
}

int bm25f_set_final_date(bm25f_handle* h, const double* date_add) {
  if (!h) return fail(BM25F_EINVAL, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));
  for (auto& A : h->arenas)
    if (A.submitted) return fail(BM25F_EINVAL, "collect the submitted batches before changing the weighting");
  if (!date_add) {
    cudaFree(h->d_final_add);
    cudaFree(h->d_final_blk);
    h->d_final_add = nullptr;
    h->d_final_blk = nullptr;
    return 0;
  }
  const size_t nblk = (size_t)(h->n_docs / 32 + 2);
  if (!h->d_final_blk) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&h->d_final_blk), nblk * sizeof(double));
    if (e != cudaSuccess) {
      h->d_final_blk = nullptr;
      return fail(BM25F_ENOMEM, "cudaMalloc(%zu): %s", nblk * sizeof(double), cudaGetErrorString(e));
    }
  }
  {
    std::vector<double> blk(nblk, -INFINITY);
    for (uint64_t d = 0; d < h->n_docs; ++d)
      if (date_add[d] > blk[d >> 5]) blk[d >> 5] = date_add[d];      // NaN (no date) never compares greater
    CU(cudaMemcpy(h->d_final_blk, blk.data(), nblk * sizeof(double), cudaMemcpyHostToDevice));
  }
  if (!h->d_final_add) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&h->d_final_add), std::max<uint64_t>(1, h->n_docs) * sizeof(double));
    if (e != cudaSuccess) {
      h->d_final_add = nullptr;
      return fail(BM25F_ENOMEM, "cudaMalloc(%llu): %s", (unsigned long long)(h->n_docs * sizeof(double)), cudaGetErrorString(e));
    }
  }
  if (h->n_docs) CU(cudaMemcpy(h->d_final_add, date_add, h->n_docs * sizeof(double), cudaMemcpyHostToDevice));
  return 0;
}

int bm25f_plan_device_results(bm25f_plan* p, uint64_t** d_keys, uint64_t** d_totals) {
  if (!p) return fail(BM25F_EINVAL, "null plan");
  if (p->final_mode) return fail(BM25F_EINVAL, "plans with a final() step have no 64-bit key lists");
  if (d_keys) *d_keys = reinterpret_cast<uint64_t*>(p->d_keys);
  if (d_totals) *d_totals = reinterpret_cast<uint64_t*>(p->d_totals);
  return 0;
}

int bm25f_search_batch(bm25f_handle* h, const bm25f_query_batch* b, int k, float* out_scores, uint32_t* out_docids,
                       uint32_t* out_counts, uint64_t* out_totals) {
  if (h && h->d_final_add) return fail(BM25F_EINVAL, "a final() weighting is set: use bm25f_prepare_arena / bm25f_execute / bm25f_fetch_final");
  bm25f_plan* p = nullptr;
  int rc = prepare_impl(h, b, k, &p, true);
  if (rc) return rc;
  rc = bm25f_execute(h, p);
  if (!rc) rc = bm25f_fetch(h, p, out_scores, out_docids, out_counts, out_totals);
  bm25f_plan_destroy(p);
  return rc;
}

int bm25f_submit(bm25f_handle* h, const bm25f_query_batch* b, int k, bm25f_plan** out) {
  if (!out) return fail(BM25F_EINVAL, "null argument");
  if (h && h->d_final_add) return fail(BM25F_EINVAL, "a final() weighting is set: use bm25f_prepare_arena / bm25f_execute / bm25f_fetch_final");
  bm25f_plan* p = nullptr;
  int rc = prepare_impl(h, b, k, &p, true);
  if (rc) return rc;
  p->submitted = true;
  rc = bm25f_execute(h, p);
  if (rc) { bm25f_plan_destroy(p); return rc; }
  h->arenas[p->arena].submitted = p;
  *out = p;
  return 0;
}

int bm25f_collect(bm25f_handle* h, bm25f_plan* p, float* out_scores, uint32_t* out_docids, uint32_t* out_counts,
                  uint64_t* out_totals) {
  if (!h || !p || p->h != h) return fail(BM25F_EINVAL, "plan does not belong to this handle");
  if (!p->submitted || p->arena < 0 || h->arenas[p->arena].submitted != p) return fail(BM25F_EINVAL, "not a submitted plan");
  CU(cudaSetDevice(h->device));
  bm25f_handle::Arena& A = h->arenas[p->arena];
  if (h->arenas[p->arena ^ 1].submitted && h->arena_next != p->arena)      // both in flight: the older one sits in arena_next
    return fail(BM25F_EINVAL, "collect submitted batches in the order they were submitted");
  cudaError_t e = cudaEventSynchronize(A.ev_done);
  A.submitted = nullptr;
  if (e != cudaSuccess) {
    bm25f_plan_destroy(p);
    return fail(BM25F_ECUDA, "cudaEventSynchronize: %s", cudaGetErrorString(e));
  }
  const size_t n = (size_t)p->Q * p->k;
  const unsigned char* base = reinterpret_cast<const unsigned char*>(p->d_totals);      // h_out mirrors [d_totals, d_counts + Q)
  const size_t o_sc = (size_t)(reinterpret_cast<const unsigned char*>(p->d_scores) - base),
               o_doc = (size_t)(reinterpret_cast<const unsigned char*>(p->d_docids) - base),
               o_cnt = (size_t)(reinterpret_cast<const unsigned char*>(p->d_counts) - base);
  if (out_scores && n) memcpy(out_scores, A.h_out + o_sc, n * 4);
  if (out_docids && n) memcpy(out_docids, A.h_out + o_doc, n * 4);
  if (out_counts && p->Q) memcpy(out_counts, A.h_out + o_cnt, (size_t)p->Q * 4);
  if (out_totals && p->Q) memcpy(out_totals, A.h_out, (size_t)p->Q * 8);
  bm25f_plan_destroy(p);
  return fold_events(h, 1);          // this batch's timings (batches finish in submission order)
}

int bm25f_merge_keys(bm25f_handle* h, const uint64_t* d_keys, int n_lists, uint32_t n_queries, int k,
                     uint64_t* d_out_keys, void* stream) {
  if (!h || !d_keys || !d_out_keys) return fail(BM25F_EINVAL, "null argument");
  if (k < 1 || k > BM25F_MAX_K || n_lists < 1) return fail(BM25F_EINVAL, "bad k or n_lists");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  int kp = 1;
  while (kp < k) kp <<= 1;
  if (n_queries) {
    if (k <= 32)
      k_merge_topk_warp<<<(n_queries + 7) / 8, 256, 0, st>>>(reinterpret_cast<const unsigned long long*>(d_keys), nullptr, 1, n_lists,
                                                           (unsigned long long)n_queries * k, n_queries, k,
                                                           reinterpret_cast<unsigned long long*>(d_out_keys));
    else
      k_merge_topk<<<n_queries, 128, (size_t)2 * kp * 8, st>>>(reinterpret_cast<const unsigned long long*>(d_keys), nullptr, 1, n_lists,
                                                               (unsigned long long)n_queries * k, n_queries, k, kp,
                                                               reinterpret_cast<unsigned long long*>(d_out_keys));
    CU(cudaGetLastError());
  }
  return 0;
}

int bm25f_plan_gather_span(bm25f_plan* p, uint64_t** d_base, uint64_t* span_words, uint64_t* totals_offset_words) {
  if (!p || !d_base || !span_words || !totals_offset_words) return fail(BM25F_EINVAL, "null argument");
  if (p->final_mode) return fail(BM25F_EINVAL, "plans with a final() step have no 64-bit key lists");
  *d_base = reinterpret_cast<uint64_t*>(p->d_keys);
  *totals_offset_words = (uint64_t)(p->d_totals - p->d_keys);
  *span_words = *totals_offset_words + p->Q;
  return 0;
}

int bm25f_merge_gathered(bm25f_handle* h, const uint64_t* d_gathered, int n_lists, uint64_t span_words, uint64_t totals_offset_words,
                         uint32_t n_queries, int k, uint64_t* d_keys, float* d_scores, uint32_t* d_docids, uint32_t* d_counts,
                         uint64_t* d_totals, void* stream) {
  if (!h || !d_gathered || !d_keys || !d_scores || !d_docids || !d_counts || !d_totals) return fail(BM25F_EINVAL, "null argument");
  if (k < 1 || k > BM25F_MAX_K || n_lists < 1 || span_words < (uint64_t)n_queries * k) return fail(BM25F_EINVAL, "bad k, n_lists or span");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  if (!n_queries) return 0;
  int kp = 1;
  while (kp < k) kp <<= 1;
  const unsigned long long* g = reinterpret_cast<const unsigned long long*>(d_gathered);
  unsigned long long* out = reinterpret_cast<unsigned long long*>(d_keys);
  if (k <= 32) k_merge_topk_warp<<<(n_queries + 7) / 8, 256, 0, st>>>(g, nullptr, 1, n_lists, (unsigned long long)span_words, n_queries, k, out);
  else k_merge_topk<<<n_queries, 128, (size_t)2 * kp * 8, st>>>(g, nullptr, 1, n_lists, (unsigned long long)span_words, n_queries, k, kp, out);
  CU(cudaGetLastError());
  k_decode_keys_sum<<<n_queries, 64, 0, st>>>(out, g, n_lists, (unsigned long long)span_words, (unsigned long long)totals_offset_words,
                                              n_queries, k, d_scores, d_docids, d_counts, reinterpret_cast<unsigned long long*>(d_totals));
  CU(cudaGetLastError());
  return 0;
}

int bm25f_plan_device_final(bm25f_plan* p, double** d_final, uint32_t** d_docids, uint64_t** d_totals) {
  if (!p) return fail(BM25F_EINVAL, "null plan");
  if (!p->final_mode) return fail(BM25F_EINVAL, "the plan was prepared without a final() step");
  if (d_final) *d_final = p->d_final;
  if (d_docids) *d_docids = p->d_docids;
  if (d_totals) *d_totals = reinterpret_cast<uint64_t*>(p->d_totals);
  return 0;
}

int bm25f_merge_final_lists(bm25f_handle* h, const double* d_vals, const uint32_t* d_docids, int n_lists, uint32_t n_queries,
                            int k, double* d_out_final, uint32_t* d_out_docids, uint32_t* d_out_counts, void* stream) {
  if (!h || !d_vals || !d_docids || !d_out_final || !d_out_docids || !d_out_counts) return fail(BM25F_EINVAL, "null argument");
  if (k < 1 || k > FAST_MAX_K || n_lists < 1) return fail(BM25F_EINVAL, "bad k (1..256) or n_lists");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  if (n_queries) {
    if (k <= 128) k_merge_final_lists<4><<<(n_queries + 7) / 8, 256, 0, st>>>(d_vals, d_docids, n_lists, n_queries, k, d_out_final, d_out_docids, d_out_counts);
    else k_merge_final_lists<8><<<(n_queries + 7) / 8, 256, 0, st>>>(d_vals, d_docids, n_lists, n_queries, k, d_out_final, d_out_docids, d_out_counts);
    CU(cudaGetLastError());
  }
  return 0;
}

int bm25f_decode_keys(bm25f_handle* h, const uint64_t* d_keys, uint32_t n_queries, int k, float* d_scores,
                      uint32_t* d_docids, uint32_t* d_counts, void* stream) {
  if (!h || !d_keys) return fail(BM25F_EINVAL, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : h->stream;
  if (n_queries) {
    k_decode_keys<<<n_queries, 64, 0, st>>>(reinterpret_cast<const unsigned long long*>(d_keys), n_queries, k, d_scores, d_docids, d_counts);
    CU(cudaGetLastError());
  }
  return 0;
}

int bm25f_put_lists(bm25f_handle* h, uint32_t n_lists, const uint64_t* offsets, const uint32_t* docids, uint32_t* first_term) {
  if (!h || !first_term || (n_lists && (!offsets || (offsets[n_lists] && !docids)))) return fail(BM25F_EINVAL, "null argument");
  if (n_lists > BM25F_MAX_FILTER_LISTS) return fail(BM25F_EINVAL, "at most %d lists a batch", BM25F_MAX_FILTER_LISTS);
  if (n_lists && offsets[0] != 0) return fail(BM25F_EINVAL, "offsets must start at 0");
  const uint64_t total = n_lists ? offsets[n_lists] : 0;
  if (total > h->dyn_cap) return fail(BM25F_EINVAL, "%llu postings in the lists, room for %llu (option filter_postings)", (unsigned long long)total, (unsigned long long)h->dyn_cap);
  for (uint32_t l = 0; l < n_lists; ++l) {
    if (offsets[l + 1] < offsets[l] || offsets[l + 1] > total) return fail(BM25F_EINVAL, "offsets not monotonic at list %u", l);
    for (uint64_t i = offsets[l]; i < offsets[l + 1]; ++i)
      if (docids[i] >= h->n_docs || (i > offsets[l] && docids[i] <= docids[i - 1]))
        return fail(BM25F_EINVAL, "list %u: docids must be < n_docs_all and strictly ascending", l);
  }
  for (auto& A : h->arenas)
    if (A.submitted) return fail(BM25F_EINVAL, "a submitted batch is in flight: bm25f_collect it before replacing the lists");
  CU(cudaSetDevice(h->device));
  CU(cudaStreamSynchronize(h->stream));            // nothing may still be reading the previous lists
  CU(cudaStreamSynchronize(h->copy_stream));
  // {docid, impact 1.0}, then a run of end markers: rows and prefetches may read past the last posting of the last list
  const size_t pad = 1024;
  std::vector<uint2> pairs(total + pad);
  const uint32_t one = 0x3F800000u;
  for (uint64_t i = 0; i < total; ++i) pairs[i] = make_uint2(docids[i], one);
  for (size_t i = 0; i < pad; ++i) pairs[total + i] = make_uint2(0xFFFFFFFFu, 0xFFFFFFFFu);
  CU(cudaMemcpyAsync(h->d_pairs + h->dyn_base, pairs.data(), pairs.size() * sizeof(uint2), cudaMemcpyHostToDevice, h->stream));
  // term table: [0, n_terms) the index, n_terms the padding between the regions, then the lists (pseudo-field n_fields)
  h->term_offsets.resize(h->n_terms + 1);
  h->term_field.resize(h->n_terms);
  h->term_offsets.push_back(h->dyn_base);
  h->term_field.push_back((uint8_t)h->n_fields);
  for (uint32_t l = 0; l < n_lists; ++l) {
    h->term_offsets.push_back(h->dyn_base + offsets[l + 1]);
    h->term_field.push_back((uint8_t)h->n_fields);
  }
  h->dyn_terms = n_lists;
  CU(cudaMemcpyAsync(h->d_term_offsets + h->n_terms, h->term_offsets.data() + h->n_terms, ((size_t)n_lists + 2) * 8, cudaMemcpyHostToDevice, h->stream));
  CU(cudaMemcpyAsync(h->d_term_field + h->n_terms, h->term_field.data() + h->n_terms, (size_t)n_lists + 1, cudaMemcpyHostToDevice, h->stream));
  CU(cudaStreamSynchronize(h->stream));            // (the sources are locals)
  *first_term = (uint32_t)h->n_terms + 1u;
  return 0;
}

int bm25f_get_stats(bm25f_handle* h, bm25f_stats* out) {
  if (!h || !out) return fail(BM25F_EINVAL, "null argument");
  if (h->stats_from_ctr) {
    CU(cudaSetDevice(h->device));
    CU(cudaStreamSynchronize(h->stream));
    const unsigned int* c = h->h_ctr;
    unsigned long long post[PL_POST_WORDS];
    memcpy(post, c + PL_CTR_WORDS, sizeof post);
    h->stats.postings_touched = post[0];
    h->stats.postings_stream = post[1];
    h->stats.postings_team = post[2];
    h->stats.postings_cta = 0;
    h->stats.postings_lookup = post[3];
    h->stats.n_items = (uint64_t)c[PL_CTR_ITEMS] + c[PL_CTR_ITEMS + 1] + c[PL_CTR_ITEMS + 2];
  }
  *out = h->stats;
  return 0;
}

int bm25f_reset_stats(bm25f_handle* h) {
  if (!h) return fail(BM25F_EINVAL, "null handle");
#ifdef BM25F_PROFILE
  {
    unsigned long long v[16];
    cudaMemcpy(v, h->d_prof, sizeof v, cudaMemcpyDeviceToHost);
    static const char* names[16] = {"c.wait_full", "c.accumulate", "c.leaf_barrier", "c.tile_epilogue", "c.prune",
                                    "c.item_epilogue", "c6", "c7", "p.bound_rows", "p.schedule", "p.wait_empty",
                                    "p.issue", "p.tail", "p13", "p14", "p15"};
    fprintf(stderr, "[bm25f profile] cycles summed over CTAs (consumer thread 0 / producer lane 0):\n");
    for (int i = 0; i < 16; ++i)
      if (v[i]) fprintf(stderr, "  %-16s %14llu\n", names[i], v[i]);
    cudaMemset(h->d_prof, 0, sizeof v);
  }
#endif
  h->stats.ms_bounds = h->stats.ms_score = h->stats.ms_merge = h->stats.ms_total = h->stats.ms_stream = 0.0f;
  h->stats.n_executes = 0;
  return 0;
}

}  // extern "C"
