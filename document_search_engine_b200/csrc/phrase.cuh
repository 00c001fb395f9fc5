// Positional filter of phrase queries (bm25f_phrase_lists; Whoosh query.Phrase, reference search-form.html:20-40).
//
// A document matches a phrase (w_0 .. w_{n-1}, slop) iff kept_{n-1} is not empty, where kept_0 is the set of
// positions of w_0 in the field and kept_j the positions p of w_j with some e in kept_{j-1}, 1 <= p - e <= slop
// (FlatIndex.phrase_docs).  The candidates are the live postings of the phrase's rarest word, read from the
// {docid, impact} pairs, so deleted documents never become candidates.
//
// One warp per (phrase, candidate) walks the document's tokens (the field's document-major word order,
// bm25f_put_positions) 32 at a time.  Lane j keeps word j and the last position of kept_j seen in earlier chunks
// (its carry).  For a chunk and each word j in order, kept_j is a ballot: the lane's token is w_j and its position is
// at most `slop` past the nearest kept_{j-1} position before it - the highest lower lane of kept_{j-1}'s ballot
// (an exclusive max-scan), else the carry of word j - 1.  Exact for any slop, with no window limit.
//
// Three passes: k_phrase_mark sets one flag bit per candidate (candidate slots are padded to 32 per phrase, so a
// flag word belongs to one phrase) and counts the matches per phrase and per chunk of flag words; k_phrase_scan
// turns the chunk counts into offsets; k_phrase_compact writes the flagged candidates, in candidate order, as
// {docid, 1.0f} pairs.  The phrases' lists are concatenated in phrase order, so the output position of a match is its
// rank among all flagged candidates: the lists come out ascending and identical from run to run.

constexpr int PH_MAX_WORDS = 32;          // one word per lane
constexpr uint32_t PH_CHUNK_WORDS = 1024; // flag words per compaction CTA (one per thread)

struct PhraseRec {                        // 168 B
  const unsigned long long* offs;         // the field's word order: document d's tokens are toks[offs[d] .. offs[d + 1])
  const uint32_t* toks;
  unsigned long long cand;                // first pair of the candidate list
  uint32_t n_cand;
  uint32_t word0;                         // first flag word of the phrase
  uint32_t n_words;
  uint32_t slop;
  uint32_t words[PH_MAX_WORDS];
};

// the record whose flag words contain word w (records are ordered by word0, every one has at least one word)
__device__ __forceinline__ uint32_t phrase_of_word(const PhraseRec* __restrict__ recs, uint32_t n_recs, uint32_t w) {
  uint32_t lo = 0, hi = n_recs - 1;
  while (lo < hi) {
    const uint32_t mid = (lo + hi + 1) >> 1;
    if (recs[mid].word0 <= w) lo = mid; else hi = mid - 1;
  }
  return lo;
}

// Does the phrase occur in toks[0 .. len)?  Called by a whole warp; lane j holds word j (nw <= 32).
__device__ bool phrase_in_doc(const uint32_t* __restrict__ toks, unsigned long long len, uint32_t my_word, uint32_t nw,
                              uint32_t slop, int lane) {
  const unsigned FULL = 0xFFFFFFFFu;
  const unsigned below = (1u << lane) - 1u;            // lanes before this one: the scan is exclusive
  const uint32_t w0 = __shfl_sync(FULL, my_word, 0);
  long long carry = -1;                                // lane j: last kept_j position of the earlier chunks (-1: none)
  for (unsigned long long c0 = 0; c0 < len; c0 += 32) {
    const unsigned long long p = c0 + lane;
    const bool in = p < len;
    const uint32_t tok = in ? __ldg(toks + p) : 0u;
    unsigned kept = __ballot_sync(FULL, in && tok == w0);
    for (uint32_t j = 1; j < nw; ++j) {
      const long long cprev = __shfl_sync(FULL, carry, j - 1);
      unsigned next = 0u;
      // word j can be kept here only after a kept word j - 1 in this chunk or one close enough before it (a later word
      // may still follow the carry of word j)
      if (kept != 0u || (cprev >= 0 && (long long)c0 - cprev <= (long long)slop)) {
        const unsigned lower = kept & below;
        const long long prev = lower ? (long long)(c0 + 31 - __clz(lower)) : cprev;
        const uint32_t wj = __shfl_sync(FULL, my_word, j);
        next = __ballot_sync(FULL, in && tok == wj && prev >= 0 && (long long)p - prev <= (long long)slop);
      }
      if (kept && lane == (int)(j - 1)) carry = (long long)(c0 + 31 - __clz(kept));
      kept = next;
    }
    if (kept) return true;                             // kept_{n-1} of this chunk
  }
  return false;
}

// One CTA per flag word: warp w tests candidates w, w + 8, w + 16, w + 24 of the word's 32.
__global__ void __launch_bounds__(256) k_phrase_mark(const PhraseRec* __restrict__ recs, uint32_t n_recs, const uint2* __restrict__ pairs,
                                                     uint32_t* __restrict__ flags, unsigned int* __restrict__ counts,
                                                     unsigned int* __restrict__ chunk_sum) {
  __shared__ uint32_t s_bits;
  __shared__ uint32_t s_rec;
  const uint32_t w = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) { s_rec = phrase_of_word(recs, n_recs, w); s_bits = 0u; }
  __syncthreads();
  const PhraseRec* R = recs + s_rec;
  const uint32_t nw = R->n_words;
  const uint32_t my_word = lane < (int)nw ? R->words[lane] : 0xFFFFFFFFu;
  const uint32_t slop = R->slop;
  for (uint32_t b = warp; b < 32; b += 8) {
    const unsigned long long c = (unsigned long long)(w - R->word0) * 32ull + b;
    if (c >= R->n_cand) break;                          // the phrase's padding slots
    const uint32_t d = pairs[R->cand + c].x;
    const unsigned long long a = R->offs[d], e = R->offs[d + 1];
    if (phrase_in_doc(R->toks + a, e - a, my_word, nw, slop, lane) && lane == 0) atomicOr(&s_bits, 1u << b);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    flags[w] = s_bits;
    const unsigned n = __popc(s_bits);
    if (n) {
      atomicAdd(counts + s_rec, n);
      atomicAdd(chunk_sum + w / PH_CHUNK_WORDS, n);
    }
  }
}

// In place: chunk_sum[c] <- matches in the chunks before c.  One CTA of 1024 threads.
__global__ void __launch_bounds__(1024) k_phrase_scan(unsigned int* __restrict__ chunk_sum, uint32_t n_chunks) {
  __shared__ unsigned int s_warp[32];
  __shared__ unsigned int s_carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_carry = 0u;
  __syncthreads();
  for (uint32_t base = 0; base < n_chunks; base += 1024) {
    const uint32_t i = base + threadIdx.x;
    const unsigned v = i < n_chunks ? chunk_sum[i] : 0u;
    unsigned x = v;
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    if (warp == 0) {
      unsigned s = s_warp[lane];
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xFFFFFFFFu, s, o);
        if (lane >= o) s += y;
      }
      s_warp[lane] = s;                                 // inclusive sums of the warps
    }
    __syncthreads();
    const unsigned carry = s_carry;
    if (i < n_chunks) chunk_sum[i] = carry + (warp ? s_warp[warp - 1] : 0u) + x - v;
    __syncthreads();
    if (threadIdx.x == 0) s_carry = carry + s_warp[31];
    __syncthreads();
  }
}

// One CTA per chunk of 1024 flag words, one word a thread: out[rank] = {docid, 1.0f} for every flagged candidate.
__global__ void __launch_bounds__(1024) k_phrase_compact(const PhraseRec* __restrict__ recs, uint32_t n_recs, const uint2* __restrict__ pairs,
                                                         const uint32_t* __restrict__ flags, uint32_t n_flag_words,
                                                         const unsigned int* __restrict__ chunk_base, uint2* __restrict__ out) {
  __shared__ unsigned int s_warp[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t w = blockIdx.x * PH_CHUNK_WORDS + threadIdx.x;
  const uint32_t f = w < n_flag_words ? flags[w] : 0u;
  const unsigned n = __popc(f);
  unsigned x = n;
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    unsigned s = s_warp[lane];
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned y = __shfl_up_sync(0xFFFFFFFFu, s, o);
      if (lane >= o) s += y;
    }
    s_warp[lane] = s;
  }
  __syncthreads();
  if (!f) return;
  unsigned long long pos = (unsigned long long)chunk_base[blockIdx.x] + (warp ? s_warp[warp - 1] : 0u) + x - n;
  const PhraseRec* R = recs + phrase_of_word(recs, n_recs, w);
  const unsigned long long c0 = R->cand + (unsigned long long)(w - R->word0) * 32ull;
  for (uint32_t bits = f; bits; bits &= bits - 1u) {
    const int b = __ffs(bits) - 1;
    out[pos++] = make_uint2(pairs[c0 + b].x, 0x3F800000u);
  }
}
