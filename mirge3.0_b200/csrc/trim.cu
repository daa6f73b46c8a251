// trim.cu -- per-read digest kernel: the body of the reference worker ``cutadapt(n)``
// (mirge/libs/digest.py:320-375) for one read per thread:
//   NextSeq trim -> quality trim -> adapter removal -> N-end trim -> unconditional cuts
//   (modifier order of stipulate(), digest.py:87-99), key emission + length filter
//   (digest.py:332-373, HEAD per-stage counting or release post-pipeline counting), and 2-bit
//   packing of every emitted key for the collapse table.
// cutadapt semantics (3P, restated in oracle/pyoracle.py): qualtrim.pyx nextseq_trim_index /
// quality_trim_index; _align.pyx Aligner.locate with (cost, origin, matches) cells and the
// "most matches, then lowest cost, then first found" objective; NEndTrimmer; UnconditionalCutter.
//
// Data movement: a CTA owns TRIM_THREADS consecutive records, whose bytes are one contiguous span
// of the FASTQ stream; the span is staged in shared memory with coalesced 128-bit streaming loads
// and every thread then works on its own record out of shared memory.  All arithmetic is integer.
//
// Kernels (see "split pipeline" below): with 3' adapters of <= 32 nt the work is cut at the adapter modifier into
// stage 1 (trim_kernel<32,true,1,true>: everything up to the adapter + exact adapter search), stage 2
// (trim_dp_kernel<true>: bit-vector DP of the listed reads) and stage 3 (trim_dp_kernel<false>: the searches that
// need cost columns); trim_kernel<32,true,2,false> runs the whole pipeline per read for the leftovers, and
// trim_kernel<32,true,1,false> + that leftover pass is the unsplit bit-parallel path (qiagen UMIs);
// trim_kernel<32|64,false,0,false> is the generic full-DP kernel (5' adapters, --no-indels, long adapters).
#include "common.cuh"
// DevParams / c_p, fill_dev_params, locate, locate_fast, the quality scans, best_match, apply_mod
#include "adapter_search.cuh"

extern "C" int mirge_trim_slots(const mirge_ctx *ctx) {
  if (!ctx || !ctx->params_set) return MIRGE_ERR_ARG;
  return trim_slots_of(&ctx->params);
}

extern "C" int mirge_set_trim_params(mirge_ctx *ctx, const mirge_trim_params *p) {
  if (!ctx || !p) return MIRGE_ERR_ARG;
  DevParams d;
  int maxm = 0, fast_ok = 1;
  const int rc = fill_dev_params(p, d, maxm, fast_ok, ctx->err, sizeof(ctx->err));
  if (rc != MIRGE_OK) return rc;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemcpyToSymbol(c_p, &d, sizeof(d)));
  ctx->params = *p;
  ctx->params_set = 1;
  ctx->max_adapter_len = maxm;
  ctx->fast_ok = fast_ok;
  // split pipeline: not with qiagen UMIs (their key needs the read bytes after the pipeline) and only when no
  // quality modifier follows the first adapter modifier (stipulate() never builds such a pipeline)
  int split_ok = fast_ok && p->umi_mode != MIRGE_UMI_QIAGEN, seen_ad = 0;
  for (int i = 0; i < p->n_mods; ++i) {
    if (p->mod_kind[i] == MIRGE_MOD_ADAPTER) seen_ad = 1;
    else if (seen_ad && (p->mod_kind[i] == MIRGE_MOD_NEXTSEQ || p->mod_kind[i] == MIRGE_MOD_QUALITY)) split_ok = 0;
  }
  ctx->split_ok = split_ok && seen_ad;
  return MIRGE_OK;
}

// the modifiers that need no adapter search (everything stage 1 of the split pipeline runs before the adapter)
__device__ __forceinline__ void apply_plain_mod(int mi, const uint8_t *seq, const uint8_t *qual, int &start, int &stop) {
  const int len = stop - start;
  const int kind = c_p.kind[mi];
  if (kind == MIRGE_MOD_NEXTSEQ) {
    stop = start + nextseq_trim_index(seq + start, qual + start, len, c_p.a[mi], c_p.b[mi]);
  } else if (kind == MIRGE_MOD_QUALITY) {
    int s, e;
    quality_trim_index(qual + start, len, c_p.a[mi], c_p.b[mi], c_p.c[mi], s, e);
    stop = start + e;
    start = start + s;
  } else if (kind == MIRGE_MOD_NEND) {
    while (start < stop && seq[start] == 'N') ++start;
    while (stop > start && seq[stop - 1] == 'N') --stop;
  } else if (kind == MIRGE_MOD_CUT) {
    const int c = c_p.a[mi];
    if (c > 0) start += min(c, len);
    else stop = start + max(len + c, 0);
  }
}

__device__ __forceinline__ int find_sub(const uint8_t *s, int n, const uint8_t *t, int tl, int from) {
  for (int p = from; p + tl <= n; ++p) {
    int j = 0;
    while (j < tl && s[p + j] == t[j]) ++j;
    if (j == tl) return p;
  }
  return -1;
}

// byte p of the emitted text read[start:stop] + read[us:ue]
__device__ __forceinline__ uint32_t key_byte(const uint8_t *seq, int start, int l1, int us, int p) {
  return p < l1 ? seq[start + p] : seq[us + p - l1];
}

// Reads of up to 16 * pack_words bases keep their 2-bit text in shared memory (pack_words + 3 rows of TRIM_THREADS
// words per CTA: + zero words so that 64-bit windows may start at any base).  The host picks 8 rows for batches of
// short reads (seven CTAs per SM fit) and MAX_PACK_WORDS for longer ones; longer reads take the whole-pipeline pass.
#define MAX_PACK_WORDS 10
#define PS_ROWS_OF(pw) ((pw) + 3)
// rows in use: a kernel argument, kept in shared memory for the device functions below (set by init_stats)
__shared__ int s_pack_words;
#define PACK_WORDS s_pack_words
#define PS_ROWS PS_ROWS_OF(s_pack_words)

// ---- split pipeline ----------------------------------------------------------------------------------------
// When every adapter qualifies for the bit-parallel search, the work of a read is cut at the first adapter
// modifier into kernels whose threads all do the same kind of work:
//   stage 1 (trim_kernel<32, true, 1>, all reads, bytes staged in shared memory): parse, 2-bit pack, the quality
//     modifiers, and an exact search for the whole adapter -- cutadapt stops at the leftmost exact occurrence, so
//     a hit settles the search.  Reads that need the DP are appended to a list (record index, window, packed
//     text); the keys of the modifiers before the adapter are emitted here.
//   stage 2 (trim_dp_kernel<true>, listed reads only, packed text only): counting sort of the CTA's reads by
//     window length, bit-vector search, remaining modifiers, emission.  Searches that need cost columns go to a
//     second list and
//   stage 3 (trim_dp_kernel<false>) runs them with recompute + traceback, again with full, sorted warps.
// Reads the split cannot take (non-ACGT characters, record groups larger than the staging buffer) go through
// trim_kernel<32, true, 2>, the whole pipeline per read from the global stream.
struct DpEntry {
  uint32_t r;      // record index in the batch
  uint32_t se;     // window at the adapter modifier: start | stop << 16
  uint32_t sl;     // read length
  uint32_t pad;
};

// first adapter modifier, and the number of emission slots stage 1 owns for a read that goes on to the search
__device__ __forceinline__ int first_adapter_mod() {
  int mi_ad = c_p.n_mods;
#pragma unroll 1
  for (int i = c_p.n_mods - 1; i >= 0; --i)
    if (c_p.kind[i] == MIRGE_MOD_ADAPTER) mi_ad = i;
  return mi_ad;
}

// Leftmost p in [start, stop - m] with read[p : p + m] == adapter, or -1.  Pure-ACGT read packed two bits per
// base (row stride TRIM_THREADS words, zero words after the text), plain adapter of m <= 32 bases in a2.  Per word
// of 16 positions, the positions whose first min(m, 4) bases agree come out of four SWAR compares at once (bit 2s
// of `cand` for position s: no branch per position); only those are compared in full, lowest first.
__device__ __forceinline__ int exact_find(const uint32_t *ps, uint64_t a2, int m, int start, int stop) {
  const int last = stop - m;
  if (last < start) return -1;
  const uint32_t a_lo = (uint32_t)a2, a_hi = (uint32_t)(a2 >> 32);
  const uint32_t lo_mask = m >= 16 ? 0xFFFFFFFFu : ((1u << (2 * m)) - 1u);
  const uint32_t hi_mask = m <= 16 ? 0u : (m >= 32 ? 0xFFFFFFFFu : ((1u << (2 * (m - 16))) - 1u));
  // adapter base k replicated into every 2-bit field (bases past m match anything: 0 fields, and no test)
  uint32_t rep[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) rep[k] = ((a_lo >> (2 * k)) & 3u) * 0x55555555u;
  int wb = start >> 4;
  uint32_t x0 = ps[wb * TRIM_THREADS], x1 = ps[(wb + 1) * TRIM_THREADS], x2 = ps[(wb + 2) * TRIM_THREADS];
#pragma unroll 1
  for (; 16 * wb <= last; ++wb) {
    uint32_t cand = 0x55555555u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (k < m) {
        const uint32_t e = (k ? __funnelshift_r(x0, x1, 2 * k) : x0) ^ rep[k];  // zero field: base s + k matches
        cand &= ~(e | (e >> 1));
      }
    }
    while (cand) {
      const int s = (__ffs((int)cand) - 1) >> 1;
      cand &= cand - 1u;
      const uint32_t lo = __funnelshift_r(x0, x1, 2 * s), hi = __funnelshift_r(x1, x2, 2 * s);
      const int p = 16 * wb + s;
      if (((lo ^ a_lo) & lo_mask) == 0u && ((hi ^ a_hi) & hi_mask) == 0u && p >= start && p <= last) return p;
    }
    x0 = x1;
    x1 = x2;
    x2 = (wb + 3 < PS_ROWS) ? ps[(wb + 3) * TRIM_THREADS] : 0u;
  }
  return -1;
}

// Insert list of the collapse: one entry per distinct key a read emits (arena / key buffer word offset, and how
// many consecutive emission slots carry that text), so that the insert kernel runs one key per lane with no
// filtered or repeated slots in between.  off == nullptr: no list wanted.
struct InsList {
  uint2 *off;  // (key word offset, count)
  uint64_t cap;
};
// ctrl[0] = insert-list entries << WORD_BITS | key words.  A batch is < 4 GiB and a record of l bases has >= 2l + 6
// bytes and <= MIRGE_MAX_MODS keys of <= 1 + l/16 + l words, so base (< 2^32) + key words of a batch < 2^36; the
// entries (<= records x slots, checked on the host side of mirge_trim) keep the 28 bits above.
#define WORD_BITS 36
#define WORD_MASK ((1ull << WORD_BITS) - 1ull)
#define MAX_LIST_ITEMS (1ull << (64 - WORD_BITS))

// per-CTA statistics: [0] emitted keys, [1] key words of all emitted keys
__shared__ unsigned int s_stats[2];
__device__ __forceinline__ void init_stats(int pack_words) {
  if (threadIdx.x < 2) s_stats[threadIdx.x] = 0;
  if (threadIdx.x == 0) s_pack_words = pack_words;
}
// all threads of the CTA, after their last emit_record
__device__ __forceinline__ void flush_stats(unsigned long long *ctrl) {
  __syncthreads();
  if (threadIdx.x == 0) {
    if (s_stats[0]) atomicAdd(ctrl + 1, (unsigned long long)s_stats[0]);
    if (s_stats[1]) atomicAdd(ctrl + 4, (unsigned long long)s_stats[1]);
  }
}

// Sizes, key space (one atomic per warp), second-pass queue and the writes of emission slots [slot_lo, slot_hi)
// of record r.  All 32 lanes of a warp must call it together.  fast_emit: the keys are slices of the packed
// pure-ACGT read in ps_mine; otherwise they are packed from the bytes in seq (exceptions included).
// to_slow: PASS 1 only, queues the record index in d_slow for the second pass (which redoes it from scratch).
template <bool FAST, int PASS>
__device__ __forceinline__ void emit_record(const bool valid, const uint64_t r, const int E, const int slot_lo, const int slot_hi,
                                            const uint8_t *seq, const bool fast_emit, const int *w_start, const int *w_stop,
                                            const int *w_us, const int *w_ue, uint32_t *w_words, const bool to_slow,
                                            ushort4 *__restrict__ win, uint32_t *__restrict__ key_off, uint32_t *__restrict__ keys,
                                            uint64_t keys_cap, unsigned long long *__restrict__ ctrl, uint32_t *__restrict__ d_slow,
                                            const uint32_t *ps_mine, const InsList il) {
  const int lane = threadIdx.x & 31;
  uint32_t my_words = 0, my_kept = 0, my_alg = 0, same_as_prev = 0, my_items = 0;
  if (valid) {
    // size of every kept key: header + payload + exceptions.  A slot whose text is the text of the slot before
    // it (a modifier that changed nothing: HEAD counting emits the read again) gets no space of its own -- its
    // key offset repeats the previous one and the collapse counts the run in one insert.
#pragma unroll 1
    for (int s = slot_lo; s < slot_hi; ++s) {
      if (!w_words[s]) continue;
      ++my_kept;
      if (s > slot_lo && w_words[s - 1] && w_start[s] == w_start[s - 1] && w_stop[s] == w_stop[s - 1] && w_us[s] == w_us[s - 1] &&
          w_ue[s] == w_ue[s - 1]) {
        w_words[s] = w_words[s - 1];
        my_alg += w_words[s];
        same_as_prev |= 1u << s;
        continue;
      }
      if (FAST && fast_emit) {
        w_words[s] = 1u + ((uint32_t)(w_stop[s] - w_start[s] + 15) >> 4);
      } else {
        const int l1 = w_stop[s] - w_start[s], len = l1 + (w_ue[s] - w_us[s]);
        uint32_t nexc = 0;
        for (int p = 0; p < len; ++p) nexc += base_code_exact(key_byte(seq, w_start[s], l1, w_us[s], p)) == 4u;
        w_words[s] = 1u + ((uint32_t)(len + 15) >> 4) + nexc;
      }
      my_words += w_words[s];
      my_alg += w_words[s];
      ++my_items;
    }
  }
  // one scan for both prefixes: key words in the low 24 bits (<= 8 slots x 545 words x 32 lanes < 2^18), insert-list
  // items (distinct keys of the read, <= 8 per lane) above
  uint32_t inc = my_words | (my_items << 24);
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= d) inc += t;
  }
  const uint32_t both_total = __shfl_sync(0xffffffffu, inc, 31);
  const uint32_t warp_total = both_total & 0xFFFFFFu, warp_items = both_total >> 24;
  const uint32_t item_before = (inc >> 24) - my_items;
  inc &= 0xFFFFFFu;
  const uint32_t kept_warp = __reduce_add_sync(0xffffffffu, my_kept);
  const uint32_t alg_warp = __reduce_add_sync(0xffffffffu, my_alg);
  // ONE global atomic per warp hands out the key words (low WORD_BITS bits of ctrl[0]) and the insert-list entries
  // (bits above) together; the two statistics go through the CTA's shared-memory counters (flushed once per CTA by
  // flush_stats): same-line atomics of every warp of the grid serialise in one L2 atomic unit, and the key-space
  // atomic is on every warp's critical path.
  unsigned long long both = 0;
  if (lane == 0) {
    if (both_total) both = atomicAdd(ctrl + 0, ((unsigned long long)warp_items << WORD_BITS) | (unsigned long long)warp_total);
    if (kept_warp) atomicAdd(&s_stats[0], kept_warp);
    if (alg_warp) atomicAdd(&s_stats[1], alg_warp);  // key words of all emitted keys (repeats included)
  }
  both = __shfl_sync(0xffffffffu, both, 0);
  const unsigned long long warp_base = both & WORD_MASK, item_base = both >> WORD_BITS;
  const bool overflow = warp_base + warp_total > keys_cap || warp_base + warp_total > 0xFFFFFFF0ull;
  if (overflow && lane == 0 && warp_total) atomicOr(ctrl + 2, 2ull);
  if (PASS == 1) {  // queue the deferred reads for the second pass (one atomic per warp)
    const unsigned sm_ = __ballot_sync(0xffffffffu, to_slow);
    if (sm_) {
      unsigned long long base = 0;
      if (lane == __ffs(sm_) - 1) base = atomicAdd(ctrl + 5, (unsigned long long)__popc(sm_));
      base = __shfl_sync(0xffffffffu, base, __ffs(sm_) - 1);
      if (to_slow) d_slow[base + __popc(sm_ & ((1u << lane) - 1u))] = (uint32_t)r;
    }
  }
  if (!valid) return;
  uint32_t off = (uint32_t)warp_base + inc - my_words;
  uint64_t item = item_base + item_before;
#pragma unroll 1
  for (int s = slot_lo; s < slot_hi; ++s) {
    const uint64_t e = r * (uint64_t)E + s;
    if (win) win[e] = make_ushort4((unsigned short)w_start[s], (unsigned short)w_stop[s], (unsigned short)w_us[s], (unsigned short)w_ue[s]);
    if (!w_words[s] || overflow) {
      if (key_off) key_off[e] = 0xFFFFFFFFu;
      continue;
    }
    if ((same_as_prev >> s) & 1u) {  // same text as the previous slot: same key
      if (key_off) key_off[e] = off - w_words[s];
      continue;
    }
    if (key_off) key_off[e] = off;
    if (il.off && item < il.cap) {  // one insert per distinct key: the run of slots that repeat it is its count
      const uint32_t run = (uint32_t)__ffs((int)(~(same_as_prev >> (s + 1)) | (1u << (slot_hi - s - 1))));
      il.off[item] = make_uint2(off, run);
      ++item;
    }
    const int l1 = w_stop[s] - w_start[s], len = l1 + (w_ue[s] - w_us[s]);
    const uint32_t npay = (uint32_t)(len + 15) >> 4;
    uint32_t *k = keys + off;
    if (FAST && fast_emit) {
      // key = 2-bit text of read[w_start : w_stop): a slice of the packed read in shared memory
      k[0] = (uint32_t)len;
      const int wi = w_start[s] >> 4;
      const uint32_t bs = 2u * (uint32_t)(w_start[s] & 15);
      uint32_t lo = ps_mine[wi * TRIM_THREADS];
#pragma unroll 1
      for (uint32_t w = 0; w < npay; ++w) {
        const uint32_t hi = ps_mine[(wi + w + 1) * TRIM_THREADS];
        uint32_t v = __funnelshift_r(lo, hi, bs);
        lo = hi;
        const int rem = len - 16 * (int)w;
        if (rem < 16) v &= (1u << (2 * rem)) - 1u;
        k[1 + w] = v;
      }
    } else {
      const uint32_t nexc = w_words[s] - 1u - npay;
      k[0] = (uint32_t)len | (nexc << 16);
      uint32_t word = 0, xi = 0;
      for (int p = 0; p < len; ++p) {
        const uint32_t ch = key_byte(seq, w_start[s], l1, w_us[s], p);
        const uint32_t code = base_code_exact(ch);
        if (code == 4u) k[1 + npay + xi++] = ((uint32_t)p << 8) | ch;
        else word |= code << (2 * (p & 15));
        if ((p & 15) == 15) { k[1 + (p >> 4)] = word; word = 0; }
      }
      if (len & 15) k[1 + (len >> 4)] = word;
    }
    off += w_words[s];
  }
}

// window of the read after modifier mi_ -> its emission slot (HEAD: one slot per modifier, digest.py:354-373)
#define RECORD_SLOT(mi_)                                                                         \
  if (!qia && (E != 1 || (mi_) == n_mods - 1)) {                                                 \
    const int slot_ = (E == 1) ? 0 : (mi_);                                                      \
    int ln_ = stop - start;                                                                      \
    if (c_p.umi_mode == MIRGE_UMI_FLANKS) ln_ = max(ln_ - c_p.umi5 - c_p.umi3, 0);               \
    w_start[slot_] = start; w_stop[slot_] = stop; w_words[slot_] = ln_ >= c_p.min_len;           \
  }

struct SplitOut {  // where stage 1 leaves the reads that need the DP
  DpEntry *entries;
  uint32_t *pk;   // packed text, word w of list entry e at pk[w * cap + e]
  uint64_t cap;
};

// Everything a thread does for record r once its bytes are addressable through B (shared-memory staging or
// the global stream).  PASS 0: single pass; PASS 1: first pass (reads whose adapter search needs cost
// columns are appended to d_slow and emit nothing); PASS 2: second pass over those reads.
// SPLIT (PASS 1 of the bit-parallel kernel): stage 1 of the split pipeline described above.
template <int MAXM, bool FAST, int PASS, bool SPLIT>
__device__ __forceinline__ void process_record(const bool valid, const uint64_t r, const uint8_t *B, uint64_t nbytes,
                                               const uint32_t *__restrict__ line_start, ushort4 *__restrict__ win,
                                               uint32_t *__restrict__ key_off, uint32_t *__restrict__ keys, uint64_t keys_cap,
                                               unsigned long long *__restrict__ ctrl, uint32_t *__restrict__ d_slow, FastCtx &fc,
                                               uint32_t *ps_mine, const SplitOut so, const uint4 ls, const uint32_t nxt,
                                               const InsList il) {
  const int lane = threadIdx.x & 31;
  bool is_slow = false;
  const int E = c_p.slots;
  const int n_mods = c_p.n_mods;
  const bool qia = c_p.umi_mode == MIRGE_UMI_QIAGEN;
  // per-slot windows live in local memory (dynamic slot index keeps the code small)
  int w_start[MIRGE_MAX_MODS], w_stop[MIRGE_MAX_MODS], w_us[MIRGE_MAX_MODS], w_ue[MIRGE_MAX_MODS];
  uint32_t w_words[MIRGE_MAX_MODS];  // 0 = not kept
#pragma unroll 1
  for (int s = 0; s < E; ++s) { w_start[s] = w_stop[s] = w_us[s] = w_ue[s] = 0; w_words[s] = 0; }
  const uint8_t *seq = nullptr, *qual = nullptr;
  uint32_t seq_off = 0;
  bool fast_emit = FAST, good = false;
  int sl = 0, start = 0, stop = 0;
  if (valid) {  // ls / nxt: line_start[4r .. 4r+4], loaded by the caller
    sl = (int)(ls.z - 1 - ls.y);
    int ql = (int)(nxt - 1 - ls.w);
    if (sl > 0 && B[ls.y + sl - 1] == '\r') --sl;
    if (ql > 0 && B[ls.w + ql - 1] == '\r') --ql;
    const bool bad = B[ls.x] != '@' || B[ls.z] != '+' || sl != ql || sl > MIRGE_MAX_READ_LEN;
    if (bad) {
      atomicOr(ctrl + 2, (sl > MIRGE_MAX_READ_LEN && sl == ql) ? 4ull : 1ull);
      atomicMax(ctrl + 3, ~(unsigned long long)r);
    } else {
      good = true;
      seq_off = ls.y;
      seq = B + ls.y;
      qual = B + ls.w;
      stop = sl;
    }
  }
  // lanes that run the modifier pipeline together; used to re-converge them after every modifier,
  // whose data-dependent loops (quality scans, adapter search) otherwise leave the warp split
  const unsigned good_lanes = __ballot_sync(0xffffffffu, good);
  if (good && FAST) {
    // 2-bit text of the whole read once, four bytes per step (SIMD-in-register), into shared memory:
    // used by the exact search, the traceback jumps and by key emission
    fast_emit = sl <= 16 * PACK_WORDS;
    if (PASS == 2 && (uint64_t)seq_off + 16 * ((sl + 15) >> 4) + 8 > nbytes) fast_emit = false;  // no over-read past the stream
    if (fast_emit) {
      const uint32_t *ap = (const uint32_t *)((uintptr_t)seq & ~(uintptr_t)3);
      const uint32_t bs = ((uint32_t)(uintptr_t)seq & 3u) * 8u;
      const int nwords = (sl + 15) >> 4;
      uint32_t anyexc = 0, prev = ap[0];
      int k = 1;
#pragma unroll 1
      for (int w = 0; w < nwords; ++w) {
        uint32_t word = 0;
#pragma unroll
        for (int q4 = 0; q4 < 4; ++q4) {
          const uint32_t nx = ap[k++];
          const uint32_t quad = __funnelshift_r(prev, nx, bs);
          prev = nx;
          const int nb = sl - (16 * w + 4 * q4);  // bytes of this quad that belong to the read
          uint32_t codes = ((quad >> 1) ^ (quad >> 2)) & 0x03030303u;
          // the byte each 2-bit code stands for, looked up with one PRMT: a byte that differs is not ACGT
          uint32_t sel = codes | (codes >> 4);
          sel = (sel & 0xFFu) | ((sel >> 8) & 0xFF00u);
          uint32_t diff = __byte_perm(0x54474341u, 0u, sel) ^ quad;
          if (nb < 4) {
            const uint32_t tm = nb <= 0 ? 0u : (0xFFFFFFFFu >> (8 * (4 - nb)));
            codes &= tm;
            diff &= tm;
          }
          anyexc |= diff;
          word |= ((codes * 0x01041040u) >> 24) << (8 * q4);
        }
        ps_mine[w * TRIM_THREADS] = word;
      }
#pragma unroll 1
      for (int w = nwords; w < PS_ROWS; ++w) ps_mine[w * TRIM_THREADS] = 0;
      if (anyexc) fast_emit = false;
    }
    fc.jump_ok = fast_emit;
  }

#define RUN_MODS(from_, to_)                                                                     \
  _Pragma("unroll 1") for (int mi = (from_); mi < (to_); ++mi) {                                 \
    if (!is_slow) is_slow = apply_mod<MAXM, FAST, PASS == 1>(mi, seq, qual, start, stop, fc);    \
    __syncwarp(good_lanes);                                                                      \
    RECORD_SLOT(mi)                                                                              \
  }

  int slot_lo = 0, slot_hi = E;
  bool to_slow = false;
  if constexpr (!SPLIT) {
    if (good) { RUN_MODS(0, n_mods) }
  } else {
    const int mi_ad = first_adapter_mod();
    if (good) {
      _Pragma("unroll 1") for (int mi = 0; mi < mi_ad; ++mi) {
        apply_plain_mod(mi, seq, qual, start, stop);
        __syncwarp(good_lanes);
        RECORD_SLOT(mi)
      }
    }
    bool to_dp = false, resolved = false;
    if (good && mi_ad < n_mods) {
      const DevAdapter &ad0 = c_p.ad[0];
      const bool exact_ok = c_p.n_adapters == 1 && c_p.times == 1 && !ad0.wildcard_ref && ad0.acc[ad0.m] >= 0;
      int p = -1;
      if (fc.jump_ok && exact_ok) p = exact_find(ps_mine, ad0.a2, ad0.m, start, stop);
      __syncwarp(good_lanes);  // the search leaves its loop at a different word in every lane
      if (!fc.jump_ok) {
        is_slow = true;  // non-ACGT characters or a long read: whole record in the second pass
      } else if (p >= 0) {
        stop = p;
        resolved = true;
      } else {
        to_dp = true;
      }
      if (resolved) { RECORD_SLOT(mi_ad) }
    }
    if (good) {  // the modifiers after the adapter, for the reads the exact search settled (all good lanes re-converge)
      _Pragma("unroll 1") for (int mi = mi_ad + 1; mi < n_mods; ++mi) {
        if (resolved && !is_slow) {
          const int kind = c_p.kind[mi];
          if (kind == MIRGE_MOD_NEND) {
            while (start < stop && seq[start] == 'N') ++start;
            while (stop > start && seq[stop - 1] == 'N') --stop;
          } else if (kind == MIRGE_MOD_CUT) {
            const int c = c_p.a[mi], len = stop - start;
            if (c > 0) start += min(c, len);
            else stop = start + max(len + c, 0);
          } else {
            is_slow = true;  // a second adapter modifier (stipulate() builds one at most): whole record in the second pass
          }
        }
        __syncwarp(good_lanes);
        if (resolved) { RECORD_SLOT(mi) }
      }
    }
    // the reads that need the DP: one list slot per read, one atomic per warp
    const unsigned dm = __ballot_sync(0xffffffffu, to_dp);
    if (dm) {
      const int leader = __ffs(dm) - 1;
      unsigned long long base = 0;
      if (lane == leader) base = atomicAdd(ctrl + 6, (unsigned long long)__popc(dm));
      base = __shfl_sync(0xffffffffu, base, leader);
      if (to_dp) {
        const uint64_t e = base + __popc(dm & ((1u << lane) - 1u));
        DpEntry de;
        de.r = (uint32_t)r; de.se = (uint32_t)start | ((uint32_t)stop << 16); de.sl = (uint32_t)sl; de.pad = 0;
        *(uint4 *)(so.entries + e) = *(const uint4 *)&de;
        const int nwords = (sl + 15) >> 4;
#pragma unroll 1
        for (int w = 0; w < nwords; ++w) so.pk[(uint64_t)w * so.cap + e] = ps_mine[w * TRIM_THREADS];
      }
    }
    if (to_dp) slot_hi = (E == 1) ? 0 : mi_ad;  // the later slots belong to stage 2
  }
#undef RUN_MODS

  if (good) {
    if (qia) {
      const int tl = stop - start, U = c_p.umi3;
      int us = 0, ue = 0;
      if (tl > 0) {
        const int first = find_sub(seq, sl, seq + start, tl, 0);
        const int after = first + tl;
        const int nx = find_sub(seq, sl, seq + start, tl, after);
        int seg_end = nx < 0 ? sl : nx;
        seg_end = min(seg_end, after + c_p.qia_len + U);
        ue = seg_end;
        us = (U != 0) ? max(seg_end - U, after) : after;
      }
      w_start[0] = start; w_stop[0] = stop; w_us[0] = us; w_ue[0] = ue;
      w_words[0] = (tl >= c_p.min_len) ? 1u : 0u;
      if (ue > us) fast_emit = false;  // concatenated key: generic packing
    }
    if (PASS == 1 && is_slow) {
      // second pass will redo this read from scratch; emit nothing now
      slot_hi = slot_lo;
      to_slow = true;
    }
  }
  emit_record<FAST, PASS>(valid, r, E, slot_lo, slot_hi, seq, fast_emit, w_start, w_stop, w_us, w_ue, w_words, to_slow, win, key_off,
                          keys, keys_cap, ctrl, d_slow, ps_mine, il);
}

// FAST = bit-parallel adapter search (locate_fast) + packed-read key emission; requires the CTA's span to be
// staged in shared memory, otherwise the batch is flagged (ctrl[2] bit 3) for the generic kernel.
// SPLIT: stage 1 of the split pipeline (only with FAST and PASS 1).
template <int MAXM, bool FAST, int PASS, bool SPLIT>
__global__ void __launch_bounds__(TRIM_THREADS, (FAST && PASS == 1) ? 7 : 1)
trim_kernel(const uint8_t *__restrict__ fq, uint64_t nbytes, const uint32_t *__restrict__ line_start, uint64_t n_records,
            ushort4 *__restrict__ win, uint32_t *__restrict__ key_off, uint32_t *__restrict__ keys, uint64_t keys_cap,
            unsigned long long *__restrict__ ctrl, uint32_t smem_bytes, uint32_t *__restrict__ d_slow, const SplitOut so,
            const InsList il, const int pack_words) {
  extern __shared__ uint4 smem4[];
  uint8_t *sbuf = (uint8_t *)smem4;
  const int tid = threadIdx.x;
  FastCtx fc;
  fc.s_eq = nullptr; fc.ps = nullptr; fc.jump_ok = false; fc.rbase = 0;
  uint32_t *ps_mine = nullptr;
  init_stats(pack_words);  // (a barrier follows before any emission on every path below)
  if (FAST) {
    // smem: [staging smem_bytes][eq tables n_adapters * 256 words][packed reads PS_ROWS * T words]
    uint32_t *eq = (uint32_t *)(sbuf + smem_bytes);
    for (int e = tid; e < c_p.n_adapters * 256; e += TRIM_THREADS) {
      const uint32_t code = base_code_upper((uint32_t)(e & 255));
      eq[e] = code < 4u ? (uint32_t)c_p.ad[e >> 8].peq[code] : 0u;
    }
    fc.s_eq = eq;
    ps_mine = eq + c_p.n_adapters * 256 + tid;
    fc.ps = ps_mine;
  }
  if (PASS == 2) {
    // second pass: the deferred reads, addressed in the global stream; whole warps iterate together
    __syncthreads();
    const unsigned long long n_slow = ctrl[5];
    const uint64_t first = (uint64_t)blockIdx.x * TRIM_THREADS + (tid & ~31);
    for (uint64_t base = first; base < n_slow; base += (uint64_t)gridDim.x * TRIM_THREADS) {
      const uint64_t idx = base + (tid & 31);
      const bool valid = idx < n_slow;
      uint64_t r = 0;
      fc.jump_ok = false;
      uint4 ls = make_uint4(0, 0, 0, 0);
      uint32_t nxt = 0;
      if (valid) {
        r = d_slow[idx];
        ls = *(const uint4 *)(line_start + 4 * r);
        nxt = line_start[4 * r + 4];
      }
      process_record<MAXM, FAST, 2, false>(valid, r, fq, nbytes, line_start, win, key_off, keys, keys_cap, ctrl,
                                           d_slow, fc, ps_mine, so, ls, nxt, il);
      __syncwarp();
    }
    flush_stats(ctrl);
    return;
  }
  const uint64_t r0 = (uint64_t)blockIdx.x * TRIM_THREADS;
  const uint64_t r = r0 + tid;
  const bool valid = r < n_records;
  const uint64_t r_end = min(r0 + (uint64_t)TRIM_THREADS, n_records);
  const uint32_t span_lo = line_start[4 * r0];
  const uint64_t span_hi = min((uint64_t)line_start[4 * r_end], nbytes);
  const uint32_t alo = span_lo & ~15u;
  const bool staged = (span_hi - alo) <= smem_bytes;
  if (FAST && !staged) {  // uniform per CTA
    if (PASS == 1) {
      // this group's bytes do not fit the staging buffer: hand all of its reads to the second pass
      const unsigned vm = __ballot_sync(0xffffffffu, valid);
      if (vm) {
        const int lane = tid & 31;
        unsigned long long base = 0;
        if (lane == __ffs(vm) - 1) base = atomicAdd(ctrl + 5, (unsigned long long)__popc(vm));
        base = __shfl_sync(0xffffffffu, base, __ffs(vm) - 1);
        if (valid) d_slow[base + __popc(vm & ((1u << lane) - 1u))] = (uint32_t)r;
      }
      return;
    }
    if (tid == 0) atomicOr(ctrl + 2, 8ull);
    return;
  }
  if (staged) {
    for (uint64_t o = (uint64_t)tid * 16; alo + o < span_hi; o += TRIM_THREADS * 16) {
      const uint64_t g = alo + o;
      if (g + 16 <= nbytes) {
        cp_async_16(sbuf + o, fq + g);  // all of a thread's pieces in flight together, L1 bypassed
      } else {
        for (int b = 0; b < 16 && g + b < nbytes; ++b) sbuf[o + b] = fq[g + b];
      }
    }
    cp_async_wait_all();
  }
  __syncthreads();
  // (fetching these ahead of the staging wait measured slower: 19.0-19.3 vs 18.5 ms per 50 M reads)
  uint4 ls = make_uint4(0, 0, 0, 0);
  uint32_t nxt = 0;
  if (valid) { ls = *(const uint4 *)(line_start + 4 * r); nxt = line_start[4 * r + 4]; }
  const uint8_t *B = staged ? (const uint8_t *)(sbuf - alo) : fq;  // B[absolute stream offset]
  process_record<MAXM, FAST, PASS, SPLIT>(valid, r, B, nbytes, line_start, win, key_off, keys, keys_cap, ctrl, d_slow, fc, ps_mine, so, ls, nxt, il);
  flush_stats(ctrl);
}

// Stages 2 and 3 of the split pipeline: the adapter search (and everything after it) of the listed reads, from
// their packed text alone.  FIRST: stage 2 -- entries [0, ctrl[6]), searches that need cost columns are appended
// to `redo` (ctrl[7]); !FIRST: stage 3 -- the entries listed in `redo`, resolved with recompute + traceback.
template <bool FIRST>
__global__ void __launch_bounds__(TRIM_THREADS, FIRST ? 7 : 4)
trim_dp_kernel(const DpEntry *__restrict__ entries, const uint32_t *__restrict__ pk, uint64_t cap, uint32_t *__restrict__ redo,
               ushort4 *__restrict__ win, uint32_t *__restrict__ key_off, uint32_t *__restrict__ keys, uint64_t keys_cap,
               unsigned long long *__restrict__ ctrl, const InsList il, const int pack_words) {
  extern __shared__ uint4 smem4[];
  // smem: [eq tables n_adapters * 256 words, entries 0..3 used][packed reads PS_ROWS * T words][entries T][hist T][order T]
  uint32_t *eq = (uint32_t *)smem4;
  uint32_t *ps_base = eq + c_p.n_adapters * 256;
  DpEntry *s_ent = (DpEntry *)(ps_base + PS_ROWS_OF(pack_words) * TRIM_THREADS);  // (the kernel argument: the shared copy is not set yet)
  uint32_t *s_hist = (uint32_t *)(s_ent + TRIM_THREADS);
  uint16_t *s_order = (uint16_t *)(s_hist + TRIM_THREADS);
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned long long n_items = FIRST ? ctrl[6] : ctrl[7];
  const uint64_t base = (uint64_t)blockIdx.x * TRIM_THREADS;
  if (base >= n_items) return;  // uniform per CTA
  init_stats(pack_words);
  for (int e = tid; e < c_p.n_adapters * 4; e += TRIM_THREADS) eq[(e >> 2) * 256 + (e & 3)] = (uint32_t)c_p.ad[e >> 2].peq[e & 3];
  const int n_here = (int)min((unsigned long long)TRIM_THREADS, n_items - base);
  // this CTA's entries, then a counting sort by window length (longest first): the lanes of a warp run column
  // loops of similar trip count
  uint32_t my_e = 0;
  int bin = TRIM_THREADS - 1;
  if (tid < n_here) {
    my_e = FIRST ? (uint32_t)(base + tid) : redo[base + tid];
    const uint4 v = *(const uint4 *)(entries + my_e);
    DpEntry de = *(const DpEntry *)&v;
    de.pad = my_e;
    s_ent[tid] = de;
    const int wl = (int)(de.se >> 16) - (int)(de.se & 0xFFFFu);
    bin = TRIM_THREADS - 1 - min(wl, TRIM_THREADS - 1);
  }
  s_hist[tid] = 0;
  __syncthreads();
  if (tid < n_here) atomicAdd(&s_hist[bin], 1u);
  __syncthreads();
  if (tid < 32) {
    uint32_t h[TRIM_THREADS / 32], sum = 0;
#pragma unroll
    for (int q = 0; q < TRIM_THREADS / 32; ++q) { h[q] = s_hist[(TRIM_THREADS / 32) * tid + q]; sum += h[q]; }
    uint32_t incl = sum;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t x = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += x;
    }
    uint32_t run = incl - sum;
#pragma unroll
    for (int q = 0; q < TRIM_THREADS / 32; ++q) { s_hist[(TRIM_THREADS / 32) * tid + q] = run; run += h[q]; }
  }
  __syncthreads();
  if (tid < n_here) s_order[atomicAdd(&s_hist[bin], 1u)] = (uint16_t)tid;
  __syncthreads();
  const bool valid = tid < n_here;
  const int E = c_p.slots, n_mods = c_p.n_mods;
  const bool qia = false;  // the split pipeline is not used with qiagen UMIs
  int w_start[MIRGE_MAX_MODS], w_stop[MIRGE_MAX_MODS], w_us[MIRGE_MAX_MODS], w_ue[MIRGE_MAX_MODS];
  uint32_t w_words[MIRGE_MAX_MODS];
#pragma unroll 1
  for (int s = 0; s < E; ++s) { w_start[s] = w_stop[s] = w_us[s] = w_ue[s] = 0; w_words[s] = 0; }
  uint32_t *ps_mine = ps_base + tid;
  const int mi_ad = first_adapter_mod();
  uint64_t r = 0;
  bool need_redo = false;
  int slot_lo = (E == 1) ? 0 : mi_ad, slot_hi = E;
  uint32_t ent_id = 0;
  if (valid) {
    const DpEntry de = s_ent[s_order[tid]];
    r = de.r;
    ent_id = de.pad;
    int start = (int)(de.se & 0xFFFFu), stop = (int)(de.se >> 16);
    const int nwords = ((int)de.sl + 15) >> 4;
    // the packed rows of this read: asynchronous copies, all in flight together (own column only: no barrier)
#pragma unroll 1
    for (int w = 0; w < PS_ROWS_OF(pack_words); ++w) {
      if (w < nwords) cp_async_4(ps_mine + w * TRIM_THREADS, pk + (uint64_t)w * cap + ent_id);
      else ps_mine[w * TRIM_THREADS] = 0u;
    }
    cp_async_wait_all();
    FastCtx fc;
    fc.s_eq = eq; fc.ps = ps_mine; fc.jump_ok = true; fc.rbase = 0;
#pragma unroll 1
    for (int mi = mi_ad; mi < n_mods && !need_redo; ++mi) {
      const int kind = c_p.kind[mi];
      if (kind == MIRGE_MOD_ADAPTER) {
#pragma unroll 1
        for (int t = 0; t < c_p.times; ++t) {
          fc.rbase = start;
          const PackedRead rv{ps_mine, start};
          const int n = stop - start;
          Match best;
          int which = -1;
#pragma unroll 1
          for (int a = 0; a < c_p.n_adapters; ++a) {
            Match mt;
            const int rc = locate_fast<FIRST>(a, rv, n, fc, mt);
            if (rc == 2) { need_redo = true; break; }
            if (rc == 0) continue;
            if (which < 0 || mt.matches > best.matches || (mt.matches == best.matches && mt.errors < best.errors)) { best = mt; which = a; }
          }
          if (need_redo || which < 0) break;
          stop = start + best.rstart;  // every adapter of the bit-parallel path is a 3' adapter
        }
      } else if (kind == MIRGE_MOD_CUT) {
        const int c = c_p.a[mi], len = stop - start;
        if (c > 0) start += min(c, len);
        else stop = start + max(len + c, 0);
      }  // MIRGE_MOD_NEND: a pure-ACGT read has no N to strip; quality modifiers cannot follow (checked on the host)
      if (!need_redo) { RECORD_SLOT(mi) }
    }
  }
  if (FIRST) {  // searches that need cost columns: third stage
    const unsigned rm = __ballot_sync(0xffffffffu, need_redo);
    if (rm) {
      const int leader = __ffs(rm) - 1;
      unsigned long long b2 = 0;
      if (lane == leader) b2 = atomicAdd(ctrl + 7, (unsigned long long)__popc(rm));
      b2 = __shfl_sync(0xffffffffu, b2, leader);
      if (need_redo) redo[b2 + __popc(rm & ((1u << lane) - 1u))] = ent_id;
    }
    if (need_redo) slot_hi = slot_lo;
  }
  emit_record<true, 0>(valid, r, E, slot_lo, slot_hi, nullptr, true, w_start, w_stop, w_us, w_ue, w_words, false, win, key_off, keys, keys_cap,
                       ctrl, nullptr, ps_mine, il);
  flush_stats(ctrl);
}

// scratch layout of mirge_trim: [second-pass list u32[n]][stage-3 list u32[n]][DpEntry[n]][packed text u32[MAX_PACK_WORDS][n]]
static uint64_t align16(uint64_t x) { return (x + 15) & ~15ull; }
extern "C" uint64_t mirge_trim_scratch_bytes(uint64_t n_records) {
  const uint64_t n = n_records ? n_records : 1;
  return 2 * align16(4 * n) + align16(sizeof(DpEntry) * n) + align16(4ull * MAX_PACK_WORDS * n) + 64;
}

extern "C" int mirge_trim(mirge_ctx *ctx, const uint8_t *d_fastq, uint64_t nbytes, const uint32_t *d_line_start, uint64_t n_records,
                          uint16_t *d_win, uint32_t *d_key_off, uint32_t *d_keys, uint64_t keys_capacity_words,
                          uint64_t *d_trim_ctrl, void *d_scratch, uint64_t *d_ins, uint64_t ins_capacity, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!ctx->params_set) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: mirge_set_trim_params has not been called");
  if (n_records == 0) return MIRGE_OK;
  if (!d_fastq || !d_line_start || !d_keys || !d_trim_ctrl) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: null buffer");
  if (!d_win != !d_key_off) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: d_win and d_key_off go together");
  if (!d_key_off && !d_ins) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: neither per-slot outputs nor an insert list requested");
  if (d_ins && (ins_capacity == 0 || ((uintptr_t)d_ins & 7))) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: bad insert list");
  if (n_records * (uint64_t)trim_slots_of(&ctx->params) >= MAX_LIST_ITEMS)
    MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: more than 2^28 emission slots in one batch (use smaller batches)");
  if (((uintptr_t)d_line_start & 15) || ((uintptr_t)d_win & 7) || ((uintptr_t)d_scratch & 15))
    MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: misaligned buffer");
  const InsList il{(uint2 *)d_ins, d_ins ? ins_capacity : 0};
  if (n_records >= 0x80000000ull) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: more than 2^31 records in one batch");
  // same convention as the tokeniser: line_start offsets are relative to the 16-byte aligned stream
  {
    const uint32_t skew = (uint32_t)((uintptr_t)d_fastq & 15);
    d_fastq -= skew;
    nbytes += skew;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  const uint64_t avg = (nbytes + n_records - 1) / n_records;
  const bool fast = ctx->fast_ok && ctx->trim_mode != 1;
  const bool split = fast && ctx->split_ok && ctx->trim_mode == 0;
  // staging buffer: the bit-parallel kernel keeps it tight (7 CTAs per SM); a record group that does not fit
  // is handed to its second pass.  The generic kernel reads such groups straight from global memory.
  uint64_t want = fast ? avg * TRIM_THREADS * 33 / 32 + 512 : avg * TRIM_THREADS * 5 / 4 + 64;
  want = (want + 255) & ~255ull;
  if (want < 4096) want = 4096;
  if (want > 96 * 1024) want = 96 * 1024;
  const uint32_t smem = (uint32_t)want;
  const unsigned grid = (unsigned)((n_records + TRIM_THREADS - 1) / TRIM_THREADS);
  unsigned long long *ctrl = (unsigned long long *)d_trim_ctrl;
  ushort4 *win = (ushort4 *)d_win;
  SplitOut so;
  so.entries = nullptr; so.pk = nullptr; so.cap = 0;
  if (fast) {
    if (!d_scratch) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "trim: scratch of mirge_trim_scratch_bytes(n_records) bytes is required");
    uint8_t *sc = (uint8_t *)d_scratch;
    uint32_t *d_slow = (uint32_t *)sc;
    uint32_t *d_redo = (uint32_t *)(sc + align16(4 * n_records));
    so.entries = (DpEntry *)(sc + 2 * align16(4 * n_records));
    so.pk = (uint32_t *)(sc + 2 * align16(4 * n_records) + align16(sizeof(DpEntry) * n_records));
    so.cap = n_records;
    // packed-read rows: 8 words cover reads of up to 128 bases (record = header + 2 x read + 6 bytes)
    const int pack_words = avg <= 2 * 112 + 40 ? 8 : MAX_PACK_WORDS;
    const size_t extra = (size_t)ctx->params.n_adapters * 1024 + (size_t)PS_ROWS_OF(pack_words) * TRIM_THREADS * 4;
    if (split) {
      // stage 1: every read up to the adapter modifier; exact adapter occurrences are settled here
      MIRGE_CUDA(ctx, cudaFuncSetAttribute(trim_kernel<32, true, 1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      trim_kernel<32, true, 1, true><<<grid, TRIM_THREADS, smem + extra, stream>>>(d_fastq, nbytes, d_line_start, n_records, win, d_key_off,
                                                                                 d_keys, keys_capacity_words, ctrl, smem, d_slow, so, il, pack_words);
      MIRGE_LAUNCH_CHECK(ctx, "trim_kernel(stage 1)");
      // stages 2 and 3: the listed reads (counts live on the device: CTAs beyond the list exit at once)
      const size_t dp_smem = extra + (size_t)TRIM_THREADS * (sizeof(DpEntry) + 4 + 2);
      trim_dp_kernel<true><<<grid, TRIM_THREADS, dp_smem, stream>>>(so.entries, so.pk, so.cap, d_redo, win, d_key_off, d_keys,
                                                                    keys_capacity_words, ctrl, il, pack_words);
      MIRGE_LAUNCH_CHECK(ctx, "trim_dp_kernel(stage 2)");
      trim_dp_kernel<false><<<grid, TRIM_THREADS, dp_smem, stream>>>(so.entries, so.pk, so.cap, d_redo, win, d_key_off, d_keys,
                                                                     keys_capacity_words, ctrl, il, pack_words);
      MIRGE_LAUNCH_CHECK(ctx, "trim_dp_kernel(stage 3)");
    } else {
      MIRGE_CUDA(ctx, cudaFuncSetAttribute(trim_kernel<32, true, 1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      // pass 1: every read; adapter searches that need cost columns are deferred to the list d_slow
      trim_kernel<32, true, 1, false><<<grid, TRIM_THREADS, smem + extra, stream>>>(d_fastq, nbytes, d_line_start, n_records, win,
                                                                                  d_key_off, d_keys, keys_capacity_words, ctrl, smem,
                                                                                  d_slow, so, il, pack_words);
      MIRGE_LAUNCH_CHECK(ctx, "trim_kernel(pass 1)");
    }
    // pass 2: the reads left over (whole pipeline per read, from the global stream; grid-stride over the list)
    // (one read per thread where possible: a read's whole pipeline is a long dependent chain, so the list is
    // spread over many warps instead of looping inside few)
    unsigned grid2 = split ? grid / 4 + 1 : grid / 16 + 1;
    if (grid2 > (unsigned)ctx->sm_count * (split ? 64u : 8u)) grid2 = (unsigned)ctx->sm_count * (split ? 64u : 8u);
    trim_kernel<32, true, 2, false><<<grid2, TRIM_THREADS, extra, stream>>>(d_fastq, nbytes, d_line_start, n_records, win, d_key_off,
                                                                          d_keys, keys_capacity_words, ctrl, 0u, d_slow, so, il, pack_words);
  } else if (ctx->max_adapter_len <= 32) {
    MIRGE_CUDA(ctx, cudaFuncSetAttribute(trim_kernel<32, false, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    trim_kernel<32, false, 0, false><<<grid, TRIM_THREADS, smem, stream>>>(d_fastq, nbytes, d_line_start, n_records, win, d_key_off,
                                                                           d_keys, keys_capacity_words, ctrl, smem, nullptr, so, il, 8);
  } else {
    MIRGE_CUDA(ctx, cudaFuncSetAttribute(trim_kernel<64, false, 0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
    trim_kernel<64, false, 0, false><<<grid, TRIM_THREADS, smem, stream>>>(d_fastq, nbytes, d_line_start, n_records, win, d_key_off,
                                                                           d_keys, keys_capacity_words, ctrl, smem, nullptr, so, il, 8);
  }
  MIRGE_LAUNCH_CHECK(ctx, "trim_kernel");
  return MIRGE_OK;
}

extern "C" int mirge_trim_mode(mirge_ctx *ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return MIRGE_ERR_ARG;
  ctx->trim_mode = mode;
  return MIRGE_OK;
}
