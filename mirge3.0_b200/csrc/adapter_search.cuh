// adapter_search.cuh -- the per-read arithmetic of the trim kernels that restates cutadapt (3P; SURVEY Appendix A2-A4):
// the device view of the trim parameters, the literal full-column DP (locate), the bit-parallel search with traceback
// on demand (locate_fast) and the NextSeq / BWA quality scans.  Included by trim.cu; tests/test_adapter_search_host.py compiles the same text
// for the host (ADAPTER_SEARCH_HOST: one thread, CUDA intrinsics replaced by host_shims.h) and holds the two
// searches against each other and against the oracle on adversarial inputs.
#pragma once
#ifdef ADAPTER_SEARCH_HOST
#include "host_shims.h"
#else
#include "common.cuh"
#endif

#define TRIM_THREADS 128
#define OB 64  // origin bias inside the packed (origin, matches) word

struct DevAdapter {
  int where, m, min_overlap, indel_cost, wildcard_ref, k, effective_length;
  int link;  // mirge_adapter.link: 0 plain, (1 + index of the 3' half) | MIRGE_LINK_*_OPTIONAL (5' half of a linked pair), MIRGE_LINK_BACK_HALF
  uint64_t peq[5];  // bit i-1 set <=> adapter row i matches read class c (A,C,G,T,other)
  int n_counts[MIRGE_MAX_ADAPTER_LEN + 1];
  int max_err[MIRGE_MAX_ADAPTER_LEN + 1];
  int acc[MIRGE_MAX_ADAPTER_LEN + 1];  // 3' adapters: max errors of a candidate ending in adapter row i, -1 = never
  uint64_t a2;                         // 2-bit text of the adapter (row t at bits 2(t-1)); plain ACGT adapters <= 32 nt
  int wildcard_read;                   // --match-read-wildcards
  int general;  // placement other than plain 3' / 5', or read wildcards: searched by locate<MAXM, true>
};
struct DevParams {
  int n_mods, kind[MIRGE_MAX_MODS], a[MIRGE_MAX_MODS], b[MIRGE_MAX_MODS], c[MIRGE_MAX_MODS];
  int n_adapters, times, min_len, umi_mode, umi5, umi3, qia_len, slots;
  int w_mis, w_indel;  // what a mismatch / an indel adds to the merit a DP cell carries: 0, 0 (matches) or -1, -2 (cutadapt >= 4 score)
  DevAdapter ad[MIRGE_MAX_ADAPTERS];
};
#ifdef ADAPTER_SEARCH_HOST
static DevParams c_p;
#else
__constant__ DevParams c_p;
#endif

// Host side: the device view of the trim parameters.  Shared by mirge_set_trim_params (trim.cu) and the host harness of
// tests/test_adapter_search_host.py; returns MIRGE_OK or MIRGE_ERR_ARG with a message in err.
static int trim_slots_of(const mirge_trim_params *p) {
  return (p->umi_mode != MIRGE_UMI_QIAGEN && p->count_mode == MIRGE_COUNT_HEAD) ? p->n_mods : 1;
}

// largest cutoff / quality base of the NextSeq and quality modifiers (bases start at 1): what keeps the keys of the
// quality scans (quality_scan_max) inside an int
#define QUAL_PARAM_MAX 1000

#define FILL_FAIL(...)                  \
  do {                                  \
    snprintf(err, err_len, __VA_ARGS__); \
    return MIRGE_ERR_ARG;               \
  } while (0)

static int fill_dev_params(const mirge_trim_params *p, DevParams &d, int &maxm, int &fast_ok, char *err, size_t err_len) {
  if (p->n_mods < 0 || p->n_mods > MIRGE_MAX_MODS) FILL_FAIL("n_mods out of range");
  if (p->n_adapters < 0 || p->n_adapters > MIRGE_MAX_ADAPTERS) FILL_FAIL("n_adapters out of range");
  memset(&d, 0, sizeof(d));
  d.n_mods = p->n_mods;
  for (int i = 0; i < p->n_mods; ++i) {
    if (p->mod_kind[i] < MIRGE_MOD_NEXTSEQ || p->mod_kind[i] > MIRGE_MOD_CUT) FILL_FAIL("unknown modifier kind %d", p->mod_kind[i]);
    d.kind[i] = p->mod_kind[i];
    d.a[i] = p->mod_a[i];
    d.b[i] = p->mod_b[i];
    d.c[i] = p->mod_c[i];
    const bool nextseq = d.kind[i] == MIRGE_MOD_NEXTSEQ, quality = d.kind[i] == MIRGE_MOD_QUALITY;
    const int base = nextseq ? d.b[i] : d.c[i];
    if ((nextseq || quality) && (d.a[i] < 0 || d.a[i] > QUAL_PARAM_MAX || (quality && (d.b[i] < 0 || d.b[i] > QUAL_PARAM_MAX)) ||
                                 base < 1 || base > QUAL_PARAM_MAX))
      FILL_FAIL("%s trimming: quality cutoffs must lie in 0..%d and the quality base in 1..%d", nextseq ? "NextSeq" : "quality",
                QUAL_PARAM_MAX, QUAL_PARAM_MAX);
  }
  d.n_adapters = p->n_adapters;
  d.times = p->times;
  d.min_len = p->min_len;
  d.umi_mode = p->umi_mode;
  d.umi5 = p->umi5;
  d.umi3 = p->umi3;
  d.qia_len = p->qia_adapter_len;
  d.slots = trim_slots_of(p);
  if (p->compat != MIRGE_COMPAT_CUTADAPT23 && p->compat != MIRGE_COMPAT_CUTADAPT4) FILL_FAIL("unknown cutadapt compat %d", p->compat);
  d.w_mis = p->compat == MIRGE_COMPAT_CUTADAPT4 ? -1 : 0;
  d.w_indel = p->compat == MIRGE_COMPAT_CUTADAPT4 ? -2 : 0;
  if (p->umi_mode < MIRGE_UMI_NONE || p->umi_mode > MIRGE_UMI_QIAGEN) FILL_FAIL("bad umi_mode");
  if (p->umi_mode != MIRGE_UMI_NONE && (p->umi5 < 0 || p->umi3 < 0)) FILL_FAIL("negative UMI length");
  if (p->umi_mode == MIRGE_UMI_QIAGEN && p->n_adapters < 1) FILL_FAIL("qiagen UMI mode needs an adapter");
  maxm = 0;
  fast_ok = p->n_adapters <= MIRGE_FAST_ADAPTERS;  // (the bit-parallel kernels stage one match table per adapter in shared memory)
  for (int a = 0; a < p->n_adapters; ++a) {
    const mirge_adapter *s = &p->adapters[a];
    if (s->m < 1 || s->m > MIRGE_MAX_ADAPTER_LEN) FILL_FAIL("adapter %d length %d unsupported", a, s->m);
    if (s->where < MIRGE_WHERE_BACK || s->where > MIRGE_WHERE_FRONT_NOT_INTERNAL) FILL_FAIL("adapter %d: unknown type", a);
    DevAdapter *o = &d.ad[a];
    o->where = s->where; o->m = s->m; o->min_overlap = s->min_overlap; o->indel_cost = s->indel_cost;
    o->wildcard_ref = s->wildcard_ref; o->k = s->k; o->effective_length = s->effective_length;
    o->link = s->link;
    o->wildcard_read = s->wildcard_read ? 1 : 0;
    o->general = (s->where > MIRGE_WHERE_FRONT || s->wildcard_read) ? 1 : 0;
    if (s->link != 0 && s->link != MIRGE_LINK_BACK_HALF) {
      const int b = (s->link & MIRGE_LINK_INDEX_MASK) - 1;
      if ((s->link & ~(MIRGE_LINK_INDEX_MASK | MIRGE_LINK_FRONT_OPTIONAL | MIRGE_LINK_BACK_OPTIONAL)) || !MIRGE_WHERE_IS_FRONT(s->where) ||
          b <= a || b >= p->n_adapters || MIRGE_WHERE_IS_FRONT(p->adapters[b].where) || p->adapters[b].link != MIRGE_LINK_BACK_HALF)
        FILL_FAIL("adapter %d: a linked pair is a 5' adapter followed by its 3' half", a);
      if (p->umi_mode == MIRGE_UMI_QIAGEN) FILL_FAIL("linked adapters are not supported with qiagen UMIs");
    }
    if (s->link != 0) fast_ok = 0;  // linked pairs run on the full-DP kernel
    for (int c = 0; c < 4; ++c) {
      uint64_t bits = 0;
      for (int i = 0; i < s->m; ++i)
        if (s->mask[i] & (1 << c)) bits |= 1ull << i;
      o->peq[c] = bits;
    }
    o->peq[4] = 0;  // a read character outside ACGT never matches (match_read_wildcards=False)
    memcpy(o->n_counts, s->n_counts, sizeof(o->n_counts));
    memcpy(o->max_err, s->max_err, sizeof(o->max_err));
    for (int i = 0; i <= s->m; ++i) {
      const int eff = s->wildcard_ref ? i - s->n_counts[i] : i;
      o->acc[i] = (i >= s->min_overlap && i >= 1 && eff >= 0) ? s->max_err[eff] : -1;
    }
    o->a2 = 0;
    if (!s->wildcard_ref && s->m <= 32)
      for (int i = 0; i < s->m; ++i) {
        const uint64_t code = s->ascii[i] == 'A' ? 0 : s->ascii[i] == 'C' ? 1 : s->ascii[i] == 'G' ? 2 : 3;
        o->a2 |= code << (2 * i);
      }
    if (s->where != MIRGE_WHERE_BACK || s->wildcard_read || s->indel_cost != 1 || s->m > 32 || s->min_overlap < 1 || s->m + 2 * s->k + 3 > 48) fast_ok = 0;
    if (p->compat != MIRGE_COMPAT_CUTADAPT23) fast_ok = 0;  // the bit-parallel search is built on the matches objective
    if (s->m > maxm) maxm = s->m;
  }
  return MIRGE_OK;
}
#undef FILL_FAIL

// ------------------------------------------------------------------ adapter alignment -------

struct Match { int rstart, rstop, matches, errors; };

// cutadapt Aligner.locate: full-column DP in registers, one column per read base.  A cell's origin and merit -- its
// matches, or with MIRGE_COMPAT_CUTADAPT4 its score (match +1, mismatch -1, indel -2; biased by SB so that the field
// stays positive: a path has at most MIRGE_MAX_READ_LEN + MAXM steps of -2) -- travel in one word.
#define MS 12
#define MM 0xFFF
// GEN = false: plain 3' / 5' adapters (-a SEQ / -g SEQ), read characters outside ACGT never match.  GEN = true: every
// placement cutadapt's Where flags describe (anchored ^SEQ / SEQ$, non-internal XSEQ / SEQX: which ends of the alignment
// are free decides the first column, the columns that matter and the rows that are candidates) and --match-read-wildcards
// (the read's IUPAC characters match as sets).  With GEN = false every flag below is a constant of the two plain forms.
__host__ __device__ __forceinline__ uint32_t iupac_set_upper(uint32_t c) {
  c &= 0xDFu;  // upper case
  switch (c) {
    case 'A': return 1; case 'C': return 2; case 'G': return 4; case 'T': case 'U': return 8;
    case 'R': return 5; case 'Y': return 10; case 'S': return 6; case 'W': return 9; case 'K': return 12; case 'M': return 3;
    case 'B': return 14; case 'D': return 13; case 'H': return 11; case 'V': return 7; case 'N': return 15; default: return 0;
  }
}

template <int MAXM, bool GEN>
__device__ __noinline__ bool locate(const int a, const uint8_t *read, const int n, Match &out) {
  const DevAdapter &ad = c_p.ad[a];
  const int m = ad.m, ic = ad.indel_cost, k = ad.k;
  const bool back = ad.where == 0;
  const int w = ad.where;
  const bool start_in_ref = GEN ? (w == MIRGE_WHERE_FRONT || w == MIRGE_WHERE_FRONT_NOT_INTERNAL) : !back;
  const bool stop_in_ref = GEN ? (w == MIRGE_WHERE_BACK || w == MIRGE_WHERE_BACK_NOT_INTERNAL) : back;
  const bool start_in_query = GEN ? (w != MIRGE_WHERE_PREFIX && w != MIRGE_WHERE_FRONT_NOT_INTERNAL) : true;
  const bool stop_in_query = GEN ? (w != MIRGE_WHERE_SUFFIX && w != MIRGE_WHERE_BACK_NOT_INTERNAL) : true;
  const bool wild_read = GEN && ad.wildcard_read;
  // an anchored start cannot use more than m + k read bases, an anchored end only the last m + k (Aligner.locate)
  const int max_n = (!GEN || start_in_query) ? n : min(n, m + k);
  const int min_n = (!GEN || stop_in_query) ? 0 : max(0, n - m - k);
  const int w_mis = c_p.w_mis, w_indel = c_p.w_indel;
  const int SB = w_indel ? 2048 : 0;
  const uint64_t p0 = ad.peq[0], p1 = ad.peq[1], p2 = ad.peq[2], p3 = ad.peq[3];
  int cost[MAXM + 1], om[MAXM + 1];
#pragma unroll
  for (int i = 0; i <= MAXM; ++i) {
    if (!GEN) {
      cost[i] = back ? i * ic : 0;
      om[i] = (((back ? 0 : -i) + OB) << MS) + SB + (back ? i * w_indel : 0);
    } else {
      int c, o;  // the four cases of the first column (column min_n) in _align.pyx
      if (!start_in_ref && !start_in_query) { c = max(i, min_n) * ic; o = 0; }
      else if (start_in_ref && !start_in_query) { c = min_n * ic; o = min(0, min_n - i); }
      else if (!start_in_ref && start_in_query) { c = i * ic; o = max(0, min_n - i); }
      else { c = min(i, min_n) * ic; o = min_n - i; }
      cost[i] = c;
      om[i] = ((o + OB) << MS) + SB + (start_in_ref ? 0 : i * w_indel);
    }
  }
  int best_cost = m + n, best_om = (OB << MS) + (w_indel ? 0 : SB), best_ref_stop = m, best_query_stop = n;
  bool stopped = false;
  for (int j = min_n + 1; j <= max_n; ++j) {
    uint64_t eq;
    if (wild_read) {
      const uint32_t rs = iupac_set_upper(read[j - 1]);
      eq = ((rs & 1u) ? p0 : 0ull) | ((rs & 2u) ? p1 : 0ull) | ((rs & 4u) ? p2 : 0ull) | ((rs & 8u) ? p3 : 0ull);
    } else {
      const uint32_t rc = base_code_upper(read[j - 1]);
      eq = rc == 0 ? p0 : rc == 1 ? p1 : rc == 2 ? p2 : rc == 3 ? p3 : 0ull;
    }
    int dc = cost[0], dom = om[0];
    if (!GEN || start_in_query) om[0] = ((j + OB) << MS) + SB;
    else { cost[0] = j * ic; om[0] = (OB << MS) + SB + j * w_indel; }
    int cm = 0, omm = 0;
#pragma unroll
    for (int i = 1; i <= MAXM; ++i) {
      if (i <= m) {
        int c, o;
        if ((eq >> (i - 1)) & 1ull) {
          c = dc; o = dom + 1;
        } else {
          const int cd = dc + 1, cdel = cost[i] + ic, cins = cost[i - 1] + ic;
          if (cd <= cdel && cd <= cins) { c = cd; o = dom + w_mis; }
          else if (cins <= cdel) { c = cins; o = om[i - 1] + w_indel; }
          else { c = cdel; o = om[i] + w_indel; }
        }
        dc = cost[i]; dom = om[i];
        cost[i] = c; om[i] = o;
        if (i == m) { cm = c; omm = o; }
      }
    }
    if (cm <= k && (!GEN || stop_in_query)) {
      const int origin = (omm >> MS) - OB, mt = omm & MM;
      const int length = m + min(origin, 0);
      int eff = length;
      if (ad.wildcard_ref) eff = (length < m) ? length - (ad.n_counts[m] - ad.n_counts[m - length]) : ad.effective_length;
      const int bm = best_om & MM;
      if (length >= ad.min_overlap && cm <= ad.max_err[eff] && (mt > bm || (mt == bm && cm < best_cost))) {
        best_cost = cm; best_om = omm; best_ref_stop = m; best_query_stop = j;
        if (cm == 0 && mt - SB == m) { stopped = true; break; }
      }
    }
  }
  if (!stopped && (!GEN || max_n == n)) {
    const int first_i = stop_in_ref ? 0 : m;
#pragma unroll
    for (int i = 0; i <= MAXM; ++i) {
      if (i >= first_i && i <= m) {
        const int origin = (om[i] >> MS) - OB, mt = om[i] & MM, c = cost[i];
        const int length = i + min(origin, 0);
        int eff = length;
        if (ad.wildcard_ref) {
          if (length < m) { const int ref_start = origin < 0 ? -origin : 0; eff = length - (ad.n_counts[i] - ad.n_counts[ref_start]); }
          else eff = ad.effective_length;
        }
        const int bm = best_om & MM;
        if (length >= ad.min_overlap && eff >= 0 && c <= ad.max_err[eff] && (mt > bm || (mt == bm && c < best_cost))) {
          best_cost = c; best_om = om[i]; best_ref_stop = i; best_query_stop = n;
        }
      }
    }
  }
  (void)best_ref_stop;
  if (best_cost == m + n) return false;
  const int origin = (best_om >> MS) - OB;
  out.rstart = origin >= 0 ? origin : 0;
  out.rstop = best_query_stop;
  out.matches = (best_om & MM) - SB;
  out.errors = best_cost;
  return true;
}

// Adapter.match_to's shortcut: an adapter without wildcards is first looked for literally (str.find on the upper-cased
// read).  For the alignment above that changes nothing -- the leftmost literal occurrence is where the DP stops -- except
// with --match-read-wildcards, where the DP also accepts occurrences through the read's N and would find one of those
// first; cutadapt returns the literal one.  Shift-and over the read bytes (adapter rows as bits, <= 64).
__device__ __noinline__ bool find_literal(const int a, const uint8_t *read, const int n, Match &out) {
  const DevAdapter &ad = c_p.ad[a];
  const int m = ad.m;
  const uint64_t top = 1ull << (m - 1);
  uint64_t state = 0;
  for (int j = 0; j < n; ++j) {
    const uint32_t rc = base_code_upper(read[j]);
    state = ((state << 1) | 1ull) & (rc < 4u ? ad.peq[rc] : 0ull);
    if (state & top) {
      out.rstart = j + 1 - m;
      out.rstop = j + 1;
      out.matches = m;
      out.errors = 0;
      return true;
    }
  }
  return false;
}

// the search of one adapter on the full-DP path: the plain forms keep their own instantiation
template <int MAXM>
__device__ __forceinline__ bool locate_any(const int a, const uint8_t *read, const int n, Match &out) {
  const DevAdapter &ad = c_p.ad[a];
  if (!ad.general) return locate<MAXM, false>(a, read, n, out);
  if (ad.wildcard_read && !ad.wildcard_ref && ad.where <= MIRGE_WHERE_FRONT && find_literal(a, read, n, out)) return true;
  return locate<MAXM, true>(a, read, n, out);
}

// ------------------------------------------------------------------ bit-parallel locate ------
// Same result as locate() for 3' adapters with unit indel cost and m <= 32, at ~15 instructions per
// read base instead of ~15 per DP cell:
//   1. Myers/Hyyro bit-vector recurrence gives the exact DP cost column (vertical deltas VP/VN) for
//      every read position; the cost of adapter row m is tracked incrementally.  Nothing is stored.
//   2. cutadapt's candidates are the row-m cell of every column and all rows of the last column; their
//      costs come from (1).  A candidate's (origin, matches) are those of the path cutadapt's
//      tie-breaking (mismatch, then insertion, then deletion) propagates into that cell; the path is
//      recovered by a traceback that needs only DP *costs* of neighbouring cells.  Those are recomputed
//      on demand for the last m + 2k + 2 columns before the candidate with a fresh-start Myers pass into
//      a thread-local buffer: a path with <= k errors into row i spans <= i + k columns, and every
//      neighbour whose cost can tie has an optimal path starting inside that window, so the costs the
//      rule compares are exact (larger values only lose).  cost == 0 cells are pure diagonals.
//   3. The winner is the maximum of (matches, -cost, -scan order) as in Aligner.locate, so candidates
//      may be evaluated in any order.  Cheap exact pruning keeps tracebacks rare: a row-m candidate
//      entered by a deletion is dominated by its left neighbour; one entered by an insertion is dominated
//      when the next column's cell is a character match; a candidate whose first step is not a match has
//      at most row-1 matches; candidates are tried best-first and skipped when they cannot win.
//   All tracebacks run after the column loop, so the lanes of a warp execute them together.
#define RB 48  // recompute window capacity in columns (m + 2k + 3 <= RB is checked on the host)

struct FastCtx {
  const uint32_t *s_eq;  // [n_adapters][256]: bit i-1 set <=> adapter row i matches this read byte
  const uint32_t *ps;    // this thread's 2-bit packed read (16 bases per word), stride TRIM_THREADS words
  bool jump_ok;          // ps is valid and the read is pure "ACGT": match runs can be skipped with bit tricks
  int rbase;             // offset of the window being searched inside the read
};

// How the adapter search sees the read window: eq(eqt, j) = match mask of window base j (bit i-1 set <=> adapter
// row i matches it).  ByteRead: ASCII bytes (shared-memory staging or the global stream), eqt indexed by byte.
// PackedRead: the 2-bit packed pure-ACGT read of this thread (row stride TRIM_THREADS words), eqt indexed by the
// 2-bit code -- used by the split pipeline, whose search kernel never touches the FASTQ bytes again.
struct ByteRead {
  const uint8_t *p;
  __device__ __forceinline__ uint32_t eq(const uint32_t *eqt, int j) const { return eqt[p[j]]; }
  // sequential access for the column loop
  struct Cursor {
    const uint8_t *q;
    __device__ __forceinline__ uint32_t next(const uint32_t *eqt) { return eqt[*q++]; }
  };
  __device__ __forceinline__ Cursor cursor() const { return Cursor{p}; }
};
struct PackedRead {
  const uint32_t *ps;
  int base;  // offset of the window inside the read
  __device__ __forceinline__ uint32_t eq(const uint32_t *eqt, int j) const {
    const int a = base + j;
    return eqt[(ps[(a >> 4) * TRIM_THREADS] >> (2 * (a & 15))) & 3u];
  }
  // sequential access for the column loop: the current 16-base word lives in a register and is shifted by one
  // base per column; a new word is fetched every 16 columns
  struct Cursor {
    const uint32_t *row;
    uint32_t w;
    int left;
    __device__ __forceinline__ uint32_t next(const uint32_t *eqt) {
      if (left == 0) {
        row += TRIM_THREADS;
        w = *row;
        left = 16;
      }
      const uint32_t code = w & 3u;
      w >>= 2;
      --left;
      return eqt[code];
    }
  };
  __device__ __forceinline__ Cursor cursor() const {
    const uint32_t *row = ps + (base >> 4) * TRIM_THREADS;
    const int sh = base & 15;
    return Cursor{row, *row >> (2 * sh), 16 - sh};
  }
};

struct ColBuf {
  uint32_t vp[RB], vn[RB];
  int j0;  // entry t holds column j0 + t
};

__device__ __forceinline__ int cell_cost(uint32_t vp, uint32_t vn, int r) {
  const uint32_t mask = r >= 32 ? 0xFFFFFFFFu : ((1u << r) - 1u);
  return __popc(vp & mask) - __popc(vn & mask);
}

#define MYERS_STEP(eq, vp, vn, hp_out, hn_out)                    \
  {                                                               \
    const uint32_t xv_ = (eq) | (vn);                             \
    const uint32_t xh_ = ((((eq) & (vp)) + (vp)) ^ (vp)) | (eq);  \
    uint32_t hp_ = (vn) | ~(xh_ | (vp));                          \
    uint32_t hn_ = (vp) & xh_;                                    \
    hp_out = hp_;                                                 \
    hn_out = hn_;                                                 \
    hp_ <<= 1;                                                    \
    hn_ <<= 1;                                                    \
    (vp) = hn_ | ~(xv_ | hp_);                                    \
    (vn) = hp_ & xv_;                                             \
  }

// cost columns jc - span .. jc recomputed with a fresh start (exact where it matters, see above)
template <class RV>
__device__ __noinline__ void recompute(const uint32_t *eqt, const RV read, int jc, int span, ColBuf &cb) {
  const int j0 = max(0, jc - span);
  uint32_t vp = 0xFFFFFFFFu, vn = 0u;
  cb.j0 = j0;
  cb.vp[0] = vp;
  cb.vn[0] = vn;
  int t = 1;
  for (int j = j0 + 1; j <= jc; ++j, ++t) {
    const uint32_t eq = read.eq(eqt, j - 1);
    uint32_t hp, hn;
    MYERS_STEP(eq, vp, vn, hp, hn)
    cb.vp[t] = vp;
    cb.vn[t] = vn;
  }
}

// 64 bits = 32 bases of the packed read starting at base `a0` (zero beyond the packed words)
__device__ __forceinline__ uint64_t read_window(const uint32_t *ps, int a0) {
  const int wi = a0 >> 4, sh = 2 * (a0 & 15);
  const uint32_t w0 = ps[wi * TRIM_THREADS], w1 = ps[(wi + 1) * TRIM_THREADS], w2 = ps[(wi + 2) * TRIM_THREADS];
  const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
  return ((uint64_t)hi << 32) | lo;
}

// (matches, origin) cutadapt's DP holds in cell (i, j) whose cost is c > 0, from the cost columns in cb.
// jump: adapter without wildcards and a pure-ACGT packed read -- the run of matches up a diagonal is skipped
// with one XOR + count-leading-zeros instead of one step per cell.
template <class RV>
__device__ __noinline__ void traceback(const int a, const uint32_t *eqt, const RV read, const FastCtx &fc, const ColBuf &cb,
                                          int i, int j, int c, int &matches, int &origin) {
  const bool jump = fc.jump_ok && !c_p.ad[a].wildcard_ref;
  const uint64_t a2 = c_p.ad[a].a2;
  int r = i, col = j, cost = c, nonmatch = 0;
  while (r > 0 && cost > 0) {
    if (col == 0) {  // initial column: cost r, origin 0, no further matches
      nonmatch += r;
      r = 0;
      break;
    }
    const int delta = col - r;
    if (jump && delta >= 0) {
      // rows t = 1..r of this diagonal face read bases delta + t - 1 (all in columns >= 1)
      uint64_t x = a2 ^ read_window(fc.ps, fc.rbase + delta);
      x = (x | (x >> 1)) & 0x5555555555555555ull;
      if (r < 32) x &= (1ull << (2 * r)) - 1ull;
      if (x == 0) {  // cannot happen while cost > 0 (an all-match diagonal has cost 0); kept for safety
        col -= r;
        r = 0;
        break;
      }
      const int t = (64 - __clzll((long long)x) + 1) >> 1;  // highest mismatching row <= r
      col -= r - t;
      r = t;
    } else if ((read.eq(eqt, col - 1) >> (r - 1)) & 1u) {  // equal characters: diagonal, cost unchanged
      --r; --col;
      continue;
    }
    const int t0 = col - cb.j0;  // >= 1 by the window bound
    const uint32_t vp0 = cb.vp[t0], vn0 = cb.vn[t0], vp1 = cb.vp[t0 - 1], vn1 = cb.vn[t0 - 1];
    const int cd = cell_cost(vp1, vn1, r - 1) + 1, cdel = cell_cost(vp1, vn1, r) + 1, cins = cell_cost(vp0, vn0, r - 1) + 1;
    if (cd <= cdel && cd <= cins) { --r; --col; ++nonmatch; cost = cd - 1; }
    else if (cins <= cdel) { --r; ++nonmatch; cost = cins - 1; }
    else { --col; cost = cdel - 1; }
  }
  origin = col - r;  // r > 0 here means cost == 0: r more diagonal matches
  matches = i - nonmatch;
}

// Cost-1 cells need no cost columns: slide up the diagonal to the only error and decide its kind by asking
// which neighbour has cost 0 -- a cost-0 cell (a, b) simply means adapter[0:a] == read[b-a:b], one packed
// compare.  cutadapt's rule picks mismatch if (t-1, col-1) is such a cell, else insertion if (t-1, col) is,
// else deletion.  Needs the packed pure-ACGT read and a plain adapter; returns false when it does not apply.
__device__ __forceinline__ bool traceback_cost1(const int a, const FastCtx &fc, int i, int j, int &matches, int &origin) {
  const int delta = j - i;
  if (!fc.jump_ok || c_p.ad[a].wildcard_ref || delta < 0) return false;
  const uint64_t a2 = c_p.ad[a].a2;
  const uint64_t even = 0x5555555555555555ull;
  uint64_t x = a2 ^ read_window(fc.ps, fc.rbase + delta);
  x = (x | (x >> 1)) & even;
  if (i < 32) x &= (1ull << (2 * i)) - 1ull;
  if (x == 0) return false;  // not a cost-1 cell of this diagonal (cannot happen); use the general path
  const int t = (64 - __clzll((long long)x) + 1) >> 1;  // row of the error
  const uint64_t below = t - 1 >= 32 ? ~0ull : ((1ull << (2 * (t - 1))) - 1ull);  // rows 1..t-1
  if ((x & below) == 0) {  // mismatch: rows above continue cleanly on the same diagonal
    matches = i - 1;
    origin = delta;
    return true;
  }
  uint64_t y = a2 ^ read_window(fc.ps, fc.rbase + delta + 1);
  y = (y | (y >> 1)) & even & below;
  if (y == 0) {  // insertion: adapter[0:t-1] ends at the same read base
    matches = i - 1;
    origin = delta + 1;
    return true;
  }
  if (delta < 1) return false;
  const uint64_t upto = t >= 32 ? ~0ull : ((1ull << (2 * t)) - 1ull);  // rows 1..t
  uint64_t z = a2 ^ read_window(fc.ps, fc.rbase + delta - 1);
  z = (z | (z >> 1)) & even & upto;
  if (z != 0) return false;  // inconsistent with cost 1: let the general path decide
  matches = i;  // deletion: a read base is skipped, every adapter row matches
  origin = delta - 1;
  return true;
}

// A cell (i, j) of cost c reaches i matches only if every error is a deletion; that path leaves row 0 at
// column j - i - c with a match, so adapter[0] must equal that read base (cheap necessary condition).
template <class RV>
__device__ __forceinline__ bool all_deletions_possible(const uint32_t *eqt, const RV read, int i, int j, int c) {
  const int o = j - i - c;
  return o >= 0 && (read.eq(eqt, o) & 1u);
}

// candidate with at most `u` matches, cost c, scan index idx can still beat the best so far
#define MAY_WIN(u, c, idx) (!have || (u) > b_m || ((u) == b_m && ((c) < b_c || ((c) == b_c && (idx) < b_idx))))
#define TAKE_IF_BETTER(mt, c, org, idx)                                                      \
  if (!have || (mt) > b_m || ((mt) == b_m && ((c) < b_c || ((c) == b_c && (idx) < b_idx)))) { \
    have = true; b_m = (mt); b_c = (c); b_o = (org); b_idx = (idx);                          \
  }
// queued row-m candidate: column | cost << 16 | (first step is a match) << 24 | insertion-chain length << 25
#define Q_COL(v) ((int)((v)&0xFFFFu))
#define Q_COST(v) ((int)(((v) >> 16) & 0xFFu))
#define Q_UB(v, m) ((((v) >> 24) & 1u) ? (m) : (m)-1)
#define Q_CHAIN(v) ((int)((v) >> 25))
// Cells of one column that cutadapt's rule enters by an insertion, for all rows at once: characters differ, the
// vertical delta is +1 (cins attains the cell's cost) and the diagonal predecessor does not (its cost is the
// cell's cost, i.e. the horizontal delta one row up is -1).  A run of t such cells ending in row i means the
// traceback of (i, j) walks straight up to (i - t, j): same matches and origin, t errors fewer -- which settles
// most candidates whose extra cost is adapter overhang without any cost column.
#define INS_MASK(eq, vp, hn) (~(eq) & (vp) & ((hn) << 1))
#define CHAIN_LEN(ins, i) (__clz((int)~((ins) << (32 - (i)))))

// DEFER: as soon as a candidate would need cost columns (recompute + general traceback) the search gives up
// with 2 and the read is queued for a later stage (stage 3 of the split pipeline, or the leftover pass of the
// unsplit path), which runs this function without DEFER on a compacted list, so that the rare expensive path
// executes with full warps.
// Returns 0 = no match, 1 = match in `out`, 2 = deferred.
template <bool DEFER, class RV>
__device__ __forceinline__ int locate_fast(const int a, const RV read, const int n, const FastCtx &fc, Match &out) {
  const unsigned lanes = __activemask();  // lanes searching together; re-converged after the divergent loops
  const DevAdapter &ad = c_p.ad[a];
  const int m = ad.m;
  const int span = m + 2 * ad.k + 2;
  const uint32_t *eqt = fc.s_eq + a * 256;
  const uint32_t top = 1u << (m - 1);
  const int acc_m = ad.acc[m];
  uint32_t vp = 0xFFFFFFFFu, vn = 0u, eq = 0;
  int score = m;
  bool have = false;
  int b_m = 0, b_c = 0, b_o = 0, b_idx = 0;
  bool stopped = false;
  ColBuf cb;
  // row-m candidates wait here until the column loop is over (0 = empty slot)
  uint32_t q0 = 0, q1 = 0, q2 = 0, q3 = 0;
  // a new candidate waits one column: the next column may prove it dominated
  bool pend = false, pend_ins = false, need_slow = false;
  uint32_t pend_v = 0;

// trace the queued candidates best-first (lowest cost, then leftmost), skipping those that cannot win
#define FLUSH_QUEUE()                                                                            \
  for (int it_ = 0; it_ < 4; ++it_) {                                                            \
    uint32_t v_ = 0;                                                                             \
    int which_ = -1;                                                                             \
    if (q0 && (!v_ || Q_COST(q0) < Q_COST(v_))) { v_ = q0; which_ = 0; }                         \
    if (q1 && (!v_ || Q_COST(q1) < Q_COST(v_))) { v_ = q1; which_ = 1; }                         \
    if (q2 && (!v_ || Q_COST(q2) < Q_COST(v_))) { v_ = q2; which_ = 2; }                         \
    if (q3 && (!v_ || Q_COST(q3) < Q_COST(v_))) { v_ = q3; which_ = 3; }                         \
    if (which_ < 0) break;                                                                       \
    if (which_ == 0) q0 = 0; else if (which_ == 1) q1 = 0; else if (which_ == 2) q2 = 0; else q3 = 0; \
    const int jc_ = Q_COL(v_), cc_ = Q_COST(v_), t_ = Q_CHAIN(v_);                               \
    const int ir_ = m - t_, cr_ = cc_ - t_; /* the cell the insertion chain leads to */          \
    int ub_ = t_ ? ir_ : Q_UB(v_, m);                                                            \
    if (!t_ && ub_ == m && !all_deletions_possible(eqt, read, m, jc_, cc_)) ub_ = m - 1;        \
    if (MAY_WIN(ub_, cc_, jc_)) {                                                                \
      int mt_, org_;                                                                             \
      if (cr_ == 0) {                                                                            \
        mt_ = ir_; org_ = jc_ - ir_;                                                             \
      } else if (!(cr_ == 1 && traceback_cost1(a, fc, ir_, jc_, mt_, org_))) {                   \
        if (DEFER) { need_slow = true; break; }                                                  \
        recompute(eqt, read, jc_, span, cb);                                                     \
        traceback(a, eqt, read, fc, cb, ir_, jc_, cr_, mt_, org_);                               \
      }                                                                                          \
      TAKE_IF_BETTER(mt_, cc_, org_, jc_)                                                        \
    }                                                                                            \
  }

  uint32_t hp = 0, hn = 0;  // horizontal deltas of the column just computed
  auto cur = read.cursor();
  for (int j = 1; j <= n; ++j) {
    eq = cur.next(eqt);
    MYERS_STEP(eq, vp, vn, hp, hn)
    score += (hp & top) ? 1 : 0;
    score -= (hn & top) ? 1 : 0;
    if (pend) {
      // Rule 2: the candidate (m, j-1) was entered by an insertion from (m-1, j-1) and cell (m, j) is a
      // character match from that same cell: (m, j) has one more match and one error less, is itself a
      // candidate (row m of column j, or of the last column) and therefore beats (m, j-1).
      if (!(pend_ins && (eq & top))) {
        if (!q0) q0 = pend_v;
        else if (!q1) q1 = pend_v;
        else if (!q2) q2 = pend_v;
        else if (!q3) q3 = pend_v;
        else {  // queue full (low-complexity read): resolve what is queued, then go on
          FLUSH_QUEUE()
          if (DEFER && need_slow) break;
          q0 = pend_v;
        }
      }
      pend = false;
    }
    if (score <= acc_m && j < n) {  // row-m candidate (column n is handled with the last column)
      if (score == 0) {              // exact full adapter: cutadapt stops here
        have = true; b_m = m; b_c = 0; b_o = j - m; b_idx = j;
        stopped = true;
        break;
      }
      // first traceback step of cell (m, j) from this column's step masks (see the last-column scan below):
      // mismatch <=> vertical delta + horizontal delta one row up == 1; else insertion <=> vertical delta +1
      bool is_del = false, is_ins = false;
      const bool is_match = (eq & top) != 0u;
      if (!is_match) {
        const uint32_t hps = hp << 1, hns = hn << 1;
        const bool mis = (((vp & ~hps & ~hns) | (~vp & ~vn & hps)) & top) != 0u;
        if (!mis) {
          if (vp & top) is_ins = true;
          else is_del = true;
        }
      }
      // Rule 1: entered by a deletion from (m, j-1): same matches and origin as that cell, one error
      // more; (m, j-1) is an accepted earlier candidate, so (m, j) can never win.
      if (!is_del) {
        pend = true;
        pend_ins = is_ins;
        // insertion chain: row m by the rule above, the rows below it from the column's insertion mask
        const uint32_t chain = is_ins ? 1u + (uint32_t)CHAIN_LEN(INS_MASK(eq, vp, hn), m - 1) : 0u;
        pend_v = (uint32_t)j | ((uint32_t)score << 16) | (is_match ? (1u << 24) : 0u) | (chain << 25);
      }
    }
  }
  __syncwarp(lanes);
  const unsigned scan_lanes = __ballot_sync(lanes, !stopped && !need_slow);
  if (!stopped && !need_slow) {
    // last column: rows with cost 0 are pure diagonals; the others wait in rowmask / rowub.  First traceback step
    // of every row at once: entered by an insertion (ins), by a mismatch (mis: the diagonal predecessor attains
    // cost - 1, i.e. vertical delta + horizontal delta one row up == 1), else match or deletion.
    uint32_t rowmask = 0, rowub = 0;  // rowub bit: first step is a match or a deletion (up to i matches), else i - 1
    const uint32_t hps = hp << 1, hns = hn << 1;
    const uint32_t ins = n >= 1 ? INS_MASK(eq, vp, hn) : 0u;
    const uint32_t mis = n >= 1 ? (~eq & ((vp & ~hps & ~hns) | (~vp & ~vn & hps))) : 0u;
    int c = 0;  // D[i][n]
    for (int i = 1; i <= m; ++i) {
      const uint32_t bit = 1u << (i - 1);
      c += (int)((vp >> (i - 1)) & 1u) - (int)((vn >> (i - 1)) & 1u);
      if (c > ad.acc[i]) continue;
      if (c == 0) {
        const int idx = (i == m) ? n : n + 1 + i;  // row m of column n precedes the last-column scan
        TAKE_IF_BETTER(i, 0, n - i, idx)
      } else if (ins & bit) {
        // Rule 3: a chain of t insertions from (i - t, n): same matches and origin as that cell, t errors more;
        // when (i - t, n) is an accepted candidate of this column, (i, n) can never win.
        const int t = CHAIN_LEN(ins, i);
        if (ad.acc[i - t] >= c - t) continue;
        rowmask |= bit;
      } else {
        rowmask |= bit;
        if ((eq & bit) || !(mis & bit)) rowub |= bit;
      }
    }
    __syncwarp(scan_lanes);
    FLUSH_QUEUE()
    bool have_cols = false;
    while (rowmask) {  // descending rows: the first traceback usually prunes the rest
      const int i = 32 - __clz(rowmask);
      const uint32_t bit = 1u << (i - 1);
      rowmask &= ~bit;
      const int ci = cell_cost(vp, vn, i);
      const int idx = (i == m) ? n : n + 1 + i;
      const int t = (ins & bit) ? CHAIN_LEN(ins, i) : 0;
      const int ir = i - t, cr = ci - t;  // the cell the insertion chain leads to
      int ub = t ? ir : ((rowub & bit) ? i : i - 1);
      if (!t && ub == i && !all_deletions_possible(eqt, read, i, n, ci)) ub = i - 1;
      if (MAY_WIN(ub, ci, idx)) {
        int mt, org;
        if (cr == 0) {
          mt = ir;
          org = n - ir;
        } else if (!(cr == 1 && traceback_cost1(a, fc, ir, n, mt, org))) {
          if (DEFER) { need_slow = true; break; }
          if (!have_cols) {
            recompute(eqt, read, n, span, cb);
            have_cols = true;
          }
          traceback(a, eqt, read, fc, cb, ir, n, cr, mt, org);
        }
        TAKE_IF_BETTER(mt, ci, org, idx)
      }
    }
  }
  if (DEFER && need_slow) return 2;
  if (!have) return 0;
  out.rstart = b_o;
  out.rstop = b_idx <= n ? b_idx : n;
  out.matches = b_m;
  out.errors = b_c;
  return 1;
}

// ------------------------------------------------------------------ quality trimming --------

// cutadapt's scans (qualtrim.pyx) add cutoff - (qual[i] - base) to a sum s, stop at the first s < 0 and keep the
// position of the first strict maximum of s in scan order.  Here every position carries one key k = s * 1024 + x, where
// x (0..1023) falls by one per byte in scan order: x = i scanning down from len, x = 1022 - i scanning up (x = 1023
// stands for "before position 0").  Then the first strict maximum is the maximum key, s < 0 exactly when k < 0, and a
// byte step is k += 1024 * (cutoff + base - qual[i]) - 1.  fill_dev_params bounds cutoff and base to
// 0..QUAL_PARAM_MAX (base >= 1), so |s| <= 512 * 2000 and every key fits an int.
//
// quality_scan_max runs the scan four bytes per step: one aligned 32-bit load per line (funnel-shifted to the group's
// first byte), the four keys of the group, one sign test for all four; in the group that holds the first negative sum
// only the keys before it count.  The last len % 4 bytes are scanned byte by byte.  Memory: the word loop reads only aligned words that hold a
// byte of [0, len) of seq / qual, so it never leaves the 16-byte segments the line occupies -- inside the staging
// buffer of a CTA, and inside the stream for the kernels that read it from global memory.
static_assert(MIRGE_MAX_READ_LEN <= 1022, "quality scan keys keep the position in 10 bits");

// 0xFF in every byte of x whose bit 7 is set, 0x00 in the others (PRMT's sign-replicating byte select)
__device__ __forceinline__ uint32_t byte_msb_mask(uint32_t x) {
#ifdef ADAPTER_SEARCH_HOST
  return ((x >> 7) & 0x01010101u) * 0xFFu;
#else
  uint32_t r;
  asm("prmt.b32 %0, %1, 0, 0xBA98;" : "=r"(r) : "r"(x));
  return r;
#endif
}

// qual[i] << 10 of the byte b (0..3) of a group word
__device__ __forceinline__ int qbyte_k(uint32_t w, int b) { return (int)(((w >> (8 * b)) & 0xFFu) << 10); }

// Largest key of the scan of qual[0, len) (DOWN: from len - 1 to 0, else from 0 to len - 1) that starts at key k.
// cb = cutoff + base.  NEXTSEQ: positions where seq holds 'G' add 1 to s (qualtrim's q = cutoff - 1).
template <bool DOWN, bool NEXTSEQ>
__device__ __forceinline__ int quality_scan_max(const uint8_t *qual, const uint8_t *seq, const int len, const int cb, int k) {
  const int step = cb * 1024 - 1;
  int best = k, n = len;  // bytes not scanned yet
  if (n >= 4) {
    // a G byte of seq turns into the quality byte cb - 1 (step 1024 - 1).  Clamped to a byte: when cb - 1 > 255 every
    // byte adds at least 2 to s, G or not, so the scan runs to the end and its result does not depend on the value.
    const uint32_t g4 = 0x01010101u * (uint32_t)min(cb - 1, 255);
    // Each step loads the word that holds the group's last byte in scan order (DOWN: byte n - 4, UP: byte len - n + 3);
    // the word the step before loaded holds its first byte.  The group is funnel_r(loaded, before) scanning down and
    // funnel_l(before, loaded) scanning up; when the group is word-aligned only the loaded word is used.
    const int aq = (int)((uintptr_t)qual & 3u), as = NEXTSEQ ? (int)((uintptr_t)seq & 3u) : 0;
    const uint32_t shq = DOWN ? 8u * (uint32_t)((len + aq) & 3) : 32u - 8u * (uint32_t)aq;
    const uint32_t shs = DOWN ? 8u * (uint32_t)((len + as) & 3) : 32u - 8u * (uint32_t)as;
    const uint32_t *qw = (const uint32_t *)(qual - aq), *sw = nullptr;
    uint32_t q_prev = DOWN ? qw[(len - 1 + aq) >> 2] : qw[0], s_prev = 0;
    qw += DOWN ? (len - 4 + aq) >> 2 : (3 + aq) >> 2;
    if (NEXTSEQ) {
      sw = (const uint32_t *)(seq - as);
      s_prev = DOWN ? sw[(len - 1 + as) >> 2] : sw[0];
      sw += DOWN ? (len - 4 + as) >> 2 : (3 + as) >> 2;
    }
#pragma unroll 2
    for (; n >= 4; n -= 4) {
      const uint32_t qn = *qw, q = DOWN ? __funnelshift_r(qn, q_prev, shq) : __funnelshift_l(q_prev, qn, shq);
      qw += DOWN ? -1 : 1;
      q_prev = qn;
      uint32_t w = q;
      if (NEXTSEQ) {
        const uint32_t sn = *sw, s = DOWN ? __funnelshift_r(sn, s_prev, shs) : __funnelshift_l(s_prev, sn, shs);
        sw += DOWN ? -1 : 1;
        s_prev = sn;
        const uint32_t z = s ^ 0x47474747u;  // zero bytes: 'G'
        const uint32_t not_g = byte_msb_mask(((z & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | z);
        w = (q & not_g) | (g4 & ~not_g);
      }
      const int k0 = k + step - qbyte_k(w, DOWN ? 3 : 0);
      const int k1 = k0 + step - qbyte_k(w, DOWN ? 2 : 1);
      const int k2 = k1 + step - qbyte_k(w, DOWN ? 1 : 2);
      const int k3 = k2 + step - qbyte_k(w, DOWN ? 0 : 3);
      if ((k0 | k1 | k2 | k3) < 0) {  // s < 0 in this group: the keys before the first negative one count, then the scan ends
        if (k0 >= 0) {
          best = max(best, k0);
          if (k1 >= 0) {
            best = max(best, k1);
            if (k2 >= 0) best = max(best, k2);
          }
        }
        return best;
      }
      best = max(best, max(max(k0, k1), max(k2, k3)));
      k = k3;
    }
  }
#pragma unroll 1
  for (; n > 0; --n) {  // the last len % 4 bytes (all of them when len < 4)
    const int i = DOWN ? n - 1 : len - n;
    const int d = (NEXTSEQ && seq[i] == 'G') ? 1 : cb - (int)qual[i];
    k += d * 1024 - 1;
    if (k < 0) break;
    best = max(best, k);
  }
  return best;
}

__device__ __forceinline__ int nextseq_trim_index(const uint8_t *seq, const uint8_t *qual, int len, int cutoff, int base) {
  return quality_scan_max<true, true>(qual, seq, len, cutoff + base, len) & 1023;
}

__device__ __forceinline__ void quality_trim_index(const uint8_t *qual, int len, int q5, int q3, int base, int &start, int &stop) {
  start = 1023 - (quality_scan_max<false, false>(qual, nullptr, len, q5 + base, 1023) & 1023);
  stop = quality_scan_max<true, false>(qual, nullptr, len, q3 + base, len) & 1023;
  if (start >= stop) { start = 0; stop = 0; }
}

// ------------------------------------------------------------------ modifiers ---------------

// AdapterCutter._best_match: most matches, then fewer errors, first adapter wins ties.
// returns the index of the winning adapter, -1 for none, -2 when the search was deferred (DEFER only)
template <int MAXM, bool FAST, bool DEFER>
__device__ __noinline__ int best_match(const uint8_t *read, int n, Match &best, const FastCtx &fc) {
  int which = -1;
  for (int a = 0; a < c_p.n_adapters; ++a) {
    Match mt;
    const int link = c_p.ad[a].link;
    if (link == MIRGE_LINK_BACK_HALF) continue;  // searched through its 5' half only
    if (FAST) {
      const int rc = locate_fast<DEFER>(a, ByteRead{read}, n, fc, mt);
      if (rc == 2) return -2;
      if (rc == 0) continue;
    } else if (link != 0) {
      // cutadapt LinkedAdapter.match_to: the 3' half is searched in what the 5' match leaves; a missing half ends the
      // search unless it is optional (-g "A...B": both required; -a "A...B": a half is required when it is anchored),
      // and a pair without its 5' half needs its 3' half; matches and errors of the pair are the sums.  The Match of a
      // pair carries the two cut points: rstart = first base kept, rstop = end of what is kept (both relative to `read`).
      Match f, b;
      const bool have_f = locate_any<MAXM>(a, read, n, f);
      if (!have_f && !(link & MIRGE_LINK_FRONT_OPTIONAL)) continue;
      const int rest = have_f ? f.rstop : 0;
      const bool have_b = locate_any<MAXM>((link & MIRGE_LINK_INDEX_MASK) - 1, read + rest, n - rest, b);
      if (!have_b && (!(link & MIRGE_LINK_BACK_OPTIONAL) || !have_f)) continue;
      mt.rstart = rest;
      mt.rstop = have_b ? rest + b.rstart : n;
      mt.matches = (have_f ? f.matches : 0) + (have_b ? b.matches : 0);
      mt.errors = (have_f ? f.errors : 0) + (have_b ? b.errors : 0);
    } else if (!locate_any<MAXM>(a, read, n, mt)) continue;
    if (which < 0 || mt.matches > best.matches || (mt.matches == best.matches && mt.errors < best.errors)) {
      best = mt;
      which = a;
    }
  }
  return which;
}

// returns true when the adapter search was deferred to the second pass (DEFER only)
template <int MAXM, bool FAST, bool DEFER>
__device__ __noinline__ bool apply_mod(int mi, const uint8_t *seq, const uint8_t *qual, int &start, int &stop, FastCtx &fc) {
  const int len = stop - start;
  switch (c_p.kind[mi]) {
    case MIRGE_MOD_NEXTSEQ:
      stop = start + nextseq_trim_index(seq + start, qual + start, len, c_p.a[mi], c_p.b[mi]);
      break;
    case MIRGE_MOD_QUALITY: {
      int s, e;
      quality_trim_index(qual + start, len, c_p.a[mi], c_p.b[mi], c_p.c[mi], s, e);
      stop = start + e;
      start = start + s;
      break;
    }
    case MIRGE_MOD_ADAPTER:
      for (int t = 0; t < c_p.times; ++t) {
        Match mt;
        fc.rbase = start;
        const int a = best_match<MAXM, FAST, DEFER>(seq + start, stop - start, mt, fc);
        if (a == -2) return true;
        if (a < 0) break;
        if (c_p.ad[a].link != 0) { stop = start + mt.rstop; start = start + mt.rstart; }  // a linked pair cuts both ends
        else if (!MIRGE_WHERE_IS_FRONT(c_p.ad[a].where)) stop = start + mt.rstart;  // 3' forms: read[:rstart]
        else start = start + mt.rstop;                                              // 5' forms: read[rstop:]
      }
      break;
    case MIRGE_MOD_NEND:
      while (start < stop && seq[start] == 'N') ++start;
      while (stop > start && seq[stop - 1] == 'N') --stop;
      break;
    case MIRGE_MOD_CUT: {
      const int c = c_p.a[mi];
      if (c > 0) start += min(c, len);
      else stop = start + max(len + c, 0);
      break;
    }
    default: break;
  }
  return false;
}
