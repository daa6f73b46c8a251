/*
 * mirge_b200.h -- C ABI of libmirge_b200.so: the B200 (sm_100a) implementation of miRge3.0's
 * per-read hot path (digest -> collapse -> ordered annotation rounds).
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  miRge3.0 is pure Python and reaches its
 * hot path through two function calls; the entry points below are what a ctypes binding inside
 * the reference would call instead (see INTEGRATION.md for the stub):
 *
 *   reference interface (under /root/reference)                    replaced by
 *   ---------------------------------------------------------------------------------------------
 *   mirge/libs/digest.py:105   baking(args, files, names, workDir)   mirge_set_trim_params,
 *     :140  dnaio.read_chunks + executor.submit(cutadapt, chunk)      mirge_tokenise_sync,
 *     :320  cutadapt(n) worker: parse + modifiers + key emission      mirge_line_index, mirge_trim,
 *     :141-163 parent merge (collapse)                                mirge_collapse_insert,
 *     :164-205 UMI second-level collapse                              mirge_umi_collapse,
 *     :237-261 sample x sequence matrix                               mirge_table_drain,
 *                                                                     mirge_table_export_keys
 *   mirge/libs/manifoldAlign.py:68 bwtAlign(args, df, workDir, db)   mirge_lib_kmers,
 *     :12   alignPlusParse (bowtie subprocess + SAM parse)            mirge_annotate_round
 *   mirge/libs/summary.py:677 summarize(...): per-library read sums   mirge_report_reduce
 *     (:692-698) and per-miRNA exact / isomiR sums (:716-770)
 *
 * Conventions: every function returns 0 on success or a negative MIRGE_ERR_* code and records a
 * message retrievable with mirge_last_error().  All pointers named d_* are DEVICE pointers owned
 * by the caller (torch.Tensor.data_ptr() in the Python host); the library never allocates data
 * buffers, it only owns a small control block per context.  Calls enqueue work on `stream`
 * (a cudaStream_t passed as void*) and return immediately unless suffixed _sync.  There is no
 * CPU fallback: without a CUDA device mirge_ctx_create fails.
 */
#ifndef MIRGE_B200_H
#define MIRGE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIRGE_ABI_VERSION 3

#define MIRGE_OK 0
#define MIRGE_ERR_CUDA (-1)     /* CUDA runtime error (message has the cudaError string) */
#define MIRGE_ERR_ARG (-2)      /* invalid argument / unsupported parameter combination */
#define MIRGE_ERR_FORMAT (-3)   /* malformed FASTQ (dnaio FastqFormatError equivalent) */
#define MIRGE_ERR_CAPACITY (-4) /* a caller-provided buffer / table is too small */
#define MIRGE_ERR_NODEVICE (-5) /* no usable CUDA device */

#define MIRGE_MAX_ADAPTERS 16 /* (more than MIRGE_FAST_ADAPTERS of them: full-DP kernel) */
#define MIRGE_FAST_ADAPTERS 4
#define MIRGE_MAX_ADAPTER_LEN 64
#define MIRGE_MAX_MODS 8
#define MIRGE_MAX_READ_LEN 512 /* bases per read handled by the trim kernel */

/* modifier kinds, in the order stipulate() may add them (mirge/libs/digest.py:87-99) */
#define MIRGE_MOD_NEXTSEQ 1 /* a = cutoff, b = quality base          (NextseqQualityTrimmer) */
#define MIRGE_MOD_QUALITY 2 /* a = 5' cutoff, b = 3' cutoff, c = base (QualityTrimmer)        */
#define MIRGE_MOD_ADAPTER 3 /*                                       (AdapterCutter)         */
#define MIRGE_MOD_NEND 4    /*                                       (NEndTrimmer)           */
#define MIRGE_MOD_CUT 5     /* a = length (>0: 5' end, <0: 3' end)   (UnconditionalCutter)   */

#define MIRGE_UMI_NONE 0
#define MIRGE_UMI_FLANKS 1 /* -umi f,b            (digest.py:359-366) */
#define MIRGE_UMI_QIAGEN 2 /* --qiagenumi -umi 0,U (digest.py:332-352) */

/* cutadapt's Aligner.locate picks, among the accepted alignments, the one with ...
 *   2.x - 3.x ("ADOPTED FROM CUTADAPT 2.7", digest.py:3): most matches, then lowest cost;
 *   >= 4.0: the highest score (match +1, mismatch -1, insertion / deletion -2), then lowest cost -- restated from the
 *   published description, not yet held against an install (tests/test_tier3_real_tools.py does when one is there).
 * MIRGE_COMPAT_CUTADAPT4 runs on the full-DP kernel (the bit-parallel search is built on the matches objective). */
#define MIRGE_COMPAT_CUTADAPT23 0
#define MIRGE_COMPAT_CUTADAPT4 1

#define MIRGE_COUNT_HEAD 0    /* count after every modifier, as digest.py:354-373 is written */
#define MIRGE_COUNT_RELEASE 1 /* count once after the pipeline (released 0.1.x behaviour)   */

/* mirge_adapter.where: cutadapt's Where of the placement (adapters.py; which ends of the alignment are free).
 * Odd values are the 5' forms (the match and what precedes it are removed), even ones the 3' forms. */
#define MIRGE_WHERE_BACK 0               /* -a SEQ   anywhere in the read, may hang over its 3' end; read[:start] is kept  */
#define MIRGE_WHERE_FRONT 1              /* -g SEQ   anywhere, may hang over the 5' end; read[stop:] is kept               */
#define MIRGE_WHERE_SUFFIX 2             /* -a SEQ$  anchored 3': read and adapter end together                            */
#define MIRGE_WHERE_PREFIX 3             /* -g ^SEQ  anchored 5': read and adapter start together                          */
#define MIRGE_WHERE_BACK_NOT_INTERNAL 4  /* -a SEQX  as BACK, but never inside the read                                    */
#define MIRGE_WHERE_FRONT_NOT_INTERNAL 5 /* -g XSEQ  as FRONT, but never inside the read                                   */
#define MIRGE_WHERE_IS_FRONT(w) ((w) & 1)

/* mirge_adapter.link of the 5' half of a linked pair = (1 + index of its 3' half) | flags */
#define MIRGE_LINK_BACK_HALF 0x100
#define MIRGE_LINK_INDEX_MASK 0xFF
#define MIRGE_LINK_FRONT_OPTIONAL 0x1000 /* the pair still matches when its 5' half is missing (";optional")               */
#define MIRGE_LINK_BACK_OPTIONAL 0x2000  /* ... when its 3' half is missing (the default of -a "A...B")                    */

/* One adapter in cutadapt's Aligner terms (restated in oracle/pyoracle.py::locate). */
typedef struct mirge_adapter {
  int32_t where;        /* MIRGE_WHERE_* */
  int32_t m;            /* adapter length, <= MIRGE_MAX_ADAPTER_LEN */
  int32_t min_overlap;  /* args.overlap, parse.py:90 */
  int32_t indel_cost;   /* 1, or 100000 when --no-indels (cutadapt adapters.py) */
  int32_t wildcard_ref; /* adapter contains IUPAC wildcards and -N was not given */
  int32_t wildcard_read; /* --match-read-wildcards (parse.py:97): IUPAC characters of the read match as sets */
  int32_t k;            /* int(error_rate * m) */
  int32_t effective_length;
  int32_t link;         /* 0 = plain adapter; (1 + index of the 3' half) | MIRGE_LINK_*_OPTIONAL = the 5' half of a linked
                         * pair (cutadapt parser / LinkedAdapter: -g "A...B" both halves non-anchored and required,
                         * -a "A...B" the 5' half anchored and required, the 3' half optional);
                         * MIRGE_LINK_BACK_HALF = the 3' half of a pair, never searched on its own */
  uint8_t mask[MIRGE_MAX_ADAPTER_LEN];  /* 4-bit IUPAC set per adapter base (A=1,C=2,G=4,T=8) */
  uint8_t ascii[MIRGE_MAX_ADAPTER_LEN]; /* upper-cased adapter text */
  int32_t n_counts[MIRGE_MAX_ADAPTER_LEN + 1]; /* number of 'N' before position i */
  int32_t max_err[MIRGE_MAX_ADAPTER_LEN + 1];  /* floor(L * error_rate) evaluated in double */
} mirge_adapter;

/* The hot-path subset of miRge's args namespace (mirge/libs/parse.py), resolved on the host. */
typedef struct mirge_trim_params {
  int32_t n_mods;
  int32_t mod_kind[MIRGE_MAX_MODS];
  int32_t mod_a[MIRGE_MAX_MODS];
  int32_t mod_b[MIRGE_MAX_MODS];
  int32_t mod_c[MIRGE_MAX_MODS];
  int32_t n_adapters;
  int32_t times;      /* args.times (parse.py:96) */
  int32_t min_len;    /* args.minimum_length (parse.py:83) */
  int32_t umi_mode;   /* MIRGE_UMI_* */
  int32_t umi5, umi3; /* -umi f,b */
  int32_t qia_adapter_len; /* len(args.adapters[0][1]) (digest.py:121,343) */
  int32_t count_mode; /* MIRGE_COUNT_* */
  int32_t compat;     /* MIRGE_COMPAT_*: which cutadapt's alignment objective Aligner.locate follows */
  mirge_adapter adapters[MIRGE_MAX_ADAPTERS];
} mirge_trim_params;

/* Hash table slot (collapse).  tag == 0: empty.  ref == 0: claimed, key not yet published. */
typedef struct mirge_slot {
  uint32_t tag;   /* 32-bit filter derived from the 64-bit key hash, never 0 */
  uint32_t ref;   /* 1 + word offset of the key in the arena */
  uint32_t id;    /* dense key id (creation order) */
  uint32_t count; /* occurrences since the last drain (current sample) */
} mirge_slot;

/* A collapse table: open addressing over `capacity` slots (power of two) + key arena.
 * Packed key = u32 words: [len | n_exc << 16][ceil(len/16) words, 2 bits/base, base j in bits
 * 2*(j%16) of word j/16, A=0 C=1 G=2 T=3][n_exc words: (pos << 8) | raw byte for every character
 * that is not one of "ACGT" (its 2-bit code is 0)].  Key identity is word-wise equality, i.e.
 * exact string equality of the original read text.
 * ctrl (device, 8 x u64): [0] arena words used  [1] number of keys  [2] error flags
 *                         [3] deferred count     [4] deferred count (second list) [5..7] scratch */
typedef struct mirge_table {
  mirge_slot *d_slots;
  uint64_t capacity;
  uint32_t *d_arena;
  uint64_t arena_words;
  uint32_t *d_key_ref; /* [max_keys] arena word offset of key id */
  uint64_t max_keys;
  uint64_t *d_ctrl;
} mirge_table;

/* One annotation library resident on the device (bowtie index replacement). */
#define MIRGE_LIB_PAD_WORDS 40 /* readable zero words after d_packed: > MIRGE_MAX_READ_LEN / 16 + 2 */
typedef struct mirge_library {
  const uint32_t *d_packed;  /* 2 bits/base, all references concatenated, followed by MIRGE_LIB_PAD_WORDS zero words */
  const uint32_t *d_nmask;   /* 1 bit/base, 1 = reference base is not ACGT */
  const uint32_t *d_ref_off; /* [n_refs + 1] first base of each reference */
  uint32_t n_refs;
  uint32_t n_bases;
  const uint32_t *d_idx_kmer; /* [n_idx] sorted 16-mers (first base most significant, zero padded) */
  const uint32_t *d_idx_pos;  /* [n_idx] base position of each k-mer */
  uint32_t n_idx;
  uint32_t bucket_bits;         /* d_idx_bucket is indexed by the top bucket_bits bits of a 16-mer */
  const uint32_t *d_idx_bucket; /* [2^bucket_bits + 1] */
  const uint32_t *d_ref_block;  /* [(n_bases >> ref_block_shift) + 1] reference holding base b << ref_block_shift */
  uint32_t ref_block_shift;
  uint32_t filter_bases;        /* 0 = no prefix filter, else 4..16: d_filter has 4^filter_bases bits */
  const uint32_t *d_filter;     /* presence bitmap of the first filter_bases bases of every indexed position */
  uint32_t filter16_bits;       /* 0 = none, else 16..30: d_filter16 has 2^filter16_bits bits */
  uint32_t max_ref_len;         /* length of the longest reference (0 = unknown): an end-to-end alignment of a longer
                                   query cannot exist, the round is skipped for it */
  const uint32_t *d_filter16;   /* presence bitmap of a 32-bit mix of every complete 16-mer (mirge_lib_filter16) */
} mirge_library;

#define MIRGE_SELECT_LEN_LT26 0    /* round 0 (manifoldAlign.py:93)  */
#define MIRGE_SELECT_LEN_GT25 1    /* round 1 (manifoldAlign.py:104) */
#define MIRGE_SELECT_UNANNOTATED 2 /* rounds 2.. (manifoldAlign.py:120,129) */

/* Effective bowtie policy of one round (manifoldAlign.py:85; SURVEY.md section 8a table). */
typedef struct mirge_round_policy {
  int32_t round;       /* 0..9, stored into d_annot_round on a hit */
  int32_t select;      /* MIRGE_SELECT_* */
  int32_t seed_len;    /* 28 for -n mode, 0 = whole read (-v mode) */
  int32_t seed_mm;     /* -n N / -v N */
  int32_t total_mm;    /* 2 in -n mode (-e 70 with all-'I' qualities), N in -v mode */
  int32_t trim5;       /* -5 */
  int32_t trim3;       /* -3 */
  int32_t strip_polyT; /* round 3: query = sequence without its trailing T{3,} run */
} mirge_round_policy;

#define MIRGE_NO_HIT 0xFFFFFFFFFFFFFFFFull
/* hit word: (n_mismatch << 56) | (ref_index << 28) | offset ; canonical pick = minimum */
#define MIRGE_HIT_MM(h) ((uint32_t)((h) >> 56))
#define MIRGE_HIT_REF(h) ((uint32_t)(((h) >> 28) & 0xFFFFFFFu))
#define MIRGE_HIT_OFF(h) ((uint32_t)((h)&0xFFFFFFFu))

typedef struct mirge_ctx mirge_ctx;

int mirge_abi_version(void);
int mirge_ctx_create(int device, mirge_ctx **out);
void mirge_ctx_destroy(mirge_ctx *ctx);
const char *mirge_last_error(const mirge_ctx *ctx);

/* stipulate() equivalent: install the resolved modifier pipeline (digest.py:59-101,110-122). */
int mirge_set_trim_params(mirge_ctx *ctx, const mirge_trim_params *p);
/* Emission slots per read: n_mods in HEAD mode (digest.py:354-373), else 1. */
int mirge_trim_slots(const mirge_ctx *ctx);

/* ---- stage 1a: FASTQ tokeniser (dnaio.read_chunks + FastqIter, digest.py:140,324) ---------- */
uint64_t mirge_tokenise_scratch_bytes(uint64_t nbytes);
/* Count line breaks of d_fastq[0:nbytes) (must start at a record boundary).  *n_records = number
 * of complete 4-line records, *consumed = bytes they occupy.  is_final != 0: a last line without
 * '\n' is complete (EOF rule) and trailing bytes that do not form a record are a format error. */
int mirge_tokenise_sync(mirge_ctx *ctx, const uint8_t *d_fastq, uint64_t nbytes, int is_final,
                        void *d_scratch, uint64_t *n_records, uint64_t *consumed, void *stream);
/* d_line_start[4r .. 4r+3] = first byte of the header / sequence / '+' / quality line of record r;
 * d_line_start[4 * n_records] = one past the last record's '\n'.  Uses the scratch of the
 * preceding mirge_tokenise_sync on the same bytes. */
int mirge_line_index(mirge_ctx *ctx, const uint8_t *d_fastq, uint64_t nbytes, const void *d_scratch,
                     uint32_t *d_line_start, uint64_t n_records, void *stream);

/* ---- stage 1b: trim + key emission (cutadapt(n) worker body, digest.py:325-373) ------------ */
/* For record r and emission slot s (e = r * slots + s):
 *   d_win[4e..4e+3] = (start, stop, ustart, ustop): emitted text = read[start:stop] + read[ustart:ustop]
 *   d_key_off[e]    = word offset of the packed key in d_keys, or 0xFFFFFFFF when the slot is not
 *                     counted (length filter, digest.py:348,362,368).
 * d_win / d_key_off may both be NULL when only the insert list is wanted (the product path).
 * Insert list (d_ins, u64[ins_capacity >= n_records * slots], or NULL): one entry per DISTINCT key a read emits
 * -- low 32 bits = word offset of the key, high 32 bits = number of consecutive slots of that read that carry
 * this text (digest.py:354-373 counts the same string once per modifier) -- in no particular order;
 * d_trim_ctrl[0] >> 36 counts the entries.  mirge_collapse_insert_list consumes it.
 * d_trim_ctrl (16 x u64, zeroed by the caller): [0] key words used (low 36 bits; the caller may preset them to the
 * first free word of d_keys) | insert-list entries << 36 (records x slots must be < 2^28 per call)
 * [1] emitted keys [2] error flags
 * [3] first malformed record, [4] key words of all emitted keys (a slot whose text repeats the previous slot's
 * shares that slot's key: same d_key_off, no space of its own), [5] reads left to the whole-pipeline second pass, [6] reads whose adapter search
 * ran the bit-vector DP, [7] of those, the ones that needed cost columns.
 * d_scratch: mirge_trim_scratch_bytes(n_records) bytes, 16-byte aligned.  With 3' adapters of <= 32 nt the work
 * is split at the adapter modifier: stage 1 handles every read up to there (an exact occurrence of the whole
 * adapter settles the search), the reads that need the DP are listed in the scratch (record, window, packed
 * text) and searched by list-driven kernels with sorted, full warps. */
uint64_t mirge_trim_scratch_bytes(uint64_t n_records);
int mirge_trim(mirge_ctx *ctx, const uint8_t *d_fastq, uint64_t nbytes, const uint32_t *d_line_start,
               uint64_t n_records, uint16_t *d_win, uint32_t *d_key_off, uint32_t *d_keys,
               uint64_t keys_capacity_words, uint64_t *d_trim_ctrl, void *d_scratch, uint64_t *d_ins,
               uint64_t ins_capacity, void *stream);

/* ---- stages 1a + 1b in one pass: fused tokeniser + trim (the product path) -------------------------------------
 * The same result as mirge_tokenise_sync + mirge_line_index + mirge_trim without a separate pass over the bytes: a
 * persistent kernel takes the stream tile by tile through the bulk-copy engine (cp.async.bulk + mbarrier), finds the
 * line breaks of each tile in shared memory, numbers the records by a single-pass look-back over the tiles in front
 * and runs stage 1 of the split pipeline on the bytes where they lie; stages 2 / 3 and the whole-pipeline pass follow
 * as in mirge_trim.  Applies when mirge_digest_fused_ok() (3' adapters of <= 32 nt with indels, no qiagen UMIs,
 * automatic kernel choice); otherwise use the three calls above.
 * The number of records is not known beforehand: n_cap is the caller's bound (outputs and lists are sized by it:
 * d_line_start u32[4 n_cap + 4] or NULL, d_win / d_key_off for n_cap x slots or NULL, d_ins >= n_cap x slots
 * entries, d_scratch = mirge_digest_scratch_bytes(nbytes, n_cap)).  d_trim_ctrl (16 x u64, zeroed by the caller) as
 * for mirge_trim, plus [9] line breaks of the batch (with is_final, a last line without '\n' counts as complete),
 * [10] offset just behind the last complete record, relative to d_fastq rounded down to 16 bytes,
 * [2] bit 16: more than n_cap records -- repeat with n_cap >= [9] / 4; [2] bit 8: too many records for the
 * whole-pipeline list -- use the three-call path for this batch. */
int mirge_digest_fused_ok(const mirge_ctx *ctx);
uint64_t mirge_digest_scratch_bytes(uint64_t nbytes, uint64_t n_cap);
int mirge_digest_tiles(mirge_ctx *ctx, const uint8_t *d_fastq, uint64_t nbytes, int is_final, uint64_t n_cap,
                       uint32_t *d_line_start, uint16_t *d_win, uint32_t *d_key_off, uint32_t *d_keys,
                       uint64_t keys_capacity_words, uint64_t *d_trim_ctrl, void *d_scratch, uint64_t *d_ins,
                       uint64_t ins_capacity, void *stream);

/* Kernel selection for mirge_trim: 0 = automatic (split bit-parallel pipeline when every adapter is a 3'
 * adapter with indels and <= 32 nt, else the generic full-DP kernel), 1 = always generic, 2 = bit-parallel
 * kernel without the split (one kernel + second pass; kept for the parity tests).  When the generic-free
 * path meets a record group that does not fit its shared-memory staging the group goes to the second pass. */
int mirge_trim_mode(mirge_ctx *ctx, int mode);

/* ---- stage 2: collapse (digest.py:141-163,164-205,237-245) --------------------------------- */
int mirge_table_reset(mirge_ctx *ctx, const mirge_table *t, void *stream);
/* completeDict[key] += count for the n_items (offset, count) entries of a batch's insert list (mirge_trim): the parent
 * merge of digest.py:141-163.  d_keys = the buffer the list's offsets point into; when it is the table's own arena
 * (mirge_trim called with d_keys = t->d_arena and d_trim_ctrl[0] preset to the arena words in use) the first
 * occurrence of a key becomes the table's copy where it lies, otherwise new keys are copied into the arena.
 * d_scratch: u32[2 * n_items].  Dense key ids are handed out by a second, streaming kernel (no id atomic on the
 * chain of dependent accesses of an insert). */
int mirge_collapse_insert_list(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_keys, const uint64_t *d_ins,
                               uint64_t n_items, uint32_t *d_scratch, void *stream);
/* Merge (key, count) records: d_rec = [count][key words...] back to back, d_rec_off[i] = word
 * offset of record i.  Used by the owner side of the hash-partitioned exchange. */
int mirge_collapse_merge(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_rec,
                         const uint32_t *d_rec_off, uint64_t n_rec, uint32_t *d_deferred, void *stream);
/* The same when the records were received straight into the table's arena (the all-to-all writes them at the
 * arena's end): d_rec_off holds arena word offsets, the key of the first record of a sequence becomes the table's
 * copy, nothing is moved.  The caller advances the arena counter (d_ctrl[0]) past the received words. */
int mirge_collapse_merge_inplace(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_rec_off, uint64_t n_rec,
                                 uint32_t *d_deferred, void *stream);
/* Growth: re-insert every slot of old_t into the larger slot array of new_t (zeroed here).  Both
 * tables must reference the same key text (new_t->d_arena holds a copy of the used arena words),
 * the same d_key_ref contents and the same d_ctrl.  Key ids, refs and counts are preserved. */
int mirge_table_rehash(mirge_ctx *ctx, const mirge_table *old_t, const mirge_table *new_t, void *stream);
/* Checks error flags / deferred leftovers of the table after a batch (synchronises `stream`). */
int mirge_table_check_sync(mirge_ctx *ctx, const mirge_table *t, uint64_t *n_keys,
                           uint64_t *arena_used, void *stream);
/* End of a sample: append (key id, count) of every key seen since the last drain to d_ids/d_counts,
 * zero the per-sample counts.  *d_n_out (u64 on device) receives the number of pairs. */
int mirge_table_drain(mirge_ctx *ctx, const mirge_table *t, uint32_t *d_ids, uint32_t *d_counts,
                      uint64_t out_capacity, uint64_t *d_n_out, void *stream);
/* UMI second level (digest.py:164-205): for every (key, c) drained from `first`:
 * centre = key[umi5 : len - umi3]; if len(centre) >= min_len: second[centre] += (dedup ? 1 : c). */
int mirge_umi_collapse(mirge_ctx *ctx, const mirge_table *first, const uint32_t *d_ids,
                       const uint32_t *d_counts, uint64_t n_pairs, const mirge_table *second,
                       int umi5, int umi3, int min_len, int dedup, uint32_t *d_deferred,
                       void *stream);
/* Decode keys [id0, id0 + n) to ASCII rows of `stride` bytes (zero padded); d_len[i] = length. */
int mirge_table_export_keys(mirge_ctx *ctx, const mirge_table *t, uint64_t id0, uint64_t n,
                            uint8_t *d_ascii, uint32_t stride, uint32_t *d_len, void *stream);
/* Import of sequences that are already collapsed (the DataFrame index bwtAlign receives,
 * manifoldAlign.py:93-131): string i = d_ascii[d_str_off[i] : d_str_off[i+1]].  mirge_key_sizes
 * gives the packed size of each key in words; after an exclusive scan of those sizes into
 * d_key_off, mirge_pack_keys writes the keys, which makes (d_arena, d_key_off) usable as the
 * (d_arena, d_key_ref) of a mirge_table for mirge_annotate_round with key id = string index. */
int mirge_key_sizes(mirge_ctx *ctx, const uint8_t *d_ascii, const uint64_t *d_str_off, uint64_t n,
                    uint32_t *d_words, void *stream);
int mirge_pack_keys(mirge_ctx *ctx, const uint8_t *d_ascii, const uint64_t *d_str_off, uint64_t n,
                    const uint32_t *d_key_off, uint32_t *d_arena, void *stream);
/* Hash partition for the multi-GPU exchange: d_dest[i] = hash64(centre of key id i) % n_parts,
 * d_words[i] = 1 + key words (size of its exchange record). */
int mirge_partition_plan(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_ids, uint64_t n,
                         int umi5, int umi3, uint32_t n_parts, uint32_t *d_dest, uint32_t *d_words,
                         void *stream);
/* Write exchange records [count][key words] of pairs (d_ids[i], d_counts[i]) at word offsets
 * d_rec_off[i] of d_rec. */
int mirge_partition_pack(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_ids,
                         const uint32_t *d_counts, uint64_t n, const uint32_t *d_rec_off,
                         uint32_t *d_rec, void *stream);

/* The same packing without sorting by destination.  mirge_partition_totals: d_totals[d] = words and
 * d_totals[n_parts + d] = records bound for destination d (u64[2 * n_parts], zeroed here; n_parts <= 64).
 * mirge_partition_scatter: d_cursors (u64[n_parts]) holds, per destination, (first record index of its region in
 * d_sizes) << 32 | (first word offset of its region in d_rec), both < 2^32; every pair is written as [count][key words] at the offset
 * its destination's cursor hands out and its size in words to d_sizes (order inside a destination: arbitrary). */
int mirge_partition_totals(mirge_ctx *ctx, const uint32_t *d_dest, const uint32_t *d_words, uint64_t n,
                           uint32_t n_parts, uint64_t *d_totals, void *stream);
int mirge_partition_scatter(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_ids, const uint32_t *d_counts,
                            const uint32_t *d_dest, const uint32_t *d_words, uint64_t n, uint32_t n_parts,
                            uint64_t *d_cursors, uint32_t *d_rec, uint32_t *d_sizes, void *stream);

/* Sharding BEFORE the collapse (reads of one sample spread over the ranks; the reference's counterpart is the
 * parent loop that merges the workers' dictionaries, digest.py:141-163): the insert list of a batch (d_keys, d_ins as
 * mirge_trim / mirge_digest_tiles wrote them) is cut by owner = hash(key) mod n_parts into n_parts regions of
 * d_out_items (u64 = {u32 word offset of the key inside the region's keys, u32 count}; region d starts at d * cap_items)
 * and d_out_keys (region d starts at word d * cap_words).  d_cursors[d] (u64[n_parts], zeroed here) = items << 32 | key
 * words bound for d -- it keeps counting when a region is full; the caller then repeats with regions that large.
 * mirge_shard_rebase: after the all-to-all the items of source s (item_counts[s] of them, back to back in d_items)
 * get the word offset key_bases[s] of that source's keys (host arrays of n_parts values) added to their key offsets,
 * which makes d_items an insert list for mirge_collapse_insert_list. */
int mirge_shard_scatter(mirge_ctx *ctx, const uint32_t *d_keys, const uint64_t *d_ins, uint64_t n_items, uint32_t n_parts,
                        uint32_t cap_items, uint32_t cap_words, uint64_t *d_cursors, uint64_t *d_out_items,
                        uint32_t *d_out_keys, void *stream);
int mirge_shard_rebase(mirge_ctx *ctx, uint64_t *d_items, uint32_t n_parts, const uint64_t *item_counts,
                       const uint64_t *key_bases, void *stream);

/* ---- stage 3: annotation rounds (bwtAlign, manifoldAlign.py:68-146) ------------------------ */
/* 16-mer (zero padded, truncated at reference ends / ambiguous bases) of every base position:
 * d_kmer[n_bases], d_valid[n_bases] = number of usable bases (0..16).  Input to the host-side
 * sort that builds mirge_library.d_idx_*. */
int mirge_lib_kmers(mirge_ctx *ctx, const mirge_library *lib, uint32_t *d_kmer, uint8_t *d_valid,
                    void *stream);
/* Presence bitmap over the first prefix_bases (4..16) bases of every position with at least that many usable
 * bases (d_kmer / d_valid as written by mirge_lib_kmers): d_filter (4^prefix_bases bits, zeroed here) becomes
 * mirge_library.d_filter.  A seed piece whose prefix bit is clear has no occurrence in the library. */
int mirge_lib_filter(mirge_ctx *ctx, const uint32_t *d_kmer, const uint8_t *d_valid, uint32_t n_bases,
                     uint32_t prefix_bases, uint32_t *d_filter, void *stream);
/* The same for complete 16-mers through a hash: bit (mix32(16-mer) >> (32 - bits)) of d_filter16 (2^bits bits, zeroed
 * here, bits = 16..30) is set for every position with 16 usable bases.  A 16-base seed piece whose bit is clear does
 * not occur in the library; with 64 bits per position one look-up in 64 of an absent piece passes (the prefix
 * bitmap of a small library passes one in 16-20).  mirge_library.d_filter16 / filter16_bits. */
int mirge_lib_filter16(mirge_ctx *ctx, const uint32_t *d_kmer, const uint8_t *d_valid, uint32_t n_bases,
                       uint32_t bits, uint32_t *d_filter16, void *stream);
/* One bowtie round over the keys of table t.  Keys selected by policy->select that have a valid
 * alignment get d_annot_round[id] = policy->round and d_hit[id] = canonical pick (minimum of
 * (n_mismatch, reference index, offset) over the valid hit set). */
int mirge_annotate_round(mirge_ctx *ctx, const mirge_library *lib, const mirge_round_policy *policy,
                         const mirge_table *t, uint64_t n_keys, uint8_t *d_annot_round,
                         uint64_t *d_hit, void *stream);

/* The same for several consecutive rounds (libs[i] / policies[i] = round i of the call).  At most 10 rounds per call.
 * d_scratch == NULL: one thread per sequence runs all rounds (the sequence leaves at the first round that hits it).
 * d_scratch = mirge_annotate_scratch_bytes(n_keys) bytes, 8-byte aligned (the product path): pass 1 evaluates the
 * seed-piece filters of all rounds of every sequence into a round mask; pass 2 gives a warp 256 sequences, which it
 * compacts and searches round by round from a shared-memory copy of each key; sequences that search does not take
 * (exception words, > 128 bases, many candidates) are listed and finished by pass 3 with the general code.  Same results. */
uint64_t mirge_annotate_scratch_bytes(uint64_t n_keys);
int mirge_annotate_rounds(mirge_ctx *ctx, const mirge_library *libs, const mirge_round_policy *policies,
                          int n_rounds, const mirge_table *t, uint64_t n_keys, uint8_t *d_annot_round,
                          uint64_t *d_hit, void *d_scratch, void *stream);

/* Every hit of the best stratum for the sequences d_ids[0..n_ids) that `policy`'s round annotated (bowtie
 * -a --best --strata, rounds 2 and 3; feeds the per-round SAM files of -trf / -bam, manifoldAlign.py:20-62).
 * Two calls: fill = 0 writes d_counts[i] = hits found for d_ids[i]; after an exclusive scan into d_offs, fill = 1
 * writes the hit words to d_out[d_offs[i] ...].  An alignment reachable through several seed pieces appears once
 * per piece; callers remove duplicates. */
int mirge_annotate_allhits(mirge_ctx *ctx, const mirge_library *lib, const mirge_round_policy *policy,
                           const mirge_table *t, const uint32_t *d_ids, uint64_t n_ids, const uint64_t *d_hit,
                           int fill, uint32_t *d_counts, const uint64_t *d_offs, uint64_t *d_out, void *stream);

/* The per-round SAM records of -bam / -trf (manifoldAlign.py:20-62), one per (d_ids[i], d_hits[i]) pair: key id of
 * table t and hit word of `policy`'s round against `lib`.  Record i is
 *   QNAME \t 0 \t RNAME \t POS \t 255 \t <n>M \t * \t 0 \t 0 \t SEQ \t QUAL \t XA:i:<x> \t MD:Z:<md> \t NM:i:<nm> \n
 * QNAME = the key text; SEQ = the round's query (trailing T run stripped with strip_polyT, then trim5 / trim3), n its
 * length, QUAL n x 'I'; RNAME = d_names[d_name_off[r] .. d_name_off[r + 1]) of r = MIRGE_HIT_REF; POS = offset + 1;
 * MD / NM over the reference text (ambiguous bases print as 'N'), XA = mismatches inside the seed (seed_len, 0 = all).
 * Two calls: fill = 0 writes d_lens[i] = bytes of record i; after an exclusive scan into d_offs, fill = 1 writes the
 * records to d_out + d_offs[i]. */
int mirge_sam_format(mirge_ctx *ctx, const mirge_library *lib, const mirge_round_policy *policy, const mirge_table *t,
                     const uint32_t *d_ids, const uint64_t *d_hits, uint64_t n, const uint8_t *d_names,
                     const uint64_t *d_name_off, int fill, uint32_t *d_lens, const uint64_t *d_offs, uint8_t *d_out,
                     void *stream);

/* ---- stage 4: counters of annotation.report.csv (summarize, summary.py:692-698,716-770) ---- */
/* For every (key id, count) pair of ONE sample (the output of mirge_table_drain):
 *   d_round_sum[round of the key] += count            (u64[10]; unannotated keys are skipped)
 *   d_can[ref] += count for round 0 (exact miRNA), d_iso[ref] += count for round 8 (isomiR),
 *   ref = MIRGE_HIT_REF(d_hit[id]) < n_mirna  (both rounds search the same miRNA library).
 * Accumulates into the caller-zeroed arrays; synchronises `stream` (error check). */
int mirge_report_reduce(mirge_ctx *ctx, const uint8_t *d_annot_round, const uint64_t *d_hit,
                        const uint32_t *d_ids, const uint32_t *d_counts, uint64_t n_pairs, uint32_t n_mirna,
                        uint64_t *d_round_sum, uint64_t *d_can, uint64_t *d_iso, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* MIRGE_B200_H */
