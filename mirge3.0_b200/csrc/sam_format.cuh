// sam_format.cuh -- one bowtie SAM record (the per-round SAM files of -bam / -trf, manifoldAlign.py:20-62) from a packed
// key, its hit word, the round's library and policy: the text of manifoldAlign.write_round_sam / pyoracle.sam_line,
//   QNAME \t 0 \t RNAME \t POS \t 255 \t <n>M \t * \t 0 \t 0 \t SEQ \t QUAL \t XA:i:<x> \t MD:Z:<md> \t NM:i:<nm> \n
// Included by sam.cu; tests/test_sam_format_host.py compiles the same text for the host (SAM_FORMAT_HOST) and holds it
// against the oracle.
#pragma once
#ifdef SAM_FORMAT_HOST
#define KEY_FORMAT_HOST
#include "host_shims.h"
#else
#include "common.cuh"
#endif

#include "key_format.cuh"

// Output cursor: counts bytes always, stores them only when out != nullptr (the sizing pass).
struct SamOut {
  uint8_t *out;
  uint32_t n;
  __device__ __forceinline__ void put(uint32_t c) {
    if (out) out[n] = (uint8_t)c;
    ++n;
  }
  __device__ __forceinline__ void uint(uint32_t v) {  // decimal, most significant digit first (no digit buffer)
    uint32_t p = 1;
    while (v / p >= 10u) p *= 10u;
    for (; p; p /= 10u) put('0' + (v / p) % 10u);
  }
  __device__ __forceinline__ void str(const char *s) {
    while (*s) put((uint32_t)*s++);
  }
};

// Byte j of a packed key read left to right: the 2-bit base, or the exception byte stored for j.  Every key writer
// (mirge_pack_keys, the trim emission, slice_key) lists the exceptions in ascending position, so a cursor that only
// moves forward finds them; `x` is that cursor, reset to 0 to start over.
__device__ __forceinline__ uint32_t key_char(const uint32_t *key, int nexc, const uint32_t *exc, int j, int &x) {
  while (x < nexc && (int)(exc[x] >> 8) < j) ++x;
  if (x < nexc && (int)(exc[x] >> 8) == j) return exc[x] & 0xFFu;
  return (uint32_t)"ACGT"[key_base(key, (uint32_t)j)];
}

// Reference base at library position p: "ACGT" from the 2-bit text, 'N' where the N mask is set (the FASTA's ambiguous
// bases); positions past the text, which no valid hit reaches, read as 'N' too.
__device__ __forceinline__ uint32_t sam_ref_char(const mirge_library &lib, uint64_t p) {
  if (p >= lib.n_bases) return 'N';
  if ((lib.d_nmask[p >> 5] >> (p & 31)) & 1u) return 'N';
  return (uint32_t)"ACGT"[(lib.d_packed[p >> 4] >> (2 * (p & 15))) & 3u];
}

// Query window [qs, qe) of the record, as manifoldAlign.round_query_text: with strip_polyT the trailing run of
// upper-case T goes (whatever its length), then q[trim5 : max(len - trim3, trim5)] with Python's slice clipping.
__device__ __forceinline__ void sam_window(const uint32_t *key, const mirge_round_policy &pol, int &qs, int &qe) {
  const uint32_t hdr = key[0];
  const int len = (int)key_len(hdr), nexc = (int)key_nexc(hdr);
  const uint32_t *exc = key + 1 + ((len + 15) >> 4);
  int e = len;
  if (pol.strip_polyT) {
    int x = nexc - 1;  // exceptions from the back: a lower-case 't' (or any non-"ACGT" byte) ends the run
    while (e > 0) {
      const int j = e - 1;
      while (x >= 0 && (int)(exc[x] >> 8) > j) --x;
      if ((x >= 0 && (int)(exc[x] >> 8) == j) || key_base(key, (uint32_t)j) != 3u) break;
      --e;
    }
  }
  qs = min(pol.trim5, e);
  qe = min(max(e - pol.trim3, pol.trim5), e);
  if (qe < qs) qe = qs;
}

// The record for key `key` and hit word h of round `pol` against `lib`; names = the library's reference names back to
// back, name_off[r] .. name_off[r + 1] the bytes of reference r.  Writes to out unless it is null; returns the length.
__device__ __forceinline__ uint32_t sam_record(const uint32_t *key, uint64_t h, const mirge_library &lib,
                                               const mirge_round_policy &pol, const uint8_t *names, const uint64_t *name_off,
                                               uint8_t *out) {
  const uint32_t hdr = key[0];
  const int len = (int)key_len(hdr), nexc = (int)key_nexc(hdr);
  const uint32_t *exc = key + 1 + ((len + 15) >> 4);
  int qs, qe;
  sam_window(key, pol, qs, qe);
  const int n = qe - qs;
  const uint32_t ref = MIRGE_HIT_REF(h), off = MIRGE_HIT_OFF(h);
  const uint64_t a = (uint64_t)lib.d_ref_off[ref] + off;
  const int seed = pol.seed_len == 0 ? n : min(pol.seed_len, n);
  SamOut o{out, 0};
  int x = 0;
  for (int j = 0; j < len; ++j) o.put(key_char(key, nexc, exc, j, x));  // QNAME: the key text verbatim
  o.str("\t0\t");
  for (uint64_t b = name_off[ref]; b < name_off[ref + 1]; ++b) o.put(names[b]);
  o.put('\t');
  o.uint(off + 1);
  o.str("\t255\t");
  o.uint((uint32_t)n);
  o.str("M\t*\t0\t0\t");
  x = 0;
  for (int j = qs; j < qe; ++j) o.put(key_char(key, nexc, exc, j, x));  // SEQ
  o.put('\t');
  for (int j = 0; j < n; ++j) o.put('I');  // QUAL
  // mismatches: upper(q[p]) not one of "ACGT", or not the reference base; counted once for XA (inside the seed) and NM
  int nm = 0, xa = 0;
  x = 0;
  for (int p = 0; p < n; ++p) {
    const uint32_t qc = base_code_upper(key_char(key, nexc, exc, qs + p, x));
    if (qc >= 4u || (uint32_t)"ACGT"[qc] != sam_ref_char(lib, a + p)) {
      ++nm;
      xa += p < seed;
    }
  }
  o.str("\tXA:i:");
  o.uint((uint32_t)xa);
  o.str("\tMD:Z:");
  int run = 0;
  x = 0;
  for (int p = 0; p < n; ++p) {
    const uint32_t qc = base_code_upper(key_char(key, nexc, exc, qs + p, x));
    const uint32_t rc = sam_ref_char(lib, a + p);
    if (qc < 4u && (uint32_t)"ACGT"[qc] == rc) {
      ++run;
      continue;
    }
    o.uint((uint32_t)run);
    o.put(rc);
    run = 0;
  }
  o.uint((uint32_t)run);
  o.str("\tNM:i:");
  o.uint((uint32_t)nm);
  o.put('\n');
  return o.n;
}
