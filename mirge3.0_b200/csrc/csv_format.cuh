// csv_format.cuh -- one row of mapped.csv / unmapped.csv (mirge/__main__.py:164-173) or of baking's complete_set, the
// bytes pandas' DataFrame.to_csv writes for that row of the sequence table:
//   <Sequence>,<annotFlag>,<col 0>,...,<col C-1>,<count sample 0>,...,<count sample S-1>\n
// Included by table_csv.cu; tests/test_csv_format_host.py compiles the same text for the host (CSV_FORMAT_HOST) and
// holds it against to_csv.
#pragma once
#ifdef CSV_FORMAT_HOST
#define KEY_FORMAT_HOST
#include "host_shims.h"
#else
#include "common.cuh"
#endif

#include "key_format.cuh"

// The Sequence field as csv.QUOTE_MINIMAL writes it: in double quotes when the text holds ',', '"', '\r' or '\n', inner
// '"' doubled; a byte >= 0x80 (the host decodes keys as latin-1, to_csv encodes UTF-8) as its two-byte UTF-8 form.
// Only exception bytes can be special: the 2-bit payload is "ACGT".
__device__ __forceinline__ void csv_sequence(const uint32_t *key, TextOut &o) {
  const uint32_t hdr = key[0];
  const int len = (int)key_len(hdr), nexc = (int)key_nexc(hdr);
  const uint32_t *exc = key + 1 + ((len + 15) >> 4);
  bool quote = false;
  for (int x = 0; x < nexc; ++x) {
    const uint32_t c = exc[x] & 0xFFu;
    quote |= c == ',' || c == '"' || c == '\r' || c == '\n';
  }
  if (quote) o.put('"');
  int x = 0;
  for (int j = 0; j < len; ++j) {
    const uint32_t c = key_char(key, nexc, exc, j, x);
    if (c >= 0x80u) {
      o.put(0xC0u | (c >> 6));
      o.put(0x80u | (c & 0x3Fu));
      continue;
    }
    if (c == '"') o.put('"');
    o.put(c);
  }
  if (quote) o.put('"');
}

// The row of key `key` (key id `id`).  annot: the key's annotation round (0xFF = none); h: its hit word.  names: the
// annotation column fields (finished CSV bytes) of every library back to back, name_off their offsets; the name of
// reference r of round c is bytes name_off[round_base[c] + r] .. name_off[round_base[c] + r + 1].  counts[s * stride
// + id]: the key's count in sample s.  Writes to out unless it is null; returns the length.
__device__ __forceinline__ uint32_t csv_row(const uint32_t *key, uint64_t id, uint32_t annot, uint64_t h, const uint8_t *names,
                                            const uint64_t *name_off, const uint32_t *round_base, int n_cols,
                                            const uint32_t *counts, int n_samples, uint64_t stride, uint8_t *out) {
  TextOut o{out, 0};
  csv_sequence(key, o);
  o.put(',');
  o.put(annot != 0xFFu ? '1' : '0');
  for (int c = 0; c < n_cols; ++c) {
    o.put(',');
    if (annot == (uint32_t)c) {
      const uint64_t r = (uint64_t)round_base[c] + MIRGE_HIT_REF(h);
      for (uint64_t b = name_off[r]; b < name_off[r + 1]; ++b) o.put(names[b]);
    }
  }
  for (int s = 0; s < n_samples; ++s) {
    o.put(',');
    o.uint(counts[(uint64_t)s * stride + id]);
  }
  o.put('\n');
  return o.n;
}
