// key_format.cuh -- slicing of packed keys ([len | n_exc << 16][2-bit payload][exceptions pos << 8 | byte], DESIGN.md
// section 3): the UMI flanks are cut off a first-level key to give the second-level (centre) key of digest.py:164-205,
// exceptions re-based; the byte reader and output cursor the text formatters (sam_format.cuh, csv_format.cuh) share.
// Included by collapse.cu; tests/test_key_format_host.py compiles it for the host.
#pragma once
#ifdef KEY_FORMAT_HOST
#include "host_shims.h"
#else
#include "common.cuh"
#endif

__device__ __forceinline__ uint32_t key_base(const uint32_t *key, uint32_t j) { return (key[1 + (j >> 4)] >> (2 * (j & 15))) & 3u; }

// Output cursor: counts bytes always, stores them only when out != nullptr (the sizing pass).
struct TextOut {
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

// out = key[f : len - b] as a packed key (exceptions re-based); returns its word count
__device__ __forceinline__ uint32_t slice_key(const uint32_t *key, int f, int b, uint32_t *out) {
  const uint32_t hdr = key[0];
  const int len = (int)key_len(hdr), nexc = (int)key_nexc(hdr);
  int cl = len - f - b;
  if (cl < 0) cl = 0;
  const int lo = (cl > 0) ? f : 0;
  const uint32_t npay_in = (uint32_t)(len + 15) >> 4, npay = (uint32_t)(cl + 15) >> 4;
  for (uint32_t w = 0; w < npay; ++w) {
    uint32_t word = 0;
    for (int q = 0; q < 16; ++q) {
      const int j = (int)w * 16 + q;
      if (j < cl) word |= key_base(key, (uint32_t)(lo + j)) << (2 * q);
    }
    out[1 + w] = word;
  }
  uint32_t xo = 0;
  for (int x = 0; x < nexc; ++x) {
    const uint32_t e = key[1 + npay_in + x];
    const int pos = (int)(e >> 8);
    if (pos >= lo && pos < lo + cl) out[1 + npay + xo++] = ((uint32_t)(pos - lo) << 8) | (e & 0xFFu);
  }
  out[0] = (uint32_t)cl | (xo << 16);
  return 1u + npay + xo;
}
