// common.cuh -- shared device/host helpers of libmirge_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/mirge_b200.h"

struct mirge_ctx {
  int device;
  char err[512];
  uint64_t *h_pinned;  // 8 x u64 pinned staging for small D2H reads
  uint64_t *d_small;   // 8 x u64 device scratch
  mirge_trim_params params;
  int params_set;
  int max_adapter_len;
  int fast_ok;    // every adapter is a 3' adapter with indels and m <= 32: bit-parallel trim kernel applies
  int split_ok;   // the split pipeline (exact search + list-driven DP kernels) applies
  int trim_mode;  // 0 = auto, 1 = force the generic full-DP kernel, 2 = bit-parallel kernel without the split (tests)
  int sm_count;
};

#define MIRGE_FAIL(ctx, code, ...)                         \
  do {                                                     \
    snprintf((ctx)->err, sizeof((ctx)->err), __VA_ARGS__); \
    return (code);                                         \
  } while (0)

#define MIRGE_CUDA(ctx, expr)                                                                     \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) MIRGE_FAIL(ctx, MIRGE_ERR_CUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define MIRGE_LAUNCH_CHECK(ctx, name)                                                               \
  do {                                                                                              \
    cudaError_t _e = cudaGetLastError();                                                            \
    if (_e != cudaSuccess) MIRGE_FAIL(ctx, MIRGE_ERR_CUDA, "launch %s: %s", name, cudaGetErrorString(_e)); \
  } while (0)

// ---------------------------------------------------------------- packed keys ----------------
// key[0] = len | n_exc << 16 ; payload ceil(len/16) words ; n_exc exception words (pos << 8 | byte)
__host__ __device__ __forceinline__ uint32_t key_len(uint32_t hdr) { return hdr & 0xFFFFu; }
__host__ __device__ __forceinline__ uint32_t key_nexc(uint32_t hdr) { return hdr >> 16; }
__host__ __device__ __forceinline__ uint32_t key_words(uint32_t hdr) {
  return 1u + ((key_len(hdr) + 15u) >> 4) + key_nexc(hdr);
}

// base byte -> 2-bit code (A=0 C=1 G=2 T=3) or 4 for anything that is not exactly one of "ACGT"
__device__ __forceinline__ uint32_t base_code_exact(uint32_t c) {
  // 'A'=0x41 'C'=0x43 'G'=0x47 'T'=0x54
  uint32_t code = (c == 'A') ? 0u : (c == 'C') ? 1u : (c == 'G') ? 2u : (c == 'T') ? 3u : 4u;
  return code;
}
// case-insensitive class used for matching: a/A.. -> 0..3, everything else (incl. U? no: cutadapt
// upper-cases the read, bowtie treats non-ACGT as N) -> 4
__device__ __forceinline__ uint32_t base_code_upper(uint32_t c) {
  c &= ~0x20u;
  return (c == 'A') ? 0u : (c == 'C') ? 1u : (c == 'G') ? 2u : (c == 'T') ? 3u : 4u;
}

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t h) {
  h ^= h >> 33;
  h *= 0xff51afd7ed558ccdull;
  h ^= h >> 33;
  h *= 0xc4ceb9fe1a85ec53ull;
  h ^= h >> 33;
  return h;
}
__host__ __device__ __forceinline__ uint64_t hash_step(uint64_t h, uint32_t w) {
  return (h ^ w) * 0x9E3779B97F4A7C15ull + 0x7F4A7C15u + (h >> 29);
}

__device__ __forceinline__ uint4 ld_volatile_u4(const void *p) {
  uint4 r;
  asm volatile("ld.volatile.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ld_volatile_u32(const void *p) {
  uint32_t r;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t *p) { return __ldcg(p); }
__device__ __forceinline__ uint4 ld_stream_u4(const void *p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// Asynchronous global -> shared copies (LDGSTS): every copy of a thread is in flight at once and no register is
// held for the data; the thread waits for all of its own copies with cp_async_wait_all().
__device__ __forceinline__ void cp_async_16(void *smem_dst, const void *gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_4(void *smem_dst, const void *gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// newline_mask: bit i set <=> byte i of the 32 bytes is '\n'.
// Exact zero-byte test of w ^ "\n\n\n\n" (bit 7 of every byte that is '\n'; no carry crosses a byte), then two words
// at a time: the flags of the first word move to bits 8b+3, those of the second stay at 8b+7, and one multiply by
// 2^0 + 2^7 + 2^14 + 2^21 lines all eight up in the top byte (the 32 partial products land on distinct bits, so
// the sum has no carries).
__device__ __forceinline__ uint32_t newline_flags(uint32_t w) {
  const uint32_t x = w ^ 0x0A0A0A0Au;
  const uint32_t t = (x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu;
  return ~(t | x) & 0x80808080u;
}
__device__ __forceinline__ uint32_t newline_mask(const uint32_t w[8]) {
  uint32_t m = 0;
#pragma unroll
  for (int k = 0; k < 8; k += 2) {
    const uint32_t q = newline_flags(w[k + 1]) | (newline_flags(w[k]) >> 4);
    m |= ((q * 0x00204081u) >> 24) << (4 * k);
  }
  return m;
}
