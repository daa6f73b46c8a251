// host_shims.h -- what the device headers compiled for the host by the tests need in place of common.cuh: the CUDA
// qualifiers as no-ops, the integer intrinsics they use, one-thread versions of the warp primitives, and the few
// helpers of common.cuh they call (kept identical to the originals there).
#pragma once
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "../../include/mirge_b200.h"
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
using std::max;
using std::min;
static inline int __popc(uint32_t x) { return __builtin_popcount(x); }
static inline int __clz(int x) { return x ? __builtin_clz((uint32_t)x) : 32; }
static inline int __clzll(long long x) { return x ? __builtin_clzll((unsigned long long)x) : 64; }
static inline uint32_t __brev(uint32_t x) {
  x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
  x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
  x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
  return __builtin_bswap32(x);
}
static inline uint32_t __funnelshift_r(uint32_t lo, uint32_t hi, uint32_t sh) {
  sh &= 31u;
  return sh ? (lo >> sh) | (hi << (32u - sh)) : lo;
}
static inline uint32_t __funnelshift_l(uint32_t lo, uint32_t hi, uint32_t sh) {
  sh &= 31u;
  return sh ? (hi << sh) | (lo >> (32u - sh)) : hi;
}
static inline unsigned __activemask() { return 1u; }
static inline void __syncwarp(unsigned = 0xffffffffu) {}
static inline unsigned __ballot_sync(unsigned, bool p) { return p ? 1u : 0u; }
// common.cuh
static inline uint32_t base_code_upper(uint32_t c) {
  c &= ~0x20u;
  return (c == 'A') ? 0u : (c == 'C') ? 1u : (c == 'G') ? 2u : (c == 'T') ? 3u : 4u;
}
static inline uint32_t key_len(uint32_t hdr) { return hdr & 0xFFFFu; }
static inline uint32_t key_nexc(uint32_t hdr) { return hdr >> 16; }
