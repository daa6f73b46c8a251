// collapse.cu -- GPU hash-table collapse of emitted keys into (unique sequence -> count).
// Replaces the per-chunk dict of the worker and the parent merge loop (mirge/libs/digest.py:349-373
// and :141-163), the UMI second level (:164-205) and the per-sample column extraction feeding the
// sample x sequence matrix (:237-245).
//
// Table: open addressing (linear probing) over 16-byte slots {tag, ref, id, count}.  A slot is
// claimed with one 32-bit CAS on the tag; the owner then copies the packed key into an append-only
// arena (warp-aggregated bump allocation) and publishes `ref`.  Key identity is decided by comparing
// the full packed key in the arena, never by the hash alone, so counts are exact.  A thread that
// meets a claimed-but-unpublished slot polls a bounded number of times and otherwise defers its key
// to a retry list that a follow-up kernel drains with one lane per warp (no intra-warp waiting),
// so the insert path cannot dead-lock.
#include <cooperative_groups.h>

#include <stdlib.h>

#include "common.cuh"
namespace cg = cooperative_groups;

#define COL_THREADS 256
#define SPIN_POLLS 64
#define MAX_PROBES 8192ull  // the host keeps the load factor <= 0.5; longer runs mean "table too small"
#define ERR_ARENA_FULL 1ull
#define ERR_KEYS_FULL 2ull
#define ERR_TABLE_FULL 4ull
#define ERR_STUCK 8ull
#define ERR_OUT_FULL 16ull

#define MAX_KEY_WORDS (1 + (MIRGE_MAX_READ_LEN + 15) / 16 + MIRGE_MAX_READ_LEN)

__device__ __forceinline__ uint64_t hash_key(const uint32_t *key, uint32_t nw) {
  uint64_t h = 0x243F6A8885A308D3ull;
  for (uint32_t i = 0; i < nw; ++i) h = hash_step(h, key[i]);
  return mix64(h);
}

enum { INS_OK = 0, INS_DEFER = 1, INS_FAIL = 2 };

#define NOT_IN_ARENA 0xFFFFFFFFu

// completeDict[key] += add.  `unbounded`: keep polling an unpublished slot (retry kernel only).
// in_arena: word offset of the key when it already lives in the table's arena (the trim kernel wrote it
// there): the owner then publishes that offset instead of allocating and copying.
// DEFER_ID: the owner takes no dense id here (and touches no shared counter when the key is in place): it reports
// the slot it created through *own_slot and a streaming kernel hands out the ids afterwards (assign_ids_kernel).
template <bool DEFER_ID>
__device__ __forceinline__ int table_insert(const mirge_table &t, const uint32_t *key, uint32_t nw, uint32_t add,
                                            uint64_t h, bool unbounded, uint32_t in_arena, uint32_t *own_slot = nullptr,
                                            uint32_t *dup_slot = nullptr) {
  unsigned long long *ctrl = (unsigned long long *)t.d_ctrl;
  const uint64_t mask = t.capacity - 1;
  uint32_t tag = (uint32_t)(h >> 32);
  if (tag == 0) tag = 1;
  uint64_t idx = h & mask;
  const uint64_t max_probe = t.capacity < MAX_PROBES ? t.capacity : MAX_PROBES;
  const unsigned lane = threadIdx.x & 31;
  for (uint64_t probe = 0; probe < max_probe; ++probe) {
    mirge_slot *s = t.d_slots + idx;
    uint4 v = ld_volatile_u4(s);
    if (v.x == 0) {
      const uint32_t old = atomicCAS(&s->tag, 0u, tag);
      if (old == 0) {
        // owner: dense id (and arena space unless the key is in place), one atomic for the lanes that
        // claimed a slot together
        const unsigned grp = __activemask();
        const int leader = __ffs(grp) - 1;
        const unsigned rank = __popc(grp & ((1u << lane) - 1u));
        unsigned long long base_id = 0, base_w = 0;
        uint32_t pre = 0, total = 0;
        if (in_arena == NOT_IN_ARENA) {
          for (unsigned m = grp; m; m &= m - 1) {  // exclusive prefix of the key sizes over the group
            const int src = __ffs(m) - 1;
            const uint32_t x = __shfl_sync(grp, nw, src);
            if ((unsigned)src < lane) pre += x;
            total += x;
          }
        }
        if ((int)lane == leader) {
          if (!DEFER_ID) base_id = atomicAdd(ctrl + 1, (unsigned long long)__popc(grp));
          if (in_arena == NOT_IN_ARENA) base_w = atomicAdd(ctrl + 0, (unsigned long long)total);
        }
        if (!DEFER_ID) base_id = __shfl_sync(grp, base_id, leader);
        if (!DEFER_ID || in_arena == NOT_IN_ARENA) base_w = __shfl_sync(grp, base_w, leader);
        const unsigned long long id = DEFER_ID ? 0ull : base_id + rank;
        const unsigned long long aoff = in_arena == NOT_IN_ARENA ? base_w + pre : (unsigned long long)in_arena;
        if (aoff + nw > t.arena_words || aoff + nw >= 0xFFFFFFF0ull || id >= t.max_keys) {
          atomicOr(ctrl + 2, id >= t.max_keys ? ERR_KEYS_FULL : ERR_ARENA_FULL);
          atomicExch(&s->ref, 0xFFFFFFFFu);  // poison: waiters give up immediately
          return INS_FAIL;
        }
        if (in_arena == NOT_IN_ARENA) {
          uint32_t *dst = t.d_arena + aoff;
          for (uint32_t i = 0; i < nw; ++i) dst[i] = key[i];
        }
        if (!DEFER_ID) {
          t.d_key_ref[id] = (uint32_t)aoff;
          s->id = (uint32_t)id;
        } else {
          *own_slot = (uint32_t)idx;
        }
        atomicAdd(&s->count, add);
        // release: a key text this thread just copied must be visible before ref.  A key that already sits in
        // the arena was written by an earlier kernel, and waiters read nothing else the owner wrote (they only
        // add to count, atomically; id and key_ref are read by later kernels), so no fence is needed then.
        if (in_arena == NOT_IN_ARENA) __threadfence();
        atomicExch(&s->ref, (uint32_t)aoff + 1u);
        return INS_OK;
      }
      v.x = old;
      v.y = 0;  // re-read below
    }
    if (v.x == tag) {
      uint32_t ref = v.y;
      if (ref == 0) {
        for (int k = 0; ref == 0 && (unbounded ? k < (1 << 16) : k < SPIN_POLLS); ++k) {
          __nanosleep(40);
          ref = ld_volatile_u32(&s->ref);
        }
        if (ref == 0) {
          if (unbounded) { atomicOr(ctrl + 2, ERR_STUCK); return INS_FAIL; }
          return INS_DEFER;
        }
      }
      if (ref == 0xFFFFFFFFu) return INS_FAIL;  // owner ran out of space (error already flagged)
      // the key address depends on ref, and the text is read from L2 (ld.cg), where the owner's
      // release made it visible before ref: no fence needed on this side
      const uint32_t *k2 = t.d_arena + (ref - 1u);
      bool same = true;
      if (nw <= 8u) {  // all words in flight together: a tag match is almost always the same key, an early exit saves nothing
        uint32_t d = 0;
#pragma unroll
        for (uint32_t i = 0; i < 8u; ++i)
          if (i < nw) d |= ld_cg_u32(k2 + i) ^ key[i];
        same = d == 0u;
      } else {
        for (uint32_t i = 0; i < nw; ++i) {
          if (ld_cg_u32(k2 + i) != key[i]) { same = false; break; }
        }
      }
      if (same) {
        atomicAdd(&s->count, add);
        if (dup_slot) *dup_slot = (uint32_t)idx;
        return INS_OK;
      }
    }
    idx = (idx + 1) & mask;
  }
  atomicOr(ctrl + 2, ERR_TABLE_FULL);
  return INS_FAIL;
}

__device__ __forceinline__ void defer_item(unsigned long long *counter, uint32_t *list, uint32_t item) {
  const unsigned grp = __activemask(), lane = threadIdx.x & 31;
  const int leader = __ffs(grp) - 1;
  unsigned long long base = 0;
  if ((int)lane == leader) base = atomicAdd(counter, (unsigned long long)__popc(grp));
  base = __shfl_sync(grp, base, leader);
  list[base + __popc(grp & ((1u << lane) - 1u))] = item;
}

// Exchange records of the owner-side merge: records [count][key...] at rec_off[i] that were received straight into
// the table's arena (keys == arena): the key of a record becomes the table's copy where it lies, nothing is moved.
__device__ __forceinline__ void item_key(const uint32_t *keys, const uint32_t *off, uint64_t i,
                                         const uint32_t *&key, uint32_t &add, uint32_t &in_arena) {
  const uint32_t o = off[i];
  if (o == 0xFFFFFFFFu) { key = nullptr; add = 0; in_arena = NOT_IN_ARENA; return; }
  key = keys + o + 1;
  add = keys[o];
  in_arena = o + 1;
}

// Hash of an in-arena key whose length is not known yet: the header and the next seven words are fetched together
// (clipped to the arena), so the header -> payload dependency costs one memory latency instead of two.
__device__ __forceinline__ uint64_t hash_key_in_arena(const mirge_table &t, const uint32_t *key, uint32_t aoff, uint32_t &nw,
                                                   uint32_t kw[8]) {
#pragma unroll
  for (uint32_t j = 0; j < 8u; ++j) kw[j] = ((uint64_t)aoff + j < t.arena_words) ? key[j] : 0u;
  nw = key_words(kw[0]);
  uint64_t h = 0x243F6A8885A308D3ull;
#pragma unroll
  for (uint32_t j = 0; j < 8u; ++j)
    if (j < nw) h = hash_step(h, kw[j]);
  for (uint32_t j = 8u; j < nw; ++j) h = hash_step(h, key[j]);
  return mix64(h);
}

__global__ void __launch_bounds__(COL_THREADS)
collapse_insert_kernel(mirge_table t, const uint32_t *__restrict__ keys, const uint32_t *__restrict__ off, uint64_t n,
                       uint32_t *__restrict__ deferred) {
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t *key; uint32_t add, in_arena;
  item_key(keys, off, i, key, add, in_arena);
  if (!key || add == 0) return;
  uint32_t nw, kw[8];
  const uint64_t h = hash_key_in_arena(t, key, in_arena, nw, kw);
  if (table_insert<false>(t, key, nw, add, h, false, in_arena) == INS_DEFER)
    defer_item((unsigned long long *)t.d_ctrl + 3, deferred, (uint32_t)i);
}

// drains the deferred list: one lane per warp, so a waiter never shares a warp with its claimant
__global__ void __launch_bounds__(COL_THREADS)
collapse_retry_kernel(mirge_table t, const uint32_t *__restrict__ keys, const uint32_t *__restrict__ off, uint64_t n,
                      const uint32_t *__restrict__ deferred) {
  if (threadIdx.x & 31) return;
  const unsigned long long nd = ((unsigned long long *)t.d_ctrl)[3];
  const uint64_t warp = ((uint64_t)blockIdx.x * COL_THREADS + threadIdx.x) >> 5;
  const uint64_t nwarps = ((uint64_t)gridDim.x * COL_THREADS) >> 5;
  for (uint64_t j = warp; j < nd; j += nwarps) {
    const uint64_t i = deferred[j];
    const uint32_t *key; uint32_t add, in_arena;
    item_key(keys, off, i, key, add, in_arena);
    if (!key) continue;
    const uint32_t nw = key_words(key[0]);
    table_insert<false>(t, key, nw, add, hash_key(key, nw), true, in_arena);
  }
}

__global__ void clear_deferred_kernel(unsigned long long *ctrl) { ctrl[3] = 0; }

// ---- the insert list of a batch (mirge_trim): one distinct key of a read per lane ------------------------------
#define NO_SLOT 0xFFFFFFFFu

// Hot keys.  Small-RNA samples are dominated by a few hundred sequences (the top miRNA alone is several per cent of
// the reads), and every repeat of such a key costs three transactions at ONE L2 slice -- the slot, the owner's key
// text, the count atomic -- so that slice sets the pace of the whole kernel (ncu: busiest slice 49 % busy, average
// 17 %).  A CTA therefore walks a contiguous chunk of the list and remembers the repeated keys it meets in a
// direct-mapped shared-memory cache (hash -> slot, key text, pending count): later repeats inside the chunk are
// decided against the cached text (exact comparison, not the hash) and counted in shared memory; the pending counts
// go to the slots with one atomic per entry when the CTA is done.  Only keys of <= 8 words are cached (reads of up
// to 112 bases without exceptions); longer ones take the global path.
#define HK_ENT 512
#define HK_ITEMS 4  // list items per thread (default; MIRGE_B200_HK_ITEMS overrides for experiments)
struct HotCache {
  unsigned long long hash[HK_ENT];
  uint32_t state[HK_ENT];  // 0 empty, 1 being filled, 2 valid
  uint32_t slot[HK_ENT];
  uint32_t pend[HK_ENT];
  uint32_t key[8][HK_ENT];
};

// IN_PLACE: the keys lie in the table's arena (the trim kernels wrote them there).  own[i] = slot this item
// created, NO_SLOT when the key existed (or the item was deferred).
template <bool IN_PLACE>
__global__ void __launch_bounds__(COL_THREADS)
collapse_list_kernel(mirge_table t, const uint32_t *__restrict__ keys, const uint2 *__restrict__ ins, uint64_t n,
                     uint32_t *__restrict__ own, uint32_t *__restrict__ deferred, const int per_thread) {
  __shared__ HotCache hc;
  for (int e = threadIdx.x; e < HK_ENT; e += COL_THREADS) { hc.state[e] = 0; hc.pend[e] = 0; }
  __syncthreads();
  const uint64_t chunk0 = (uint64_t)blockIdx.x * COL_THREADS * per_thread;
  for (int it = 0; it < per_thread; ++it) {
    const uint64_t i = chunk0 + (uint64_t)it * COL_THREADS + threadIdx.x;
    if (i >= n) break;
    const uint2 item = ins[i];
    const uint32_t o = item.x, add = item.y;
    const uint32_t *key = keys + o;
    uint32_t nw, slot = NO_SLOT, dslot = NO_SLOT, kw[8];
    uint64_t h;
    if (IN_PLACE) {
      h = hash_key_in_arena(t, key, o, nw, kw);
    } else {
      nw = key_words(key[0]);
#pragma unroll
      for (uint32_t j = 0; j < 8u; ++j) kw[j] = j < nw ? key[j] : 0u;
      h = hash_key(key, nw);
    }
    const uint32_t e = (uint32_t)(h >> 23) & (HK_ENT - 1);
    bool counted = false;
    if (nw <= 8u && *(volatile uint32_t *)&hc.state[e] == 2u) {
      __threadfence_block();
      if (*(volatile unsigned long long *)&hc.hash[e] == h) {
        uint32_t d = 0;
#pragma unroll
        for (uint32_t j = 0; j < 8u; ++j)
          if (j < nw) d |= *(volatile uint32_t *)&hc.key[j][e] ^ kw[j];
        if (d == 0u) {
          atomicAdd(&hc.pend[e], add);
          counted = true;
        }
      }
    }
    if (counted) {
      own[i] = NO_SLOT;
      continue;
    }
    const int rc = table_insert<true>(t, key, nw, add, h, false, IN_PLACE ? o : NOT_IN_ARENA, &slot, &dslot);
    own[i] = slot;
    if (rc == INS_DEFER) {
      defer_item((unsigned long long *)t.d_ctrl + 3, deferred, (uint32_t)i);
    } else if (dslot != NO_SLOT && nw <= 8u && atomicCAS(&hc.state[e], 0u, 1u) == 0u) {
      // a key that repeats: remember it (first come; the head of the distribution gets there first)
      hc.hash[e] = h;
      hc.slot[e] = dslot;
#pragma unroll
      for (uint32_t j = 0; j < 8u; ++j) hc.key[j][e] = kw[j];
      __threadfence_block();
      atomicExch(&hc.state[e], 2u);
    }
  }
  __syncthreads();
  for (int e = threadIdx.x; e < HK_ENT; e += COL_THREADS)
    if (hc.state[e] == 2u && hc.pend[e]) atomicAdd(&t.d_slots[hc.slot[e]].count, hc.pend[e]);
}

template <bool IN_PLACE>
__global__ void __launch_bounds__(COL_THREADS)
collapse_list_retry_kernel(mirge_table t, const uint32_t *__restrict__ keys, const uint2 *__restrict__ ins,
                           uint32_t *__restrict__ own, const uint32_t *__restrict__ deferred) {
  if (threadIdx.x & 31) return;
  const unsigned long long nd = ((unsigned long long *)t.d_ctrl)[3];
  const uint64_t warp = ((uint64_t)blockIdx.x * COL_THREADS + threadIdx.x) >> 5;
  const uint64_t nwarps = ((uint64_t)gridDim.x * COL_THREADS) >> 5;
  for (uint64_t j = warp; j < nd; j += nwarps) {
    const uint64_t i = deferred[j];
    const uint2 it = ins[i];
    const uint32_t o = it.x;
    const uint32_t *key = keys + o;
    const uint32_t nw = key_words(key[0]);
    uint32_t slot = NO_SLOT;
    table_insert<true>(t, key, nw, it.y, hash_key(key, nw), true, IN_PLACE ? o : NOT_IN_ARENA, &slot);
    own[i] = slot;
  }
}

// Dense key ids for the slots a batch created: a block-wide scan of the ownership flags and ONE atomic per CTA on
// the key counter; then id -> slot and id -> key offset.  Runs after the inserts, off their dependent chain.
template <bool IN_PLACE>
__global__ void __launch_bounds__(COL_THREADS)
assign_ids_kernel(mirge_table t, const uint2 *__restrict__ ins, const uint32_t *__restrict__ own, uint64_t n) {
  __shared__ uint32_t warp_tot[COL_THREADS / 32];
  __shared__ unsigned long long block_base;
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  const uint32_t slot = i < n ? own[i] : NO_SLOT;
  const bool mine = slot != NO_SLOT;
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned bal = __ballot_sync(0xffffffffu, mine);
  if (lane == 0) warp_tot[warp] = __popc(bal);
  __syncthreads();
  uint32_t before = 0, total = 0;
#pragma unroll
  for (int w = 0; w < COL_THREADS / 32; ++w) {
    const uint32_t x = warp_tot[w];
    if ((unsigned)w < warp) before += x;
    total += x;
  }
  if (total == 0) return;
  if (threadIdx.x == 0) block_base = atomicAdd((unsigned long long *)t.d_ctrl + 1, (unsigned long long)total);
  __syncthreads();
  if (!mine) return;
  const unsigned long long id = block_base + before + __popc(bal & ((1u << lane) - 1u));
  if (id >= t.max_keys) {
    atomicOr((unsigned long long *)t.d_ctrl + 2, ERR_KEYS_FULL);
    return;
  }
  mirge_slot *s = t.d_slots + slot;
  s->id = (uint32_t)id;
  t.d_key_ref[id] = IN_PLACE ? ins[i].x : s->ref - 1u;
}

static int check_table(mirge_ctx *ctx, const mirge_table *t) {
  if (!t || !t->d_slots || !t->d_arena || !t->d_key_ref || !t->d_ctrl) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table: null buffer");
  if (t->capacity < 2 || (t->capacity & (t->capacity - 1))) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table: capacity must be a power of two");
  if (((uintptr_t)t->d_slots & 15)) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table: slots must be 16-byte aligned");
  return MIRGE_OK;
}

extern "C" int mirge_table_reset(mirge_ctx *ctx, const mirge_table *t, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemsetAsync(t->d_slots, 0, t->capacity * sizeof(mirge_slot), stream));
  MIRGE_CUDA(ctx, cudaMemsetAsync(t->d_ctrl, 0, 8 * sizeof(uint64_t), stream));
  return MIRGE_OK;
}

extern "C" int mirge_collapse_insert_list(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_keys, const uint64_t *d_ins,
                                          uint64_t n_items, uint32_t *d_scratch, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  if (n_items == 0) return MIRGE_OK;
  if (!d_keys || !d_ins || !d_scratch) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "collapse: null buffer");
  const uint2 *ins = (const uint2 *)d_ins;
  if (n_items > 0xFFFFFFFFull) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "collapse: more than 2^32 items in one batch");
  if (t->capacity > 0xFFFFFFFFull) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "collapse: more than 2^32 - 1 slots");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  uint32_t *own = d_scratch, *deferred = d_scratch + n_items;
  const unsigned grid = (unsigned)((n_items + COL_THREADS - 1) / COL_THREADS);
  static int per_thread = 0;
  if (!per_thread) {
    const char *e = getenv("MIRGE_B200_HK_ITEMS");
    per_thread = e ? atoi(e) : HK_ITEMS;
    if (per_thread < 1 || per_thread > 4096) per_thread = HK_ITEMS;
  }
  const unsigned lgrid = (unsigned)((n_items + (uint64_t)COL_THREADS * per_thread - 1) / ((uint64_t)COL_THREADS * per_thread));
  if (d_keys == t->d_arena) {
    collapse_list_kernel<true><<<lgrid, COL_THREADS, 0, stream>>>(*t, d_keys, ins, n_items, own, deferred, per_thread);
    collapse_list_retry_kernel<true><<<ctx->sm_count, COL_THREADS, 0, stream>>>(*t, d_keys, ins, own, deferred);
    assign_ids_kernel<true><<<grid, COL_THREADS, 0, stream>>>(*t, ins, own, n_items);
  } else {
    collapse_list_kernel<false><<<lgrid, COL_THREADS, 0, stream>>>(*t, d_keys, ins, n_items, own, deferred, per_thread);
    collapse_list_retry_kernel<false><<<ctx->sm_count, COL_THREADS, 0, stream>>>(*t, d_keys, ins, own, deferred);
    assign_ids_kernel<false><<<grid, COL_THREADS, 0, stream>>>(*t, ins, own, n_items);
  }
  MIRGE_LAUNCH_CHECK(ctx, "collapse list kernels");
  clear_deferred_kernel<<<1, 1, 0, stream>>>((unsigned long long *)t->d_ctrl);
  MIRGE_LAUNCH_CHECK(ctx, "clear_deferred_kernel");
  return MIRGE_OK;
}

extern "C" int mirge_collapse_merge_inplace(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_rec_off, uint64_t n_rec,
                                            uint32_t *d_deferred, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!t) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "collapse: null table");
  int rc = check_table(ctx, t);
  if (rc) return rc;
  if (n_rec == 0) return MIRGE_OK;
  if (!d_rec_off || !d_deferred) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "collapse: null buffer");
  if (n_rec > 0xFFFFFFFFull) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "collapse: more than 2^32 items in one batch");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned grid = (unsigned)((n_rec + COL_THREADS - 1) / COL_THREADS);
  collapse_insert_kernel<<<grid, COL_THREADS, 0, stream>>>(*t, t->d_arena, d_rec_off, n_rec, d_deferred);
  MIRGE_LAUNCH_CHECK(ctx, "collapse_insert_kernel");
  collapse_retry_kernel<<<ctx->sm_count, COL_THREADS, 0, stream>>>(*t, t->d_arena, d_rec_off, n_rec, d_deferred);
  MIRGE_LAUNCH_CHECK(ctx, "collapse_retry_kernel");
  clear_deferred_kernel<<<1, 1, 0, stream>>>((unsigned long long *)t->d_ctrl);
  MIRGE_LAUNCH_CHECK(ctx, "clear_deferred_kernel");
  return MIRGE_OK;
}

extern "C" int mirge_table_check_sync(mirge_ctx *ctx, const mirge_table *t, uint64_t *n_keys, uint64_t *arena_used, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemcpyAsync(ctx->h_pinned, t->d_ctrl, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost, stream));
  MIRGE_CUDA(ctx, cudaStreamSynchronize(stream));
  const uint64_t *c = ctx->h_pinned;
  if (n_keys) *n_keys = c[1];
  if (arena_used) *arena_used = c[0];
  if (c[2] & ERR_STUCK) MIRGE_FAIL(ctx, MIRGE_ERR_CUDA, "collapse: a claimed slot was never published (internal error)");
  if (c[2] & (ERR_ARENA_FULL | ERR_KEYS_FULL | ERR_TABLE_FULL | ERR_OUT_FULL))
    MIRGE_FAIL(ctx, MIRGE_ERR_CAPACITY, "collapse: table capacity exceeded (flags 0x%llx: 1 arena, 2 key ids, 4 slots, 16 output)",
               (unsigned long long)c[2]);
  return MIRGE_OK;
}

// ------------------------------------------------------------------ growth (rehash) ---------

// Re-insert every occupied slot of `o` into the (larger, zeroed) slot array of `n`.  Keys are
// distinct already, so no comparison is needed; ids, refs and counts are preserved.
__global__ void __launch_bounds__(COL_THREADS) rehash_kernel(mirge_table o, mirge_table n) {
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  if (i >= o.capacity) return;
  const uint4 v = *(const uint4 *)(o.d_slots + i);
  if (v.x == 0) return;
  const uint32_t *key = n.d_arena + (v.y - 1u);
  const uint64_t h = hash_key(key, key_words(key[0]));
  const uint64_t mask = n.capacity - 1;
  uint64_t idx = h & mask;
  for (uint64_t probe = 0; probe < n.capacity; ++probe) {
    mirge_slot *s = n.d_slots + idx;
    if (atomicCAS(&s->tag, 0u, v.x) == 0u) {
      s->ref = v.y; s->id = v.z; s->count = v.w;
      return;
    }
    idx = (idx + 1) & mask;
  }
  atomicOr((unsigned long long *)n.d_ctrl + 2, ERR_TABLE_FULL);
}

extern "C" int mirge_table_rehash(mirge_ctx *ctx, const mirge_table *old_t, const mirge_table *new_t, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, old_t);
  if (rc) return rc;
  rc = check_table(ctx, new_t);
  if (rc) return rc;
  if (new_t->capacity < old_t->capacity) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "rehash: new table is smaller");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemsetAsync(new_t->d_slots, 0, new_t->capacity * sizeof(mirge_slot), stream));
  rehash_kernel<<<(unsigned)((old_t->capacity + COL_THREADS - 1) / COL_THREADS), COL_THREADS, 0, stream>>>(*old_t, *new_t);
  MIRGE_LAUNCH_CHECK(ctx, "rehash_kernel");
  return MIRGE_OK;
}

// ------------------------------------------------------------------ per-sample drain --------

#define DRAIN_PER_THREAD 4
// Sweep of the slot array: every CTA owns COL_THREADS * DRAIN_PER_THREAD consecutive slots (coalesced 16-byte
// loads), compacts the counted ones with a block-wide scan and reserves its output range with ONE atomic, so
// the sweep runs at streaming bandwidth instead of at the rate of same-address atomics.
__global__ void __launch_bounds__(COL_THREADS)
drain_kernel(mirge_table t, uint32_t *__restrict__ ids, uint32_t *__restrict__ counts, uint64_t cap, unsigned long long *n_out) {
  __shared__ uint32_t warp_tot[COL_THREADS / 32];
  __shared__ unsigned long long block_base;
  const uint64_t first = (uint64_t)blockIdx.x * (COL_THREADS * DRAIN_PER_THREAD) + threadIdx.x;
  uint4 v[DRAIN_PER_THREAD];
  uint32_t mine = 0;
#pragma unroll
  for (int k = 0; k < DRAIN_PER_THREAD; ++k) {
    const uint64_t i = first + (uint64_t)k * COL_THREADS;
    v[k] = make_uint4(0, 0, 0, 0);
    if (i < t.capacity) v[k] = *(const uint4 *)(t.d_slots + i);
    if (v[k].x != 0 && v[k].w != 0) ++mine;
  }
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  uint32_t inc = mine;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t x = __shfl_up_sync(0xffffffffu, inc, d);
    if (lane >= (unsigned)d) inc += x;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  uint32_t before = 0, total = 0;
#pragma unroll
  for (int w = 0; w < COL_THREADS / 32; ++w) {
    const uint32_t x = warp_tot[w];
    if ((unsigned)w < warp) before += x;
    total += x;
  }
  if (total == 0) return;
  if (threadIdx.x == 0) block_base = atomicAdd(n_out, (unsigned long long)total);
  __syncthreads();
  unsigned long long o = block_base + before + inc - mine;
#pragma unroll
  for (int k = 0; k < DRAIN_PER_THREAD; ++k) {
    if (v[k].x == 0 || v[k].w == 0) continue;
    if (o < cap) {
      ids[o] = v[k].z;
      counts[o] = v[k].w;
    } else {
      atomicOr((unsigned long long *)t.d_ctrl + 2, ERR_OUT_FULL);
    }
    ++o;
    t.d_slots[first + (uint64_t)k * COL_THREADS].count = 0;
  }
}

extern "C" int mirge_table_drain(mirge_ctx *ctx, const mirge_table *t, uint32_t *d_ids, uint32_t *d_counts, uint64_t out_capacity,
                                 uint64_t *d_n_out, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  if (!d_ids || !d_counts || !d_n_out) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "drain: null buffer");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemsetAsync(d_n_out, 0, 8, stream));
  const uint64_t per_cta = (uint64_t)COL_THREADS * DRAIN_PER_THREAD;
  const unsigned grid = (unsigned)((t->capacity + per_cta - 1) / per_cta);
  drain_kernel<<<grid, COL_THREADS, 0, stream>>>(*t, d_ids, d_counts, out_capacity, (unsigned long long *)d_n_out);
  MIRGE_LAUNCH_CHECK(ctx, "drain_kernel");
  return MIRGE_OK;
}

// ------------------------------------------------------------------ key slicing --------------
// key_base, slice_key (also compiled for the host by the tests)
#include "key_format.cuh"

__global__ void __launch_bounds__(128)
umi_collapse_kernel(mirge_table first, const uint32_t *__restrict__ ids, const uint32_t *__restrict__ counts, uint64_t n,
                    mirge_table second, int f, int b, int min_len, int dedup, uint32_t *__restrict__ deferred, int retry) {
  uint32_t buf[MAX_KEY_WORDS];
  unsigned long long *ctrl2 = (unsigned long long *)second.d_ctrl;
  uint64_t i, stride;
  uint64_t n_items = n;
  if (retry) {
    if (threadIdx.x & 31) return;
    n_items = ctrl2[3];
    i = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    stride = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  } else {
    i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    stride = (uint64_t)gridDim.x * blockDim.x;
  }
  for (; i < n_items; i += stride) {
    const uint64_t item = retry ? deferred[i] : i;
    const uint32_t *key = first.d_arena + first.d_key_ref[ids[item]];
    const int len = (int)key_len(key[0]);
    int cl = len - f - b;
    if (cl < 0) cl = 0;
    if (cl < min_len) continue;
    const uint32_t nw = slice_key(key, f, b, buf);
    const uint32_t add = dedup ? 1u : counts[item];
    const int rc = table_insert<false>(second, buf, nw, add, hash_key(buf, nw), retry != 0, NOT_IN_ARENA);
    if (rc == INS_DEFER) defer_item(ctrl2 + 3, deferred, (uint32_t)item);
  }
}

extern "C" int mirge_umi_collapse(mirge_ctx *ctx, const mirge_table *first, const uint32_t *d_ids, const uint32_t *d_counts,
                                  uint64_t n_pairs, const mirge_table *second, int umi5, int umi3, int min_len, int dedup,
                                  uint32_t *d_deferred, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, first);
  if (rc) return rc;
  rc = check_table(ctx, second);
  if (rc) return rc;
  if (n_pairs == 0) return MIRGE_OK;
  if (!d_ids || !d_counts || !d_deferred) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "umi_collapse: null buffer");
  if (umi5 < 0 || umi3 < 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "umi_collapse: negative UMI length");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned grid = (unsigned)((n_pairs + 127) / 128);
  umi_collapse_kernel<<<grid, 128, 0, stream>>>(*first, d_ids, d_counts, n_pairs, *second, umi5, umi3, min_len, dedup, d_deferred, 0);
  MIRGE_LAUNCH_CHECK(ctx, "umi_collapse_kernel");
  umi_collapse_kernel<<<ctx->sm_count, 128, 0, stream>>>(*first, d_ids, d_counts, n_pairs, *second, umi5, umi3, min_len, dedup, d_deferred, 1);
  MIRGE_LAUNCH_CHECK(ctx, "umi_collapse_kernel(retry)");
  clear_deferred_kernel<<<1, 1, 0, stream>>>((unsigned long long *)second->d_ctrl);
  return MIRGE_OK;
}

// ------------------------------------------------------------------ export -------------------

__global__ void __launch_bounds__(COL_THREADS)
export_keys_kernel(mirge_table t, uint64_t id0, uint64_t n, uint8_t *__restrict__ ascii, uint32_t stride, uint32_t *__restrict__ lens) {
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t *key = t.d_arena + t.d_key_ref[id0 + i];
  const uint32_t hdr = key[0], len = key_len(hdr), nexc = key_nexc(hdr), npay = (len + 15) >> 4;
  uint8_t *row = ascii + i * stride;
  const uint32_t lim = len < stride ? len : stride;
  for (uint32_t j = 0; j < lim; ++j) row[j] = "ACGT"[key_base(key, j)];
  for (uint32_t j = lim; j < stride; ++j) row[j] = 0;
  for (uint32_t x = 0; x < nexc; ++x) {
    const uint32_t e = key[1 + npay + x];
    if ((e >> 8) < lim) row[e >> 8] = (uint8_t)(e & 0xFFu);
  }
  lens[i] = len;
}

extern "C" int mirge_table_export_keys(mirge_ctx *ctx, const mirge_table *t, uint64_t id0, uint64_t n, uint8_t *d_ascii,
                                       uint32_t stride, uint32_t *d_len, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  if (n == 0) return MIRGE_OK;
  if (!d_ascii || !d_len || stride == 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "export: null buffer");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  export_keys_kernel<<<(unsigned)((n + COL_THREADS - 1) / COL_THREADS), COL_THREADS, 0, stream>>>(*t, id0, n, d_ascii, stride, d_len);
  MIRGE_LAUNCH_CHECK(ctx, "export_keys_kernel");
  return MIRGE_OK;
}

// ------------------------------------------------------------------ import (ASCII -> keys) ---

// mode 0: words[i] = size of the packed key of string i; mode 1: write the key at key_off[i]
__global__ void __launch_bounds__(COL_THREADS)
pack_keys_kernel(const uint8_t *__restrict__ ascii, const uint64_t *__restrict__ str_off, uint64_t n, int mode,
                 uint32_t *__restrict__ words, const uint32_t *__restrict__ key_off, uint32_t *__restrict__ arena) {
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint8_t *s = ascii + str_off[i];
  const uint32_t len = (uint32_t)(str_off[i + 1] - str_off[i]);
  const uint32_t npay = (len + 15) >> 4;
  if (mode == 0) {
    uint32_t nexc = 0;
    for (uint32_t p = 0; p < len; ++p) nexc += base_code_exact(s[p]) == 4u;
    words[i] = 1u + npay + nexc;
    return;
  }
  uint32_t *k = arena + key_off[i];
  uint32_t word = 0, xi = 0;
  for (uint32_t p = 0; p < len; ++p) {
    const uint32_t ch = s[p], code = base_code_exact(ch);
    if (code == 4u) k[1 + npay + xi++] = (p << 8) | ch;
    else word |= code << (2 * (p & 15));
    if ((p & 15) == 15) { k[1 + (p >> 4)] = word; word = 0; }
  }
  if (len & 15) k[1 + (len >> 4)] = word;
  k[0] = len | (xi << 16);
}

extern "C" int mirge_key_sizes(mirge_ctx *ctx, const uint8_t *d_ascii, const uint64_t *d_str_off, uint64_t n, uint32_t *d_words,
                               void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (n == 0) return MIRGE_OK;
  if (!d_ascii || !d_str_off || !d_words) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "key_sizes: null buffer");
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  pack_keys_kernel<<<(unsigned)((n + COL_THREADS - 1) / COL_THREADS), COL_THREADS, 0, (cudaStream_t)stream_>>>(
      d_ascii, d_str_off, n, 0, d_words, nullptr, nullptr);
  MIRGE_LAUNCH_CHECK(ctx, "pack_keys_kernel(sizes)");
  return MIRGE_OK;
}

extern "C" int mirge_pack_keys(mirge_ctx *ctx, const uint8_t *d_ascii, const uint64_t *d_str_off, uint64_t n,
                               const uint32_t *d_key_off, uint32_t *d_arena, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (n == 0) return MIRGE_OK;
  if (!d_ascii || !d_str_off || !d_key_off || !d_arena) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "pack_keys: null buffer");
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  pack_keys_kernel<<<(unsigned)((n + COL_THREADS - 1) / COL_THREADS), COL_THREADS, 0, (cudaStream_t)stream_>>>(
      d_ascii, d_str_off, n, 1, nullptr, d_key_off, d_arena);
  MIRGE_LAUNCH_CHECK(ctx, "pack_keys_kernel");
  return MIRGE_OK;
}

// ------------------------------------------------------------------ hash partition -----------

__global__ void __launch_bounds__(128)
partition_plan_kernel(mirge_table t, const uint32_t *__restrict__ ids, uint64_t n, int f, int b, uint32_t n_parts,
                      uint32_t *__restrict__ dest, uint32_t *__restrict__ words) {
  uint32_t buf[MAX_KEY_WORDS];
  const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t *key = t.d_arena + t.d_key_ref[ids[i]];
  uint64_t h;
  if (f == 0 && b == 0) {
    h = hash_key(key, key_words(key[0]));
  } else {
    const uint32_t nw = slice_key(key, f, b, buf);
    h = hash_key(buf, nw);
  }
  dest[i] = (uint32_t)(mix64(h ^ 0x5851F42D4C957F2Dull) % n_parts);
  words[i] = 1u + key_words(key[0]);
}

extern "C" int mirge_partition_plan(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_ids, uint64_t n, int umi5, int umi3,
                                    uint32_t n_parts, uint32_t *d_dest, uint32_t *d_words, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  if (n == 0) return MIRGE_OK;
  if (!d_ids || !d_dest || !d_words || n_parts == 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "partition_plan: bad argument");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  partition_plan_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(*t, d_ids, n, umi5, umi3, n_parts, d_dest, d_words);
  MIRGE_LAUNCH_CHECK(ctx, "partition_plan_kernel");
  return MIRGE_OK;
}

// ---- exchange packing without a sort: per-destination totals, then a scatter with per-destination cursors ----

#define MAX_PARTS 64

__global__ void __launch_bounds__(COL_THREADS)
partition_totals_kernel(const uint32_t *__restrict__ dest, const uint32_t *__restrict__ words, uint64_t n, uint32_t n_parts,
                        unsigned long long *__restrict__ totals) {
  __shared__ unsigned long long s_w[MAX_PARTS], s_r[MAX_PARTS];
  if (threadIdx.x < MAX_PARTS) { s_w[threadIdx.x] = 0; s_r[threadIdx.x] = 0; }
  __syncthreads();
  for (uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x; i < n; i += (uint64_t)gridDim.x * COL_THREADS) {
    const uint32_t d = dest[i];
    // one shared-memory atomic per group of lanes with the same destination
    const unsigned peers = __match_any_sync(__activemask(), d);
    const int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
    uint32_t w = words[i], sum = 0;
    for (unsigned m = peers; m; m &= m - 1) sum += __shfl_sync(peers, w, __ffs(m) - 1);
    if (lane == leader) {
      atomicAdd(&s_w[d], (unsigned long long)sum);
      atomicAdd(&s_r[d], (unsigned long long)__popc(peers));
    }
  }
  __syncthreads();
  if (threadIdx.x < n_parts) {
    if (s_w[threadIdx.x]) atomicAdd(totals + threadIdx.x, s_w[threadIdx.x]);
    if (s_r[threadIdx.x]) atomicAdd(totals + n_parts + threadIdx.x, s_r[threadIdx.x]);
  }
}

extern "C" int mirge_partition_totals(mirge_ctx *ctx, const uint32_t *d_dest, const uint32_t *d_words, uint64_t n, uint32_t n_parts,
                                      uint64_t *d_totals, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!d_totals || n_parts == 0 || n_parts > MAX_PARTS) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "partition_totals: 1..%d destinations", MAX_PARTS);
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemsetAsync(d_totals, 0, 2ull * n_parts * sizeof(uint64_t), stream));
  if (n == 0) return MIRGE_OK;
  if (!d_dest || !d_words) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "partition_totals: null buffer");
  uint64_t grid = (n + COL_THREADS - 1) / COL_THREADS;
  if (grid > (uint64_t)ctx->sm_count * 8) grid = (uint64_t)ctx->sm_count * 8;
  partition_totals_kernel<<<(unsigned)grid, COL_THREADS, 0, stream>>>(d_dest, d_words, n, n_parts, (unsigned long long *)d_totals);
  MIRGE_LAUNCH_CHECK(ctx, "partition_totals_kernel");
  return MIRGE_OK;
}

// record i goes to the send buffer of its destination: [count][key words...] at the word offset its destination's
// cursor hands out, its size to sizes[] at the record index of the second cursor.  The order inside a destination
// is arbitrary (the owner-side merge does not depend on it).  cursors[d] = record index << 32 | word offset.
__global__ void __launch_bounds__(COL_THREADS)
partition_scatter_kernel(mirge_table t, const uint32_t *__restrict__ ids, const uint32_t *__restrict__ counts,
                         const uint32_t *__restrict__ dest, const uint32_t *__restrict__ words, uint64_t n, uint32_t n_parts,
                         unsigned long long *__restrict__ cursors, uint32_t *__restrict__ rec, uint32_t *__restrict__ sizes) {
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t d = dest[i], w = words[i];
  const unsigned peers = __match_any_sync(__activemask(), d);
  const int leader = __ffs(peers) - 1, lane = threadIdx.x & 31;
  uint32_t before = 0, sum = 0;
  for (unsigned m = peers; m; m &= m - 1) {
    const int src = __ffs(m) - 1;
    const uint32_t x = __shfl_sync(peers, w, src);
    if (src < lane) before += x;
    sum += x;
  }
  // one atomic hands out the word range and the record range together (record index in the high half), so the
  // order of the records in the buffer and of their sizes in sizes[] is the same
  unsigned long long both = 0;
  if (lane == leader) both = atomicAdd(cursors + d, ((unsigned long long)__popc(peers) << 32) | (unsigned long long)sum);
  both = __shfl_sync(peers, both, leader);
  const unsigned long long wbase = both & 0xFFFFFFFFull, rbase = both >> 32;
  const uint32_t *key = t.d_arena + t.d_key_ref[ids[i]];
  uint32_t *o = rec + wbase + before;
  o[0] = counts[i];
  for (uint32_t k = 0; k + 1 < w; ++k) o[1 + k] = key[k];
  sizes[rbase + __popc(peers & ((1u << lane) - 1u))] = w;
}

extern "C" int mirge_partition_scatter(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_ids, const uint32_t *d_counts,
                                       const uint32_t *d_dest, const uint32_t *d_words, uint64_t n, uint32_t n_parts,
                                       uint64_t *d_cursors, uint32_t *d_rec, uint32_t *d_sizes, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  int rc = check_table(ctx, t);
  if (rc) return rc;
  if (n == 0) return MIRGE_OK;
  if (!d_ids || !d_counts || !d_dest || !d_words || !d_cursors || !d_rec || !d_sizes || n_parts == 0 || n_parts > MAX_PARTS)
    MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "partition_scatter: bad argument");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  partition_scatter_kernel<<<(unsigned)((n + COL_THREADS - 1) / COL_THREADS), COL_THREADS, 0, stream>>>(
      *t, d_ids, d_counts, d_dest, d_words, n, n_parts, (unsigned long long *)d_cursors, d_rec, d_sizes);
  MIRGE_LAUNCH_CHECK(ctx, "partition_scatter_kernel");
  return MIRGE_OK;
}

// ------------------------------------------------------------------ sharding before the collapse -----------
// One process per GPU, reads of ONE sample sharded over the ranks (SURVEY.md section 8e): the insert list of a batch
// -- (key offset, count) of every distinct key a read emitted -- is cut by owner = hash(key) mod ranks BEFORE any
// table sees it, the pieces travel with one all-to-all, and every rank collapses what it owns.  Nothing is inserted
// twice (a local collapse followed by a merge of the unique sequences inserts nearly every read twice when most emitted
// keys are unique, as the pre-adapter texts of HEAD counting are), and the owner's table, ids and annotation are the
// single-GPU ones.
//
// Send side: n_parts regions of fixed capacity, region d = items[cap_items] (uint2: word offset of the key inside the
// region's keys, count) and keys[cap_words].  A CTA counts its items per owner in shared memory, reserves its ranges
// with ONE global atomic per owner and then copies; the order inside a region is arbitrary (counts do not depend on
// it).  cursors[d] = items << 32 | words bound for d: it keeps counting when a region is full, so the host learns the
// exact sizes from it and repeats with larger regions.

#define XS_ITEMS 4

__device__ __forceinline__ uint32_t owner_of(uint64_t h, uint32_t n_parts) {
  return (uint32_t)(mix64(h ^ 0x5851F42D4C957F2Dull) % n_parts);
}

// CENTRE: the owner hashes the key without its f / b UMI flanks (slice_key), which is the owner partition_plan_kernel
// gives the same key: all first-level keys of one centre meet at one rank, so the UMI second level is owner-local.  The
// whole key still travels (the owner's first-level table needs it).
template <bool CENTRE>
__global__ void __launch_bounds__(COL_THREADS)
shard_scatter_kernel(const uint32_t *__restrict__ keys, const uint2 *__restrict__ ins, uint64_t n, uint32_t n_parts,
                     uint32_t cap_items, uint32_t cap_words, unsigned long long *__restrict__ cursors,
                     uint2 *__restrict__ out_items, uint32_t *__restrict__ out_keys, int f, int b) {
  // (two 32-bit counters per owner: item slot and key space of an item are handed out independently -- the item
  // carries its key's offset -- and 32-bit shared-memory atomics are native, 64-bit ones a compare-and-swap loop)
  __shared__ uint32_t s_items[MAX_PARTS], s_words[MAX_PARTS], s_bi[MAX_PARTS], s_bw[MAX_PARTS], s_ok[MAX_PARTS];
  if (threadIdx.x < MAX_PARTS) { s_items[threadIdx.x] = 0; s_words[threadIdx.x] = 0; }
  __syncthreads();
  const uint64_t chunk0 = (uint64_t)blockIdx.x * COL_THREADS * XS_ITEMS;
  const unsigned lane = threadIdx.x & 31;
  uint32_t off[XS_ITEMS], add[XS_ITEMS], nw[XS_ITEMS], dst[XS_ITEMS], l_item[XS_ITEMS], l_word[XS_ITEMS];
#pragma unroll
  for (int it = 0; it < XS_ITEMS; ++it) {
    const uint64_t i = chunk0 + (uint64_t)it * COL_THREADS + threadIdx.x;
    nw[it] = 0;
    if (i >= n) continue;
    const uint2 item = ins[i];
    const uint32_t *key = keys + item.x;
    const uint32_t w = key_words(key[0]);
    off[it] = item.x;
    add[it] = item.y;
    nw[it] = w;
    uint32_t d;
    if (CENTRE) {
      uint32_t buf[MAX_KEY_WORDS];
      d = owner_of(hash_key(buf, slice_key(key, f, b, buf)), n_parts);
    } else {
      d = owner_of(hash_key(key, w), n_parts);
    }
    dst[it] = d;
    // item slots: one atomic per group of lanes with the same owner
    const unsigned peers = __match_any_sync(__activemask(), d);
    uint32_t base = 0;
    if (lane == (unsigned)(__ffs(peers) - 1)) base = atomicAdd(&s_items[d], (uint32_t)__popc(peers));
    base = __shfl_sync(peers, base, __ffs(peers) - 1);
    l_item[it] = base + __popc(peers & ((1u << lane) - 1u));
    l_word[it] = atomicAdd(&s_words[d], w);
  }
  __syncthreads();
  if (threadIdx.x < n_parts) {
    const uint32_t ci = s_items[threadIdx.x], cw = s_words[threadIdx.x];
    uint32_t ok = 1;
    if (ci) {
      const unsigned long long g = atomicAdd(cursors + threadIdx.x, ((unsigned long long)ci << 32) | cw);
      s_bi[threadIdx.x] = (uint32_t)(g >> 32);
      s_bw[threadIdx.x] = (uint32_t)g;
      if ((g >> 32) + ci > cap_items || (g & 0xFFFFFFFFull) + cw > cap_words) ok = 0;
    }
    s_ok[threadIdx.x] = ok;
  }
  __syncthreads();
#pragma unroll
  for (int it = 0; it < XS_ITEMS; ++it) {
    if (nw[it] == 0) continue;
    const uint32_t d = dst[it];
    if (!s_ok[d]) continue;  // region full: the host sees it in the cursors and repeats with larger regions
    const uint32_t wo = s_bw[d] + l_word[it];
    out_items[(uint64_t)d * cap_items + s_bi[d] + l_item[it]] = make_uint2(wo, add[it]);
    const uint32_t *key = keys + off[it];
    uint32_t *o = out_keys + (uint64_t)d * cap_words + wo;
    for (uint32_t k = 0; k < nw[it]; ++k) o[k] = key[k];
  }
}

template <bool CENTRE>
static int shard_scatter(mirge_ctx *ctx, const uint32_t *d_keys, const uint64_t *d_ins, uint64_t n_items, uint32_t n_parts,
                         int f, int b, uint32_t cap_items, uint32_t cap_words, uint64_t *d_cursors, uint64_t *d_out_items,
                         uint32_t *d_out_keys, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!d_cursors || n_parts == 0 || n_parts > MAX_PARTS) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "shard_scatter: 1..%d owners", MAX_PARTS);
  if (f < 0 || b < 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "shard_scatter: negative UMI length");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  MIRGE_CUDA(ctx, cudaMemsetAsync(d_cursors, 0, n_parts * sizeof(uint64_t), stream));
  if (n_items == 0) return MIRGE_OK;
  if (!d_keys || !d_ins || !d_out_items || !d_out_keys) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "shard_scatter: null buffer");
  const uint64_t per_cta = (uint64_t)COL_THREADS * XS_ITEMS;
  shard_scatter_kernel<CENTRE><<<(unsigned)((n_items + per_cta - 1) / per_cta), COL_THREADS, 0, stream>>>(
      d_keys, (const uint2 *)d_ins, n_items, n_parts, cap_items, cap_words, (unsigned long long *)d_cursors, (uint2 *)d_out_items,
      d_out_keys, f, b);
  MIRGE_LAUNCH_CHECK(ctx, "shard_scatter_kernel");
  return MIRGE_OK;
}

extern "C" int mirge_shard_scatter(mirge_ctx *ctx, const uint32_t *d_keys, const uint64_t *d_ins, uint64_t n_items, uint32_t n_parts,
                                   uint32_t cap_items, uint32_t cap_words, uint64_t *d_cursors, uint64_t *d_out_items,
                                   uint32_t *d_out_keys, void *stream_) {
  return shard_scatter<false>(ctx, d_keys, d_ins, n_items, n_parts, 0, 0, cap_items, cap_words, d_cursors, d_out_items, d_out_keys,
                              stream_);
}

extern "C" int mirge_shard_scatter_centre(mirge_ctx *ctx, const uint32_t *d_keys, const uint64_t *d_ins, uint64_t n_items,
                                          uint32_t n_parts, int umi5, int umi3, uint32_t cap_items, uint32_t cap_words,
                                          uint64_t *d_cursors, uint64_t *d_out_items, uint32_t *d_out_keys, void *stream_) {
  return shard_scatter<true>(ctx, d_keys, d_ins, n_items, n_parts, umi5, umi3, cap_items, cap_words, d_cursors, d_out_items,
                             d_out_keys, stream_);
}

// Receive side: the items of the n_parts sources lie back to back (source s = items [item_end[s-1], item_end[s])) and
// their key offsets count from the start of their source's keys; the keys of source s rest at word key_base[s] of the
// buffer the collapse reads (the table's arena): make the offsets absolute.
struct ShardSources {
  uint32_t item_end[MAX_PARTS];
  uint32_t key_base[MAX_PARTS];
};

__global__ void __launch_bounds__(COL_THREADS)
shard_rebase_kernel(uint2 *__restrict__ items, uint64_t n, uint32_t n_parts, const ShardSources src) {
  const uint64_t i = (uint64_t)blockIdx.x * COL_THREADS + threadIdx.x;
  if (i >= n) return;
  uint32_t s = 0;
  while (s + 1 < n_parts && i >= src.item_end[s]) ++s;
  items[i].x += src.key_base[s];
}

extern "C" int mirge_shard_rebase(mirge_ctx *ctx, uint64_t *d_items, uint32_t n_parts, const uint64_t *item_counts,
                                  const uint64_t *key_bases, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!item_counts || !key_bases || n_parts == 0 || n_parts > MAX_PARTS) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "shard_rebase: 1..%d sources", MAX_PARTS);
  ShardSources src;
  uint64_t n = 0;
  for (uint32_t s = 0; s < n_parts; ++s) {
    n += item_counts[s];
    if (n > 0xFFFFFFFFull || key_bases[s] >= 0xFFFFFFF0ull) MIRGE_FAIL(ctx, MIRGE_ERR_CAPACITY, "shard_rebase: offsets beyond 2^32");
    src.item_end[s] = (uint32_t)n;
    src.key_base[s] = (uint32_t)key_bases[s];
  }
  if (n == 0) return MIRGE_OK;
  if (!d_items) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "shard_rebase: null buffer");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  shard_rebase_kernel<<<(unsigned)((n + COL_THREADS - 1) / COL_THREADS), COL_THREADS, 0, stream>>>((uint2 *)d_items, n, n_parts, src);
  MIRGE_LAUNCH_CHECK(ctx, "shard_rebase_kernel");
  return MIRGE_OK;
}
