// sam.cu -- the per-round SAM records of -bam / -trf (manifoldAlign.py:20-62) formatted on the device, where the packed
// keys, the hit words and the library text already are.  Two launches in the style of mirge_annotate_allhits: the sizes
// of all records, then (after the caller's exclusive scan) their bytes.  The per-record text is sam_format.cuh.
#include "common.cuh"

#include "sam_format.cuh"

#define SAM_THREADS 128

__global__ void __launch_bounds__(SAM_THREADS)
sam_format_kernel(mirge_library lib, mirge_round_policy pol, mirge_table t, const uint32_t *__restrict__ ids,
                  const uint64_t *__restrict__ hits, uint64_t n, const uint8_t *__restrict__ names,
                  const uint64_t *__restrict__ name_off, int fill, uint32_t *__restrict__ lens,
                  const uint64_t *__restrict__ offs, uint8_t *__restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * SAM_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t *key = t.d_arena + t.d_key_ref[ids[i]];
  const uint32_t len = sam_record(key, hits[i], lib, pol, names, name_off, fill ? out + offs[i] : nullptr);
  if (!fill) lens[i] = len;
}

extern "C" int mirge_sam_format(mirge_ctx *ctx, const mirge_library *lib, const mirge_round_policy *policy, const mirge_table *t,
                                const uint32_t *d_ids, const uint64_t *d_hits, uint64_t n, const uint8_t *d_names,
                                const uint64_t *d_name_off, int fill, uint32_t *d_lens, const uint64_t *d_offs, uint8_t *d_out,
                                void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!lib || !policy || !t || !d_ids || !d_hits || !d_names || !d_name_off) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "sam: null argument");
  if (fill ? (!d_offs || !d_out) : !d_lens) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "sam: null output buffer");
  if (n == 0) return MIRGE_OK;
  if (!lib->d_packed || !lib->d_nmask || !lib->d_ref_off || lib->n_refs == 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "sam: empty library");
  if (!t->d_arena || !t->d_key_ref) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "sam: table has no keys");
  if (policy->trim5 < 0 || policy->trim3 < 0 || policy->seed_len < 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "sam: unsupported policy");
  if (n > 0xFFFFFFFFull * SAM_THREADS) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "sam: too many records in one call");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  sam_format_kernel<<<(unsigned)((n + SAM_THREADS - 1) / SAM_THREADS), SAM_THREADS, 0, stream>>>(
      *lib, *policy, *t, d_ids, d_hits, n, d_names, d_name_off, fill, d_lens, d_offs, d_out);
  MIRGE_LAUNCH_CHECK(ctx, "sam_format_kernel");
  return MIRGE_OK;
}
