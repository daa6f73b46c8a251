// table_csv.cu -- the rows of mapped.csv / unmapped.csv (or of baking's complete_set) formatted on the device, where
// the packed keys, the annotation and the sample x key count matrix already are.  Two launches in the style of
// mirge_sam_format: the sizes of all rows, then (after the caller's exclusive scan) their bytes.  The per-row text is
// csv_format.cuh.
#include "common.cuh"

#include "csv_format.cuh"

#define CSV_THREADS 128

__global__ void __launch_bounds__(CSV_THREADS)
table_csv_kernel(mirge_table t, const uint32_t *__restrict__ rows, uint64_t n, const uint8_t *__restrict__ annot,
                 const uint64_t *__restrict__ hit, const uint8_t *__restrict__ names, const uint64_t *__restrict__ name_off,
                 const uint32_t *__restrict__ round_base, int n_cols, const uint32_t *__restrict__ counts, int n_samples,
                 uint64_t stride, int fill, uint32_t *__restrict__ lens, const uint64_t *__restrict__ offs,
                 uint8_t *__restrict__ out) {
  const uint64_t i = (uint64_t)blockIdx.x * CSV_THREADS + threadIdx.x;
  if (i >= n) return;
  const uint32_t id = rows[i];
  const uint32_t *key = t.d_arena + t.d_key_ref[id];
  const uint32_t a = annot ? annot[id] : 0xFFu;
  const uint64_t h = hit ? hit[id] : 0;
  const uint32_t len = csv_row(key, id, a, h, names, name_off, round_base, n_cols, counts, n_samples, stride,
                               fill ? out + offs[i] : nullptr);
  if (!fill) lens[i] = len;
}

extern "C" int mirge_table_csv_format(mirge_ctx *ctx, const mirge_table *t, const uint32_t *d_rows, uint64_t n,
                                      const uint8_t *d_annot, const uint64_t *d_hit, const uint8_t *d_names,
                                      const uint64_t *d_name_off, const uint32_t *d_round_base, int n_cols,
                                      const uint32_t *d_counts, int n_samples, uint64_t count_stride, int fill,
                                      uint32_t *d_lens, const uint64_t *d_offs, uint8_t *d_out, void *stream_) {
  if (!ctx) return MIRGE_ERR_ARG;
  if (!t || !d_rows) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: null argument");
  if (!d_annot != !d_hit) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: annotation rounds and hit words go together");
  if (d_annot && (!d_names || !d_name_off || !d_round_base)) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: annotation without names");
  if (n_cols < 0 || n_cols > 10 || n_samples < 0) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: bad column count");
  if (n_samples > 0 && !d_counts) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: null counts");
  if (fill ? (!d_offs || !d_out) : !d_lens) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: null output buffer");
  if (n == 0) return MIRGE_OK;
  if (!t->d_arena || !t->d_key_ref) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: table has no keys");
  if (n > 0xFFFFFFFFull * CSV_THREADS) MIRGE_FAIL(ctx, MIRGE_ERR_ARG, "table_csv: too many rows in one call");
  cudaStream_t stream = (cudaStream_t)stream_;
  MIRGE_CUDA(ctx, cudaSetDevice(ctx->device));
  table_csv_kernel<<<(unsigned)((n + CSV_THREADS - 1) / CSV_THREADS), CSV_THREADS, 0, stream>>>(
      *t, d_rows, n, d_annot, d_hit, d_names, d_name_off, d_round_base, n_cols, d_counts, n_samples,
      count_stride, fill, d_lens, d_offs, d_out);
  MIRGE_LAUNCH_CHECK(ctx, "table_csv_kernel");
  return MIRGE_OK;
}
