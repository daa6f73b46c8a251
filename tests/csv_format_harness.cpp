// Host harness of mirge3.0_b200/csrc/csv_format.cuh (built by tests/test_csv_format_host.py with g++).
#define CSV_FORMAT_HOST
#include "csv_format.cuh"

// row of key id `id` into out (or its length with out = NULL)
extern "C" uint32_t hc_row(const uint32_t *key, uint64_t id, uint32_t annot, uint64_t hit, const uint8_t *names,
                           const uint64_t *name_off, const uint32_t *round_base, int n_cols, const uint32_t *counts,
                           int n_samples, uint64_t stride, uint8_t *out) {
  return csv_row(key, id, annot, hit, names, name_off, round_base, n_cols, counts, n_samples, stride, out);
}
