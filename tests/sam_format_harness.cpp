// Host harness of mirge3.0_b200/csrc/sam_format.cuh (built by tests/test_sam_format_host.py with g++).
#define SAM_FORMAT_HOST
#include "sam_format.cuh"

// record of (key, hit) into out (or its length with out = NULL)
extern "C" uint32_t hs_record(const uint32_t *key, uint64_t hit, const mirge_library *lib, const mirge_round_policy *pol,
                              const uint8_t *names, const uint64_t *name_off, uint8_t *out) {
  return sam_record(key, hit, *lib, *pol, names, name_off, out);
}
