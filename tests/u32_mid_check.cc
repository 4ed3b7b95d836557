// tests/u32_mid_check.cc -- mcgpu::u32_mid_f32 (mcpar_b200/csrc/mcgpu_math.cuh) against the fp64 uniform narrowed
// to fp32, (float)u32_mid(w), for every 32-bit word; prints the mismatch counts as JSON.  Built and run by
// tests/test_u32_mid.py.  As a check of the check, it also counts the words where one plain conversion,
// (float)w 2^-32 + 2^-33, differs from the reference: that form rounds twice and must be caught.
#include <stdio.h>
#include <string.h>
#define MCGPU_TABLE_QUAL static
#include "../mcpar_b200/csrc/mcgpu_tables.h"
#include "../mcpar_b200/csrc/mcgpu_math.cuh"

static uint32_t bits(float f) { uint32_t b; memcpy(&b, &f, 4); return b; }

int main()
{
  unsigned long long bad = 0, naive_bad = 0;
  uint32_t first_bad = 0;
  for (uint64_t i = 0; i < (1ull << 32); ++i) {
    const uint32_t w = (uint32_t)i;
    const float ref = (float)(((double)w + 0.5) * (1.0 / 4294967296.0));
    const float got = mcgpu::u32_mid_f32(w);
    const float naive = (float)w * 2.3283064365386963e-10f + 1.1641532182693481e-10f;
    if (bits(got) != bits(ref)) { if (!bad) first_bad = w; ++bad; }
    naive_bad += bits(naive) != bits(ref);
  }
  printf("{\"mismatches\": %llu, \"first_mismatch\": %u, \"naive_mismatches\": %llu}\n", bad, first_bad, naive_bad);
  return 0;
}
