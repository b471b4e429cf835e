// Philox4x32-10 counter-based generator and the multiply-shift integer mapping shared by the on-device generator
// (generate.cu) and the training-batch augmentation (augment.cu); oracle/philox_oracle.py restates both in numpy.
#pragma once
#include <stdint.h>

namespace ssd3d {

struct Philox4 {
  uint32_t v[4];
};

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  return Philox4{{c0, c1, c2, c3}};
}

// randint(lo, hi) = lo + ((u32 * (hi - lo)) >> 32): uniform over [lo, hi)
__device__ __forceinline__ int randint_ms(uint32_t u, int lo, int hi) {
  return lo + (int)(((uint64_t)u * (uint64_t)(uint32_t)(hi - lo)) >> 32);
}

}  // namespace ssd3d
