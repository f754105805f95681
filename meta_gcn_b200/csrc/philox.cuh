// Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3", SC 2011; the constants
// and round structure of Random123's philox4x32 with 10 rounds).  A counter-based generator: the output is a pure
// function of (counter, key), so any thread can produce any draw without state — the dropout masks of
// csrc/dropout.cu depend on (seed, layer, row, column) only, never on thread mapping or completion order.
#pragma once
#include <stdint.h>

namespace mgcn {

constexpr uint32_t kPhiloxM0 = 0xD2511F53u;
constexpr uint32_t kPhiloxM1 = 0xCD9E8D57u;
constexpr uint32_t kPhiloxW0 = 0x9E3779B9u;   // key schedule (golden ratio)
constexpr uint32_t kPhiloxW1 = 0xBB67AE85u;   // key schedule (sqrt(3) - 1)

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(kPhiloxM0, c.x), lo0 = kPhiloxM0 * c.x;
    const uint32_t hi1 = __umulhi(kPhiloxM1, c.z), lo1 = kPhiloxM1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0);
    k0 += kPhiloxW0;
    k1 += kPhiloxW1;
  }
  return c;
}

}  // namespace mgcn
