// The uniform number of one sampled word (include/slimt_b200.h, DESIGN §4.4b): Philox4x32-10 (Salmon et al., "Parallel
// random numbers: as easy as 1, 2, 3", SC 2011) of counter (step, key_lo, key_hi, 0) under key (seed_lo, seed_hi), and
// u = (((uint64)x0 << 32 | x1) >> 11) * 2^-53 in [0, 1).  Host and device compile the same code, so a host program can
// restate every draw the kernels make.
#pragma once
#include <stdint.h>

#ifdef __CUDACC__
#define SB_HD __host__ __device__ __forceinline__
#else
#define SB_HD inline
#endif

namespace sb {

struct Philox4 {
  uint32_t x[4];
};

SB_HD void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
  const uint64_t p = static_cast<uint64_t>(a) * b;
  hi = static_cast<uint32_t>(p >> 32), lo = static_cast<uint32_t>(p);
}

// Philox4x32 with 10 rounds: the round constants and key schedule of Random123's philox4x32_R(10, ...).
SB_HD Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
  for (int r = 0; r < 10; r++) {
    if (r > 0) k0 += 0x9E3779B9u, k1 += 0xBB67AE85u;
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(0xD2511F53u, c0, hi0, lo0);
    philox_mulhilo(0xCD9E8D57u, c2, hi1, lo1);
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0, c1 = lo1, c2 = n2, c3 = lo0;
  }
  return Philox4{{c0, c1, c2, c3}};
}

// The uniform number of decode step `step` for the row whose sampling key is `key`, under the call's `seed`.
SB_HD double sample_uniform(uint64_t seed, uint64_t key, uint32_t step) {
  const Philox4 r = philox4x32_10(step, static_cast<uint32_t>(key), static_cast<uint32_t>(key >> 32), 0u,
                                  static_cast<uint32_t>(seed), static_cast<uint32_t>(seed >> 32));
  const uint64_t bits = (static_cast<uint64_t>(r.x[0]) << 32) | r.x[1];
  return static_cast<double>(bits >> 11) * 0x1.0p-53;
}

}  // namespace sb

#undef SB_HD
