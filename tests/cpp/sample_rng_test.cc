// Host build of slimt_b200/csrc/sample_rng.cuh, the generator the sampling kernel runs (tests/test_sample_rng.py).
// Reads lines from stdin and answers one line each:
//   "philox c0 c1 c2 c3 k0 k1" (hex)  ->  "x0 x1 x2 x3" (hex, 8 digits)
//   "u seed key step" (decimal)       ->  u * 2^53 (decimal: an integer in [0, 2^53))
#include <cinttypes>
#include <cstdio>
#include <cstring>

#include "sample_rng.cuh"

int main() {
  char op[16];
  while (std::scanf("%15s", op) == 1) {
    if (std::strcmp(op, "philox") == 0) {
      uint32_t v[6];
      for (uint32_t &x : v)
        if (std::scanf("%" SCNx32, &x) != 1) return 2;
      const sb::Philox4 r = sb::philox4x32_10(v[0], v[1], v[2], v[3], v[4], v[5]);
      std::printf("%08" PRIx32 " %08" PRIx32 " %08" PRIx32 " %08" PRIx32 "\n", r.x[0], r.x[1], r.x[2], r.x[3]);
    } else if (std::strcmp(op, "u") == 0) {
      uint64_t seed, key;
      uint32_t step;
      if (std::scanf("%" SCNu64 " %" SCNu64 " %" SCNu32, &seed, &key, &step) != 3) return 2;
      const double u = sb::sample_uniform(seed, key, step);
      std::printf("%" PRIu64 "\n", static_cast<uint64_t>(u * 0x1.0p53));
    } else {
      return 2;
    }
  }
  return 0;
}
