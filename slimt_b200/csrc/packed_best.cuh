// The greedy choice of one output row as a single 64-bit word that atomicMax can raise from any thread of any CTA:
// (order-preserving 32-bit key of the score << 32) | (0xFFFFFFFF - column).  A larger score wins; between equal scores
// the lower column wins, which is the reference's first strict maximum (greedy_sample, slimt/Transformer.cc:279-339).
// The zero word is below every packed candidate, so a zeroed row means "nothing seen yet".
//
// The score is a float logit (exact mode and the logits tap) or the output GEMM's integer proxy (tolerance mode on the
// digit encoding, out_argmax.cu); the column is an index into the vocabulary or the shortlist.
#pragma once
#include <stdint.h>

namespace sb {

__device__ __forceinline__ unsigned long long pack_best_key(uint32_t key, uint32_t idx) {
  return (static_cast<unsigned long long>(key) << 32) | static_cast<unsigned long long>(0xFFFFFFFFu - idx);
}

__device__ __forceinline__ unsigned long long pack_best(float v, uint32_t idx) {
  if (v == 0.0f) v = 0.0f;  // canonicalise -0 so equal values compare equal
  const uint32_t b = __float_as_uint(v);
  return pack_best_key((b & 0x80000000u) ? ~b : (b | 0x80000000u), idx);
}

__device__ __forceinline__ unsigned long long pack_best_proxy(int v, uint32_t idx) {
  return pack_best_key(static_cast<uint32_t>(v) ^ 0x80000000u, idx);
}

__device__ __forceinline__ uint32_t best_index(unsigned long long packed) {
  return 0xFFFFFFFFu - static_cast<uint32_t>(packed & 0xFFFFFFFFull);
}

// The score of a packed float candidate (not of the zero word).
__device__ __forceinline__ float best_value(unsigned long long packed) {
  const uint32_t key = static_cast<uint32_t>(packed >> 32);
  return __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
}

// The score of a packed proxy candidate (not of the zero word).
__device__ __forceinline__ int best_proxy(unsigned long long packed) {
  return static_cast<int>(static_cast<uint32_t>(packed >> 32) ^ 0x80000000u);
}

}  // namespace sb
