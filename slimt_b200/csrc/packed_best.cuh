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

// The vocabulary word of a packed candidate: its column, through the shortlist when one is given.
__device__ __forceinline__ uint32_t best_word(unsigned long long packed, const uint32_t* shortlist) {
  const uint32_t idx = best_index(packed);
  return shortlist ? shortlist[idx] : idx;
}

// record() (slimt/Model.cc:127-137) of row b's word at one step, then re-arm the row's packed best.  The word is
// written to step_tokens; a row not yet finished grows by one and finishes at EOS.  was_done and len_before are
// done[b] and tgt_len[b] as the caller loaded them: this helper loads nothing, so a caller can issue those loads early
// and run the record off its critical path.
__device__ __forceinline__ void record_word(uint32_t word, uint32_t was_done, uint32_t len_before, uint32_t eos_id,
                                            int step, int B, int b, uint32_t* step_tokens, uint8_t* done,
                                            uint32_t* tgt_len, int* n_done, unsigned long long* best) {
  step_tokens[static_cast<size_t>(step) * B + b] = word;
  if (!was_done) {
    tgt_len[b] = len_before + 1;
    if (word == eos_id) {
      done[b] = 1;
      atomicAdd(n_done, 1);
    }
  }
  best[b] = 0ull;
}

}  // namespace sb
