// The one reduction order of a token score (log-probability), shared by every route that produces one.
//
// score[s][b] = y[c] - log sum_n exp(y[n]) over the step's output columns n (the shortlist's, or the vocabulary's).
// The columns are cut into 64-column strips; a strip's logits reduce to a partial (m, s) = (max_j y_j,
// sum_j exp(y_j - m)) with strip_partial below, and the partials of a row are combined in ascending strip order by
// combine_partials.  Both the fused output GEMM's scores epilogue (out_argmax.cu) and the row kernel over the logits
// tap call strip_partial on the same 64 values, so the two routes give the same bits; nothing in either order depends
// on which CTA evaluated a strip, on the grid size or on the running greedy state.
#pragma once
#include <stdint.h>

#include <cuda_runtime.h>

namespace sb {

constexpr int kScoreStrip = 64;  // columns per partial

// exp(x) for x <= 0 through the SFU: ex2.approx.ftz (relative error < 2^-22) of one rounded product.  exp(-inf) = 0.
__device__ __forceinline__ float score_exp(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(__fmul_rn(x, 1.4426950408889634f)));
  return e;
}

// (m, s) of one strip: y0 = columns 0..31, y1 = columns 32..63; a column past N holds -inf and adds nothing.  The strip
// holds at least one finite column (N % 8 == 0 and the strip starts below N).  Order: the maximum (exact in any order),
// then eight sequential sums of eight consecutive columns, then the pairwise tree (0+1)+(2+3), (4+5)+(6+7).
__device__ __forceinline__ float2 strip_partial(const float (&y0)[32], const float (&y1)[32]) {
  float t[8];
#pragma unroll
  for (int k = 0; k < 4; k++) {
    t[k] = fmaxf(fmaxf(fmaxf(y0[8 * k], y0[8 * k + 1]), fmaxf(y0[8 * k + 2], y0[8 * k + 3])),
                 fmaxf(fmaxf(y0[8 * k + 4], y0[8 * k + 5]), fmaxf(y0[8 * k + 6], y0[8 * k + 7])));
    t[4 + k] = fmaxf(fmaxf(fmaxf(y1[8 * k], y1[8 * k + 1]), fmaxf(y1[8 * k + 2], y1[8 * k + 3])),
                     fmaxf(fmaxf(y1[8 * k + 4], y1[8 * k + 5]), fmaxf(y1[8 * k + 6], y1[8 * k + 7])));
  }
  const float m = fmaxf(fmaxf(fmaxf(t[0], t[1]), fmaxf(t[2], t[3])), fmaxf(fmaxf(t[4], t[5]), fmaxf(t[6], t[7])));
#pragma unroll
  for (int k = 0; k < 4; k++) {
    float a = 0.0f, b = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      a = __fadd_rn(a, score_exp(__fsub_rn(y0[8 * k + j], m)));
      b = __fadd_rn(b, score_exp(__fsub_rn(y1[8 * k + j], m)));
    }
    t[k] = a, t[4 + k] = b;
  }
  const float s = __fadd_rn(__fadd_rn(__fadd_rn(t[0], t[1]), __fadd_rn(t[2], t[3])),
                            __fadd_rn(__fadd_rn(t[4], t[5]), __fadd_rn(t[6], t[7])));
  return make_float2(m, s);
}

// Sampling at a temperature other than 1 (DESIGN §4.4b): the strip's tempered logits z = fl32(y * inv_t), in place.
// inv_t > 0, so -inf stays -inf.
__device__ __forceinline__ void temper64(float (&y0)[32], float (&y1)[32], float inv_t) {
#pragma unroll
  for (int j = 0; j < 32; j++) y0[j] = __fmul_rn(y0[j], inv_t), y1[j] = __fmul_rn(y1[j], inv_t);
}

}  // namespace sb
