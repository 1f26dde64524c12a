// Output projection fused with the greedy argmax (out_argmax.cu): [M rows] x [N vocabulary or shortlist columns],
// K = E, each row's choice published into a packed best word (packed_best.cuh).
//
// The column-dependent part of a logit reaches the kernel in one of two encodings, chosen per model at load:
//   digits        each column's offset round(c127 + pb / um) rides through the tensor core as 32 int8 digits, an extra
//                 K = 32 block; they hold |offset| <= 500 093;
//   bound filter  for a model whose offsets exceed that: a per-32-column float upper bound (dmax, eta) decides which
//                 chunks are evaluated exactly.
// A subset of a model's columns (the shortlist) fits the model's encoding and its eta.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

namespace sb {

constexpr int kOutBN = 256;  // columns per output tile; the per-column tables are read by whole tiles

// One set of output columns and what the fused argmax reads of them: the model's vocabulary, or a shortlist's
// gathered copy.
struct OutColumns {
  int N = 0;
  float um = 0;              // 1 / (aq * bq) of the output layer
  int8_t* w = nullptr;       // [N][K] s8 weights
  float* pb = nullptr;       // [N] prepared bias
  int32_t* c127 = nullptr;   // [N] 127 * colsum
  CUtensorMap map_w;         // w with box {128 B, 256 rows}
  bool digits = false;       // the encoding: digits, or the bound filter
  uint8_t* ext = nullptr;    // digits: [pad(N)][128] rows of 32 digits
  int32_t* dshift = nullptr; // digits: [pad(N)] c127 - offset: proxy -> shifted accumulator
  CUtensorMap map_ext;       // ext with box {128 B, 256 rows}
  float* dmax = nullptr;     // bound filter: [ceil(N/32)] per-chunk max of c127 * um + pb, rounded up
  float eta = 0;             // bound filter: slack covering the float roundings of the exact formula

  static size_t pad(int n) { return (static_cast<size_t>(n) + kOutBN - 1) / kOutBN * kOutBN; }
  // The tables of this encoding for N columns, as add(pointer slot, element count): the model loader and the
  // workspace plan both allocate them from here.
  template <class Add>
  void tables(Add&& add) {
    if (digits) {
      add(ext, 128 * pad(N));
      add(dshift, pad(N));
    } else {
      add(dmax, (static_cast<size_t>(N) + 31) / 32);
    }
  }
};

// Fills the tables of c's encoding from c.c127, c.pb and c.um.  overflow (digits only, optional, device int,
// pre-zeroed) is set when some column's offset does not fit the digits.
void launch_out_tables(const OutColumns& c, int* overflow, cudaStream_t stream);

// best[M] (pre-zeroed, packed_best.cuh) receives each row's first maximum over c's columns of the logits of the s8
// activations in tma_a ([M][K], box {128 B, 128 rows}).  fast selects tolerance mode, which on the digits takes the
// integer proxy as the score; the bound filter always gives the exact first maximum of the float logits.  Returns
// nonzero for an unsupported K (128 * {2, 4} are built).
int launch_out_argmax(const OutColumns& c, const CUtensorMap& tma_a, bool fast, int M, int K, unsigned long long* best,
                      int num_sms, cudaStream_t stream);

// The same GEMM with the scores epilogue, in either encoding and arithmetic mode (it reads c.w, c.pb, c.c127 and
// c.map_w, none of the encoding's tables): every logit is evaluated exactly, best[M] (pre-zeroed) receives each row's
// first maximum of them, and partials[ceil(N / 64)][M] each 64-column strip's (max, sum of exp) in the order of
// score_partial.cuh.  inv_t != 1: the partials (and the maximum) are of the tempered logits fl32(y * inv_t), for
// sampling.  Returns nonzero for an unsupported K.
int launch_out_scores(const OutColumns& c, const CUtensorMap& tma_a, int M, int K, unsigned long long* best,
                      float2* partials, float inv_t, int num_sms, cudaStream_t stream);

}  // namespace sb
