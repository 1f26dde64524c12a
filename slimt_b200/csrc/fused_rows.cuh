// Row-tile fused kernels of the decoder step (fused_rows.cu).
//
// A decoder step is row-local: every sentence's row goes through the same chain of small GEMMs
// (K = 256/1536) with LayerNorm / ReLU / highway epilogues in between (reference DecoderLayer::forward,
// slimt/Modules.cc:237-259; SSRU::forward :190-235; FFN :277-280).  Launching them one by one leaves the
// GPU latency-bound (28 rows per SM at B = 4096).  Here one CTA owns a tile of 32 rows and walks the whole
// chain with the activations resident in shared memory: the WEIGHTS are the MMA's A operand (128 output
// features per tcgen05.mma, streamed from L2 by TMA), the tile's u8 activations are the B operand
// (N = 32), int32 accumulators sit in TMEM with output features on the lanes, and each epilogue writes the
// next GEMM's operand straight back into shared memory in the UMMA 128B-swizzled K-major layout.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sb {

constexpr int kRowTile = 32;

// Attention output projection + residual + LayerNorm, then the feed-forward block with its own residual +
// LayerNorm (encoder and decoder layers):  y = LN1(res + Wo a + bo);  z = LN2(y + W2 relu(W1 y + b1) + b2).
struct RowsFfnArgs {
  CUtensorMap map_a;                   // u8 [M][E], box {128 B, rows_per_tile}: attention output quantised with Wo's a_quant
  CUtensorMap map_wo, map_w1, map_w2;  // s8 weights [N][K], box {128 B, 128 rows}
  const float* pb_o;                   // prepared biases (Int8Shift::PrepareBias, precomputed at load)
  const float* pb_1;
  const float* pb_2;
  float um_o, um_1, um_2;              // 1 / (a_quant * b_quant)
  float aq_1, aq_2;                    // a_quant of W1 (quantises y) and W2 (quantises relu(W1 y + b1))
  const float* res;                    // residual of the attention block, f32 [M][E]
  const float* ln1_scale;
  const float* ln1_bias;
  const float* ln2_scale;
  const float* ln2_bias;
  float eps;
  float* y_park;                       // f32 [M][E] scratch for y, required when rows_per_tile == 128
  float* z_out;                        // f32 [M][E] or null
  uint8_t* zq[4];                      // quantised copies of z for the consumers (next layer's projections, output layer)
  float zaq[4];
  int n_zq;
  int zq_signed;                       // bit k: zq[k] receives the signed value instead of u8 = q + 127
  int M;
};

// SSRU cell + query projection:  c = sigmoid(Wf x + bf) * c_prev + (1 - sigmoid(.)) * (W x);
// h = LN(x + relu(c));  q = Wq h + bq.
struct DecSsruArgs {
  CUtensorMap map_xf, map_xw;          // u8 [M][E], box {128 B, 32 rows}: x quantised with Wf's / W's a_quant
  CUtensorMap map_wf, map_w, map_wq;   // s8 weights
  const float* pb_f;
  const float* pb_w;
  const float* pb_q;
  float um_f, um_w, um_q;
  float aq_q;                          // a_quant of Wq (quantises h)
  const float* x;                      // f32 [M][E]
  float* state;                        // f32 [M][E], read and overwritten with c
  const float* ln_scale;
  const float* ln_bias;
  float eps;
  float* h_out;                        // f32 [M][E]
  float* q_out;                        // f32 [M][E]
  int M;
  // ---- layer 0 from the second step on (embed != 0): the kernel's front does what finalize_step_kernel does for the
  // PREVIOUS step -- packed argmax -> word id (through the shortlist), record into step_tokens[prev_step][M], EOS
  // bookkeeping (Model.cc:127-137), re-arm `best` -- and builds this step's input from the word's embedding row
  // (* sqrt(E) + position-0 signal; quirk Q1) straight into the operand tiles: x, map_xf and map_xw are then unused.
  int embed;
  int prev_step;
  unsigned long long* best;
  const uint32_t* shortlist;           // or null
  const uint32_t* forced;              // teacher forcing [steps][M] or null
  uint32_t* step_tokens;
  uint8_t* done;
  uint32_t* tgt_len;
  int* n_done;
  uint32_t eos_id;
  const int8_t* emb_q;                 // stored embedding [V][E]
  float inv_qm, sqrt_e;
  const float* pos0;                   // position-0 signal [E]
  float aq_xf, aq_xw;                  // a_quant of Wf / W (quantise x)
};

// The SSRU cell of the scoring pass, where every decoder input of a sentence is known before the first position: the
// projections Wf x + bf and W x of all B * T rows come from one GEMM, and this kernel runs what remains sequential --
// c_j = sg_j * c_{j-1} + (1 - sg_j) * (W x)_j from c_{-1} = 0 -- then h = LN(x + relu(c)) and h's u8 copy for Wq.  Rows
// are b * T + j; the arithmetic is dec_ssru_kernel's bit-exact branch, so each row equals the step path's row at step j.
struct DecSsruScanArgs {
  const float* f;                      // f32 [B * T][E]: Wf x + bf
  const float* wx;                     // f32 [B * T][E]: W x
  const float* x;                      // f32 [B * T][E]: the layer's input
  const float* ln_scale;
  const float* ln_bias;
  float eps;
  float aq_q;                          // a_quant of Wq (quantises h)
  float* h_out;                        // f32 [B * T][E]
  uint8_t* hq;                         // u8 [B * T][E]
  int B, T;
};

// E = 256, F = 1536 (tiny) and E = 512, F = 2048 (base) are built.  Returns nonzero when unsupported.
// rows_per_tile: 32 (decoder step) or 128 (encoder; E = 256 only).
int launch_rows_ffn(const RowsFfnArgs& a, int E, int F, int rows_per_tile, bool fast, cudaStream_t stream);
int launch_dec_ssru(const DecSsruArgs& a, int E, bool fast, cudaStream_t stream);
int launch_dec_ssru_scan(const DecSsruScanArgs& a, int E, cudaStream_t stream);

}  // namespace sb
