// Non-GEMM kernels of the hot path (embedding, attention, SSRU, step bookkeeping).
// Each one reproduces the reference's f32 arithmetic bit for bit (see
// exact_math.cuh) while emitting the int8 operands of the GEMMs that consume it.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sb {

constexpr int kMaxQ = 4;

struct QuantOuts {
  int8_t* ptr[kMaxQ];
  float aq[kMaxQ];
  int n;
};

// x[r] = float(emb_q[tok[r]]) * inv_qm * sqrt_e + pos[(r % T) or 0]   (index_select + transform_embedding,
// slimt/TensorOps.cc:227-243, Transformer.cc:24-49, Io.cc:275-283).  zero_embed=1 is decoder step 0.
void launch_embed(const uint32_t* tokens, const int8_t* emb_q, float inv_qm, float sqrt_e, const float* pos,
                  int rows, int T, int E, int pos_from_row, int zero_embed, float* x, QuantOuts q,
                  cudaStream_t stream);

// f32 -> int8 copies (PrepareA as a standalone op, for the qmm:: operator API).
void launch_quantize(const float* x, size_t n, QuantOuts q, cudaStream_t stream);

// Encoder self-attention on unsplit [B*T][E] Q,K,V (scaled_dot_product_attention, slimt/Modules.cc:24-86,
// with split_heads/join_heads folded into the addressing).  Emits the Wo operand (int8) and/or f32.
int launch_self_attention(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T,
                           int H, int dh, float* out_f32, QuantOuts q, cudaStream_t stream);

// The same operation as a register-tiled kernel (self_attention_tiled.cu): 64 query rows of one (sentence, head) per
// block, every output still one sequential chain.  The default for every shape the fused encoder kernel does not take.
// Returns nonzero when the shape does not fit: head sizes 32 and 64, T up to 556 (head size 32) or 400 (64), which
// self_attention_tiled_supported tells without launching.
int launch_self_attention_tiled(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T,
                                int H, int dh, float* out_f32, QuantOuts q, cudaStream_t stream);
bool self_attention_tiled_supported(int T, int dh);

// The same operation for sentences the tiled kernel cannot hold (self_attention_long.cu): 32 query rows per block, K
// and V streamed in 128-key tiles, the same chains and so the same bits.  Head sizes 32 and 64, T up to 1024.
int launch_self_attention_long(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T,
                               int H, int dh, float* out_f32, QuantOuts q, cudaStream_t stream);
bool self_attention_long_supported(int T, int dh);

// Decoder cross-attention for one query row per sentence over cached K,V [B][S][E] (cross_attention.cu).
// mapK/mapV: f32 tensor maps over [B*S][E] with box {32 floats, cross_attention_box_rows(S)}, 128B swizzle.
// attn_head0 (optional) receives head 0's probabilities [B][S] (alignment, slimt/Model.cc:84-108).
// S <= 1024; returns nonzero for a shape it does not take (S beyond that, heads other than 8 of 32 or 64).
int cross_attention_box_rows(int S);
int launch_cross_attention(const CUtensorMap& mapK, const CUtensorMap& mapV, const float* Qr,
                            const uint32_t* lengths, int B, int S, int H, int dh, int num_sms, float* out_f32,
                            QuantOuts q, float* attn_head0, cudaStream_t stream);

// The same attention with K and V re-projected from the quantised encoder output on the tensor cores every step
// instead of read from an f32 cache (cross_attention_rc.cu): 4x less HBM traffic, bit-identical results.
struct CrossRcArgs {
  CUtensorMap map_ak, map_av;  // u8 [B*S][E], box {128 B, 32 rows}: encoder output quantised with Wk's / Wv's a_quant
  CUtensorMap map_wk, map_wv;  // s8 [E][E], box {128 B, 128 rows}
  const float* pb_k;           // prepared biases
  const float* pb_v;
  float um_k, um_v;            // 1 / (a_quant * b_quant)
  const float* q;              // f32 [B][E]
  const uint32_t* lengths;
  int B, T;
  float dk;                    // 1 / sqrt(head size)
  float* out_f32;              // optional f32 [B][E]
  QuantOuts qo;                // int8 copies of the output (Wo's operand)
  float* attn_head0;           // optional [B][T]
  long long* trace;            // optional phase stamps (clock64) of consumer thread 0, 128 slots per CTA (SLIMT_B200_TRACE)
};
bool cross_attention_rc_supported(int E, int H, int dh, int S);
int launch_cross_attention_rc(const CrossRcArgs& a, int num_sms, bool fast, cudaStream_t stream);
// The same for long source sentences (S <= 256), one sentence at a time (cross_attention_rcl.cu); bit-exact mode only.
bool cross_attention_rcl_supported(int E, int H, int dh, int S);
int launch_cross_attention_rcl(const CrossRcArgs& a, int num_sms, cudaStream_t stream);

// Encoder self-attention fused with its q/k/v projections (enc_attention.cu): Q, K and V never reach HBM.
// Bit-identical to launch_gemm_i8(EPI_F32) x 3 followed by launch_self_attention.
struct EncAttnArgs {
  CUtensorMap map_aq, map_ak, map_av;  // u8 [B*T][E], box {128 B, 128 rows}: x quantised with Wq's / Wk's / Wv's a_quant
  CUtensorMap map_aq32, map_ak32, map_av32;  // the same tensors with box {128 B, 32 rows} (T <= 32: a box per sentence)
  CUtensorMap map_wq, map_wk, map_wv;  // s8 [E][E], box {128 B, 32 rows}
  const float* pb_q;                   // prepared biases
  const float* pb_k;
  const float* pb_v;
  float um_q, um_k, um_v;              // 1 / (a_quant * b_quant)
  const uint32_t* lengths;
  int B, T;
  float dk;                            // 1 / sqrt(head size)
  uint8_t* out_q;                      // u8 [B*T][E]: Wo's operand
  float aq_out;
};
bool enc_attention_supported(int E, int H, int dh, int T);
int launch_enc_attention(const EncAttnArgs& a, int num_sms, cudaStream_t stream);

// SSRU cell tail (slimt/Modules.cc:190-235): c = highway(c_prev, Wx, f); h = LN(x + relu(c)); state <- c.
void launch_ssru_ln(const float* f, const float* wx, float* state, const float* x, const float* ln_scale,
                    const float* ln_bias, float eps, int B, int E, float* h, QuantOuts q, cudaStream_t stream);

// Per decode step: packed argmax -> word id (through the shortlist when given), record into
// step_tokens[step][B], EOS bookkeeping, re-arm `best`, and build the next step's decoder input
// (embedding * sqrt(E) + position-0 signal; quirk Q1) with its int8 copies.
void launch_finalize_step(unsigned long long* best, const uint32_t* shortlist, const uint32_t* forced, int step,
                          uint32_t* step_tokens, uint8_t* done, uint32_t* tgt_len, int* n_done, uint32_t eos_id,
                          const int8_t* emb_q, float inv_qm, float sqrt_e, const float* pos0, int B, int E, float* x,
                          QuantOuts q, cudaStream_t stream);

// Shortlist: gather rows of the output weight and its prepared bias / shift terms.
// c127 / c127_sel (127 * column sums, used by the fused output GEMM's bound filter) may be null.
void launch_gather_rows(const int8_t* W, const float* pb, const int32_t* c127, const uint32_t* idx, int n_idx, int K,
                        int8_t* W_sel, float* pb_sel, int32_t* c127_sel, cudaStream_t stream);

// dmax[ceil(N/32)]: per 32-column chunk, max_n(c127[n] * um + pb[n]) rounded up (see gemm_out.cu).
void launch_out_bounds(const int32_t* c127, const float* pb, float um, int N, float* dmax, cudaStream_t stream);

// ipb6[ceil(N/256)*256]: integer logit-proxy offsets of the tolerance-mode output GEMM (see gemm_out.cu).
void launch_out_ipb(const int32_t* c127, const float* pb, float um, int N, int32_t* ipb6, cudaStream_t stream);

// Digit rows ext [ceil(N/256)*256][128] and dshift [same] of the second-generation output GEMM (gemm_out_ext.cu);
// *overflow (device int, pre-zeroed) is set when a column's offset does not fit the digits.
void launch_out_ext(const int32_t* c127, const float* pb, float um, int N, uint8_t* ext, int32_t* dshift, int* overflow,
                    cudaStream_t stream);

// Row-wise first-max over f32 logits (used when logits are materialised for parity taps).
void launch_argmax_rows(const float* logits, int rows, int cols, unsigned long long* best, cudaStream_t stream);
// dst[c][r] = src[r][c] for r < rows, c < cols (dst rows are dst_stride apart): step-major token matrix -> sentence-major
void launch_transpose_u32(const uint32_t* src, int rows, int cols, uint32_t* dst, int dst_stride, cudaStream_t stream);

}  // namespace sb
