// Non-GEMM kernels of the hot path (embedding, attention, step bookkeeping).
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
// shift=1 is the teacher-forced decoder input of the scoring pass: row r = b * T + j takes the zero embedding at j = 0
// and tokens[r - 1] after that, the inputs the decode steps 0 .. T - 1 would see.
void launch_embed(const uint32_t* tokens, const int8_t* emb_q, float inv_qm, float sqrt_e, const float* pos,
                  int rows, int T, int E, int pos_from_row, int zero_embed, float* x, QuantOuts q,
                  cudaStream_t stream, int shift = 0);

// f32 -> int8 copies (PrepareA as a standalone op, for the qmm:: operator API).
void launch_quantize(const float* x, size_t n, QuantOuts q, cudaStream_t stream);

// Encoder self-attention on unsplit [B*T][E] Q,K,V (scaled_dot_product_attention, slimt/Modules.cc:24-86,
// with split_heads/join_heads folded into the addressing).  Emits the Wo operand (int8).
int launch_self_attention(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T,
                           int H, int dh, QuantOuts q, cudaStream_t stream);

// The same operation as a register-tiled kernel (self_attention_tiled.cu): 64 query rows of one (sentence, head) per
// block, every output still one sequential chain.  Which of the self-attention kernels runs for a shape is decided in
// one place, choose_routes in engine.cu.
// Returns nonzero when the shape does not fit: head sizes 32 and 64, T up to 556 (head size 32) or 400 (64), which
// self_attention_tiled_supported tells without launching.
// Tq > 0 makes it the decoder cross-attention of the scoring pass: Q is [B][Tq][E], every row a query, against the T
// keys of K, V [B][T][E] masked by lengths; attn_head0 (optional) then receives head 0's probabilities [B][Tq][T].  The
// bound is on T alone.
int launch_self_attention_tiled(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T,
                                int H, int dh, QuantOuts q, cudaStream_t stream, int Tq = 0,
                                float* attn_head0 = nullptr);
bool self_attention_tiled_supported(int T, int dh);

// The same operation for sentences the tiled kernel cannot hold (self_attention_long.cu): 32 query rows per block, K
// and V streamed in 128-key tiles, the same chains and so the same bits.  Head sizes 32 and 64, T up to 1024.  Tq and
// attn_head0 as for the tiled kernel.
int launch_self_attention_long(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T,
                               int H, int dh, QuantOuts q, cudaStream_t stream, int Tq = 0,
                               float* attn_head0 = nullptr);
bool self_attention_long_supported(int T, int dh);

// Decoder cross-attention for one query row per sentence over cached K,V [B][S][E] (cross_attention.cu).
// mapK/mapV: f32 tensor maps over [B*S][E] with box {32 floats, cross_attention_box_rows(S)}, 128B swizzle.
// attn_head0 (optional) receives head 0's probabilities [B][S] (alignment, slimt/Model.cc:84-108).
// S <= 1024; returns nonzero for a shape it does not take (S beyond that, heads other than 8 of 32 or 64).
int cross_attention_box_rows(int S);
int launch_cross_attention(const CUtensorMap& mapK, const CUtensorMap& mapV, const float* Qr,
                            const uint32_t* lengths, int B, int S, int H, int dh, int num_sms, QuantOuts q,
                            float* attn_head0, cudaStream_t stream);

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
  QuantOuts qo;                // int8 copies of the output (Wo's operand)
  float* attn_head0;           // optional [B][T]
};
bool cross_attention_rc_supported(int E, int H, int dh, int S);
int launch_cross_attention_rc(const CrossRcArgs& a, int num_sms, bool fast, cudaStream_t stream);
// The same for long source sentences (S <= 256), one sentence at a time (cross_attention_rc.cu); bit-exact mode only.
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

// Row-wise first-max over f32 logits (used when logits are materialised for parity taps).
void launch_argmax_rows(const float* logits, int rows, int cols, unsigned long long* best, cudaStream_t stream);
// Token scores (score_partial.cuh).  launch_score_rows: the strip partials [ceil(N / 64)][B] of tap logits [B][N], or
// of the tempered logits fl32(y * inv_t) when inv_t != 1.
void launch_score_rows(const float* logits, int B, int N, float2* partials, float inv_t, cudaStream_t stream);
// One decode step's scores[step][b] = y[c] - LSE(row b) from the strip partials, c the greedy choice in best[b] or the
// column of forced[step][b] (-inf when the shortlist does not hold that word).  A forced column's logit is read from
// `logits` when given (tap route), otherwise evaluated exactly from the signed int8 operands oq [B][K] and w [N][K].
// launch_sample_step instead draws column c from the softmax of the tempered partials (sample_rng.cuh, DESIGN §4.4b),
// writes best[b] = pack_best(z[c], c) and, when scores is set, scores[step][b] = z[c] - LSE(z).
struct ScoreStepArgs {
  const float2* partials;
  unsigned long long* best;
  const uint32_t* forced;     // [max_steps][B] or null
  const uint32_t* shortlist;  // [N] sorted, or null
  const int8_t* oq;           // [B][K] signed
  const int8_t* w;            // [N][K]
  const int32_t* c127;
  const float* pb;
  const float* logits;        // [B][N] or null
  float um;
  int B, N, K, step;
  float* scores;              // [max_steps][B] (sampling: or null)
  // sampling only
  float inv_t;                // 1 / temperature
  uint64_t seed;
  const uint64_t* keys;       // [B] or null: the row index
};
int launch_score_step(const ScoreStepArgs& a, cudaStream_t stream);
int launch_sample_step(const ScoreStepArgs& a, cudaStream_t stream);
// Top-k sampling (include/slimt_b200.h, DESIGN §4.4e) over the tap logits a.logits [B][N], one block per row: the word
// is drawn from the first min(top_k, N) columns by (logit descending, column ascending), tempered, with their terms
// summed in ascending column order; best[b] = pack_best(z[c], c) and, when scores is set, scores[step][b] = z[c] -
// log-sum of the set.  Returns nonzero for top_k outside 1 .. kMaxTopK or without logits.
constexpr int kMaxTopK = 256;
int launch_topk_sample(const ScoreStepArgs& a, int top_k, cudaStream_t stream);

// Beam search (include/slimt_b200.h, DESIGN §4.4d).  Sentence b owns decoder rows b * beam + k (slot k); width[b] is
// the number of hypotheses it still has to finish (beam - finished), and its live slots are 0 .. width[b] - 1 (slot 0
// alone at step 0).
constexpr int kMaxBeam = 8;
struct BeamCand {  // one of a row's candidates: its output column and token score y[c] - LSE
  uint32_t col;
  float score;
};
struct BeamRec {  // the hypothesis a step put into a slot: its last word, the slot it extends, that word's score
  uint32_t word;
  uint32_t parent;
  float score;
};
struct BeamFin {  // a finished hypothesis: the step of its last word, the slot it extends, the word, its score, the total
  uint32_t step;
  uint32_t parent;
  uint32_t word;
  float score;
  float total;
};
struct BeamStepArgs {
  ScoreStepArgs s;                // the output layer's rows (s.B = n_sent * beam), partials and operands; s.step unused
  int beam, n_sent, step, last_step;
  BeamCand* cand;                 // [rows][beam]
  float* cum;                     // [rows] cumulative score of each live slot
  uint8_t* width;                 // [n_sent]
  BeamRec* rec;                   // [max_steps][rows]
  BeamFin* fin;                   // [n_sent][beam], in the order the hypotheses finished
  int* n_done;                    // sentences whose width reached 0
  const float* state_cur[2];      // each decoder layer's SSRU state after this step [rows][E] ...
  float* state_nxt[2];            // ... gathered by parent into the next step's state
  int Ld, E;
  uint32_t eos_id;
  const int8_t* emb_q;            // next input: embedding * sqrt(E) + position-0 signal, as finalize_step builds it
  float inv_qm, sqrt_e;
  const float* pos0;
  float* x;                       // [rows][E]
  QuantOuts q;                    // its u8 copies (layer 0's SSRU operands)
};
// Per row (32 rows per block): the row's LSE exactly as score_step forms it, the `beam` strips of largest maximum (every
// top-beam column lies in one of them), their logits re-evaluated exactly, and the row's first `beam` columns ordered by
// (logit descending, column ascending) into cand.  Rows of dead slots are skipped.
int launch_beam_topk(const BeamStepArgs& a, cudaStream_t stream);
// Per sentence (one warp): the merge of its live slots' candidates by (cum + score descending, slot ascending, rank
// ascending), the step record, finished hypotheses, the state gather and the next step's input.
int launch_beam_merge(const BeamStepArgs& a, cudaStream_t stream);
// dst[c][r] = src[r][c] for r < rows, c < cols (dst rows are dst_stride apart): step-major token matrix -> sentence-major
void launch_transpose_u32(const uint32_t* src, int rows, int cols, uint32_t* dst, int dst_stride, cudaStream_t stream);

}  // namespace sb
