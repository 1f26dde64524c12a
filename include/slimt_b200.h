/* slimt_b200.h -- C ABI of the B200-native provider for slimt's int8 hot path.
 *
 * Plain pointers and sizes only.  Every entry point names the reference
 * interface it stands in for (paths relative to the slimt tree).  All buffers
 * are HOST memory unless a name ends in _dev; the library owns device memory,
 * streams and copies.  Functions returning int return 0 on success; on failure
 * slimt_b200_last_error() describes it (shape preconditions that the reference
 * enforces with assert / SLIMT_ABORT_IF are reported this way instead of
 * aborting the caller).  There is no CPU fallback: without a CUDA device
 * slimt_b200_ctx_create fails.
 */
#ifndef SLIMT_B200_H_
#define SLIMT_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct slimt_b200_ctx slimt_b200_ctx;
typedef struct slimt_b200_model slimt_b200_model;

const char* slimt_b200_last_error(void);
const char* slimt_b200_version(void);

/* One context per GPU (device ordinal): stream, workspace arena, TMA encoder. */
int slimt_b200_ctx_create(int device, slimt_b200_ctx** out);
void slimt_b200_ctx_destroy(slimt_b200_ctx* ctx);
int slimt_b200_ctx_synchronize(slimt_b200_ctx* ctx);
/* Arithmetic mode of everything launched through the context.  0 (default): bit-exact restatement of the reference's
 * float arithmetic (results identical to slimt's CPU path with exact int32 accumulation).  1: tolerance mode
 * (FMA-contracted dequantisation, tree-reduced LayerNorm sums, ex2/rcp softmax and sigmoid, integer argmax proxy),
 * held to logits rtol 1e-3 and >= 99 % greedy token agreement instead of bit equality.  The environment variable
 * SLIMT_B200_MATH=fast sets the default of new contexts. */
int slimt_b200_ctx_set_math(slimt_b200_ctx* ctx, int fast);
int slimt_b200_ctx_get_math(const slimt_b200_ctx* ctx);

/* Device buffers and device-side timing on the context's stream, for callers
 * (bench, tests) that keep inputs resident in HBM. */
void* slimt_b200_dev_alloc(slimt_b200_ctx* ctx, size_t bytes);
void slimt_b200_dev_free(slimt_b200_ctx* ctx, void* ptr_dev);
int slimt_b200_memcpy_h2d(slimt_b200_ctx* ctx, void* dst_dev, const void* src, size_t bytes);
int slimt_b200_memcpy_d2h(slimt_b200_ctx* ctx, void* dst, const void* src_dev, size_t bytes);
int slimt_b200_timer_start(slimt_b200_ctx* ctx);          /* records a CUDA event on the stream */
int slimt_b200_timer_stop(slimt_b200_ctx* ctx, double* ms); /* records, synchronises, returns elapsed ms */
/* Writes `bytes` (> L2) of scratch on the stream so the next timed step starts with a cold L2. */
int slimt_b200_flush_l2(slimt_b200_ctx* ctx, size_t bytes);

/* ---- qmm:: operator contract (slimt/QMM.hh:48-63) -------------------------
 * "Prepared" B for this provider is simply B^T row-major: int8 [N][K], the
 * layout the model file already stores (slimt/Io.cc:227-242), immediately
 * followed in memory by the f32 b_quant when it comes from the loader. */

/* qmm::prepare_weight_quantized_transposed (QMM.hh:61; Io.cc:234): input is
 * B^T int8 [cols][rows]; output has the same logical layout. rows = K, cols = N. */
void slimt_b200_qmm_prepare_weight_quantized_transposed(const int8_t* input, int8_t* output, size_t rows,
                                                        size_t cols);

/* qmm::prepare_weight_transposed (QMM.hh:57; Io.cc:215): quantize f32 B^T
 * [rows][cols] with clamp(rne(w * quantization_multiplier), -127, 127). */
void slimt_b200_qmm_prepare_weight_transposed(const float* weights, int8_t* prepared, float quantization_multiplier,
                                              size_t cols, size_t rows);

/* qmm::affine (QMM.hh:48), qmm::dot (QMM.hh:54: bias == NULL) and
 * qmm::affine_with_select (QMM.hh:51: indices != NULL, n_indices % 8 == 0).
 *   x [M][K] f32, W prepared int8 [N][K], bias [N] or NULL, y [M][N or n_indices] f32.
 * Preconditions (intgemm's): K % 64 == 0, N % 8 == 0. */
int slimt_b200_qmm_affine(slimt_b200_ctx* ctx, const float* x, size_t M, size_t K, const int8_t* W, size_t N,
                          const float* bias, float a_quant, float b_quant, const uint32_t* indices,
                          size_t n_indices, float* y);

/* Same computation with parity taps: qa_out [M][K] receives the quantized
 * activations (the reference's PrepareA output minus 127), acc_out [M][Nout]
 * the shifted int32 accumulators sum_k (qa+127)*B exactly as Int8Shift::Multiply
 * forms them.  Either may be NULL. */
int slimt_b200_qmm_affine_debug(slimt_b200_ctx* ctx, const float* x, size_t M, size_t K, const int8_t* W, size_t N,
                                const float* bias, float a_quant, float b_quant, const uint32_t* indices,
                                size_t n_indices, float* y, int8_t* qa_out, int32_t* acc_out);

/* ---- Model contract (slimt/Model.hh:31-83, slimt/Transformer.hh:56-72) ---- */
typedef struct slimt_b200_model_config {
  int32_t encoder_layers;     /* Model::Config::encoder_layers (Model.hh:33-51) */
  int32_t decoder_layers;
  int32_t feed_forward_depth; /* must be 2 */
  int32_t num_heads;
  uint32_t eos_id;            /* Vocabulary::eos_id() (Vocabulary.hh:22): ends a sentence in record() (Model.cc:127-137) */
  uint32_t pad_id;            /* Vocabulary::pad_id() (Vocabulary.hh:23): fills the padded batch (Input.cc:20-47) */
} slimt_b200_model_config;

/* Transformer::Transformer (Transformer.cc:87-94) + io::load_items (Io.cc:114-273):
 * parses a marian binary v1 model held in host memory and uploads it. */
int slimt_b200_model_create(slimt_b200_ctx* ctx, const void* model_bin, size_t bytes,
                            const slimt_b200_model_config* config, slimt_b200_model** out);
void slimt_b200_model_destroy(slimt_b200_model* model);
/* embedding dim, ffn dim, vocabulary rows */
int slimt_b200_model_dims(const slimt_b200_model* model, int32_t* emb, int32_t* ffn, int32_t* vocab);

/* Longest sentence (source tokens, EOS included) the model accepts in slimt_b200_model_forward and in every
 * translate call; a longer one is an error ("exceeds the supported maximum of N"), never a truncation.  The reference
 * bounds segments only through the caller's wrap_length (TextProcessor::wrap, TextProcessor.cc:123-157).
 * `current` starts at 256; set_max_length raises or lowers it within [1, supported], where `supported` = 1024 is the
 * positional table's length.  n outside that range is an error and leaves the model unchanged.  Decoding runs up to
 * limit_factor x T steps, and an alignment request holds 4 * steps * B * T bytes of device workspace. */
int slimt_b200_model_set_max_length(slimt_b200_model* model, int32_t n);
int slimt_b200_model_max_length(const slimt_b200_model* model, int32_t* current, int32_t* supported);

typedef struct slimt_b200_forward_io {
  /* inputs: the padded batch of slimt::Input (Input.cc:13-63) */
  const uint32_t* tokens;   /* [B][T] row-major, padded with pad id */
  const uint32_t* lengths;  /* [B] */
  size_t batch;             /* B */
  size_t seq;               /* T */
  float limit_factor;       /* Input::limit_factor(); max steps = max(1, (size_t)(limit_factor * T)): the first decoder
                               step is unconditional (Model.cc:145-157) */
  const uint32_t* shortlist; /* Shortlist::words() (sorted, size % 8 == 0) or NULL */
  size_t n_shortlist;
  const uint32_t* forced;   /* optional teacher forcing [max_steps][B]; NULL = greedy feedback */
  int32_t device_io;        /* nonzero: tokens, lengths, shortlist, forced and step_tokens are DEVICE
                               pointers (slimt_b200_dev_alloc); no host<->device copies are made */
  /* outputs */
  uint32_t* step_tokens;    /* [max_steps][B] raw greedy choice per step (before EOS bookkeeping) */
  size_t steps;             /* out: number of decoder steps executed */
  uint64_t target_tokens;   /* out: tokens recorded by Model::decode's record() (Model.cc:127-137) */
  /* optional parity taps (NULL = skip) */
  float* encoder_out;       /* [B][T][E] */
  float* logits;            /* [max_steps][B][Nout] where Nout = n_shortlist or vocab */
  float* alignment;         /* [max_steps][B][T]: head 0 of the last layer's cross attention (Model.cc:84-108) */
} slimt_b200_forward_io;

/* Model::forward (Model.cc:187-204): embedding -> encoder -> greedy decode. */
int slimt_b200_model_forward(slimt_b200_model* model, slimt_b200_forward_io* io);

/* ---- service half on the path: Batcher + ShortlistGenerator + worker loop ----
 * Mirrors exhaust() (Frontend.cc:42-60): length-bucketed greedy batching
 * (Batcher::generate, Batcher.cc:95-120), per-batch shortlist union
 * (ShortlistGenerator::generate, Shortlist.cc:115-175) and Model::forward per
 * batch.  sentences are ragged: tokens concatenated, offsets [n+1]. */
typedef struct slimt_b200_translate_io {
  const uint32_t* tokens;
  const uint64_t* offsets;   /* [n_sentences + 1] */
  size_t n_sentences;
  size_t max_words;          /* Config::max_words (Frontend.hh:21-39) */
  float limit_factor;        /* Config::tgt_length_limit_factor */
  const void* shortlist_bin; /* lex.s2t.bin image (Shortlist.hh:78-85) or NULL */
  size_t shortlist_bytes;
  int32_t shortlist_check;   /* ShortlistGenerator's `check` (Shortlist.hh:52): verify checksum and contents at load.
                                Whatever its value, a corrupt image is an error, never an out-of-bounds access */
  int32_t shortlist_shared;  /* ShortlistGenerator's `shared` (Shortlist.cc:132-134): source words are candidates too */
  /* outputs: target sentences, ragged; capacity given by caller */
  uint32_t* out_tokens;
  size_t out_capacity;
  uint64_t* out_offsets;     /* [n_sentences + 1] */
  /* optional: Response.alignments (Model.cc:84-108, Response.hh): for sentence i, for each of its target tokens, head
   * 0 of the last decoder layer's cross-attention over the sentence's own source tokens.  Ragged: sentence i owns
   * out_alignments[out_align_offsets[i] .. out_align_offsets[i + 1]) = [target_len_i][source_len_i] floats. */
  float* out_alignments;     /* NULL = not wanted */
  size_t align_capacity;     /* floats */
  uint64_t* out_align_offsets; /* [n_sentences + 1] */
  uint64_t target_tokens;    /* out */
  uint64_t batches;          /* out */
  double device_ms;          /* out: CUDA-event time of all forward passes on the context's stream */
  uint64_t kernel_launches;  /* out: kernels this library launched during the call */
  uint64_t h2d_bytes;        /* out */
  uint64_t d2h_bytes;        /* out */
} slimt_b200_translate_io;

int slimt_b200_translate(slimt_b200_model* model, slimt_b200_translate_io* io);

/* The same request served by several replicas of one model (one per GPU, or several on one GPU) from ONE process:
 * one Batcher forms the batches, and every replica's worker thread takes the next unserved batch as soon as it is
 * free -- Async's workers pulling from the batcher queue (Frontend.cc:207-227, Batcher.hh:203-259).  Sentences are
 * independent and every batch is the one the Batcher would have formed anyway, so the output is identical to
 * slimt_b200_translate's; there is no collective on the data path.  device_ms = the longest replica's time.
 * The length bound is the smallest slimt_b200_model_max_length current over the replicas. */
int slimt_b200_translate_multi(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io);

/* Host-only pieces of the same path, callable without a GPU (used by the CPU test-suite):
 * ShortlistGenerator::generate (Shortlist.cc:115-175) and Batcher::generate (Batcher.cc:95-120). */
int slimt_b200_shortlist_generate(const void* shortlist_bin, size_t shortlist_bytes, const uint32_t* words,
                                  size_t n_words, size_t vocab, uint32_t* out, size_t out_capacity, size_t* n_out);
/* ShortlistGenerator::load with check = true (Shortlist.cc:41-98, 16-37): header, size, checksum, content_check. */
int slimt_b200_shortlist_check(const void* shortlist_bin, size_t shortlist_bytes, size_t vocab);
/* Writes sentence ids batch by batch into batch_ids [n] and the batch boundaries into
 * batch_offsets [n_batches + 1] (capacity n + 1); widths [n_batches] receives each padded length. */
int slimt_b200_batcher_plan(const uint64_t* lengths, size_t n, size_t max_words, uint64_t* batch_ids,
                            uint64_t* batch_offsets, uint64_t* widths, size_t* n_batches);

/* counters since context creation (bench.py reports gpu_launches from these) */
uint64_t slimt_b200_kernel_launches(const slimt_b200_ctx* ctx);

/* Per-kernel device timing: while enabled every launch on the context's stream is bracketed by
 * CUDA events.  read() synchronises and aggregates by kernel tag, then clears the log. */
typedef struct slimt_b200_kernel_stat {
  char name[48];
  uint64_t launches;
  double ms;     /* sum of event-timed durations */
  double ops;    /* algorithmic int8 operations (2*MAC) summed over launches */
  double bytes;  /* algorithmic HBM bytes summed over launches */
} slimt_b200_kernel_stat;
int slimt_b200_profile_enable(slimt_b200_ctx* ctx, int on);
int slimt_b200_profile_read(slimt_b200_ctx* ctx, slimt_b200_kernel_stat* out, size_t capacity, size_t* n_out);

#ifdef __cplusplus
}
#endif
#endif /* SLIMT_B200_H_ */
