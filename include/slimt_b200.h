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
  /* optional result (NULL = not wanted): log-probability of each step's word, y[c] - log sum_n exp(y[n]) over the step's
   * logits y (the shortlist's columns, or the vocabulary's), c the greedy choice or the forced word's column (-inf when
   * the shortlist does not hold it).  Every executed step has one, like step_tokens.  A DEVICE pointer with device_io. */
  float* token_scores;      /* [max_steps][B] */
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
  /* optional (NULL = not wanted): the log-probability of every recorded target token, EOS included (token_scores of
   * slimt_b200_forward_io).  Ragged exactly like out_tokens: indexed by out_offsets, capacity out_capacity. */
  float* out_scores;
} slimt_b200_translate_io;

int slimt_b200_translate(slimt_b200_model* model, slimt_b200_translate_io* io);

/* The same request served by several replicas of one model (one per GPU, or several on one GPU) from ONE process:
 * one Batcher forms the batches, and every replica's worker thread takes the next unserved batch as soon as it is
 * free -- Async's workers pulling from the batcher queue (Frontend.cc:207-227, Batcher.hh:203-259).  Sentences are
 * independent and every batch is the one the Batcher would have formed anyway, so the output is identical to
 * slimt_b200_translate's; there is no collective on the data path.  device_ms = the longest replica's time.
 * The length bound is the smallest slimt_b200_model_max_length current over the replicas. */
int slimt_b200_translate_multi(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io);

/* ---- sampling: each step's word drawn from the model's distribution instead of chosen greedily ----
 * For decode step s and row b, with y[n] the step's exact logits over the output columns (the shortlist's or the
 * vocabulary's: the values of the logits tap):
 *  - tempered logits z[n] = fl32(y[n] * inv_t), inv_t = (float)(1.0 / (double)temperature); at temperature 1, z = y.
 *  - (x0, x1, x2, x3) = Philox4x32-10(counter = (s, key_lo, key_hi, 0), key = (seed_lo, seed_hi)) and
 *    u = ((((uint64)x0 << 32) | x1) >> 11) * 2^-53 in [0, 1), with `key` the row's sampling key.
 *  - the word is the first column c, in ascending order, whose cumulative probability sum_{j<=c} exp(z[j] - LSE(z))
 *    exceeds u, summed in the order of the token scores (64-column strips, their groups, then the strip's columns); a
 *    column whose term underflows to 0 is never chosen.
 *  - the sampled word replaces the greedy choice: EOS handling, recorded tokens and alignments follow it unchanged.
 *    token_scores / out_scores, when asked for, hold z[c] - LSE(z), the word's log-probability under the distribution
 *    it was drawn from (at temperature 1 exactly the greedy call's score definition).
 * Both arithmetic modes draw from the same exact logits.  A temperature that is not finite or lies outside [1e-3, 1e3],
 * or sampling together with `forced`, is an error; the model stays usable. */
typedef struct slimt_b200_sampling {
  float temperature;     /* finite, in [1e-3, 1e3] */
  uint64_t seed;
  const uint64_t* keys;  /* one per row (forward; a DEVICE pointer with device_io) or per sentence (translate);
                            NULL = the row's index in the batch (forward) or the sentence's index in the request
                            (translate), so a translation never depends on which batch, lane or replica served it */
} slimt_b200_sampling;
/* slimt_b200_model_forward / slimt_b200_translate_multi with sampling; sampling = NULL is the greedy call. */
int slimt_b200_model_forward_sampled(slimt_b200_model* model, slimt_b200_forward_io* io,
                                     const slimt_b200_sampling* sampling);
int slimt_b200_translate_sampled(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io,
                                 const slimt_b200_sampling* sampling);

/* ---- top-k sampling: each step's word drawn from the k most likely columns only (marian's --output-sampling topk) ----
 * For decode step s and row b, with y[n] the step's exact logits over the N output columns (as for sampling above) and
 * k = top_k:
 *  - the set S_k is the first min(k, N) columns ordered by (y descending, column ascending): ties go to the lower
 *    column, so S_1 is the greedy choice.
 *  - z[n] = fl32(y[n] * inv_t) as above; M = max z over S_k; each column c of S_k has the term
 *    e_c = exp(z[c] - M), evaluated as the token scores evaluate it (ex2.approx of one rounded product), and S is the
 *    sum of the terms in ascending column order, in double.
 *  - u as above (the same Philox stream, keys and defaults); the word is the first column of S_k, in ascending column
 *    order, whose running sum exceeds u * S.  A zero term is never chosen; if rounding exhausts the set, the last
 *    column with a nonzero term is taken.
 *  - token_scores / out_scores, when asked for, hold (float)((double)z[c] - ((double)M + log S)): the word's
 *    log-probability under the distribution it was drawn from (slimt_b200_score gives the full-vocabulary one).
 *  - everything after the draw is as for sampling: EOS handling, recorded tokens, alignments, the step limit, batching.
 * k = 1 is greedy decoding in the bit-exact arithmetic, with every score 0; k >= N draws from every column.  Both
 * arithmetic modes draw from the step's exact logits.  Errors, each reported before any GPU work (the model stays
 * usable): top_k < 0 or > 256; top_k > 0 with sampling = NULL; and sampling's own errors (temperature, `forced`).
 * top_k = 0 is the _sampled call.
 * Device workspace: with top_k > 0 every step's logits are materialised, 4 * B * N bytes per batch (N the shortlist's
 * or the vocabulary's width). */
int slimt_b200_model_forward_topk(slimt_b200_model* model, slimt_b200_forward_io* io,
                                  const slimt_b200_sampling* sampling, int32_t top_k);
int slimt_b200_translate_topk(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io,
                              const slimt_b200_sampling* sampling, int32_t top_k);

/* ---- scoring: the log-probability of each word of a GIVEN translation ----
 * For sentence pair i (source tokens[offsets[i] .. offsets[i + 1]), EOS included, non-empty; target
 * targets[target_offsets[i] .. target_offsets[i + 1]), any length including 0) and each target position j, the score of
 * t_j is y[c] - log sum_n exp(y[n]), where
 *  - y is the logits of the decoder fed the zero embedding at j = 0 and t_{j-1} after that -- the decode steps' own
 *    inputs, the position-0 signal included at every step (Transformer.cc:133-160) -- so exactly the token_scores that
 *    slimt_b200_model_forward returns at step j with forced = the target;
 *  - c is t_j's column: over the vocabulary, or over the batch's shortlist when one is given (a word outside the
 *    shortlist scores -inf).
 * Every given token is scored: EOS is a word like any other, scoring neither stops at it nor requires it, and no
 * limit_factor applies.  Scoring the out_tokens of slimt_b200_translate (EOS included) reproduces its out_scores, and
 * out_alignments, bit for bit: the sentences form the same batches (the Batcher over the source lengths) and so the same
 * shortlist unions.
 * Arithmetic: scoring always runs the bit-exact arithmetic, whatever slimt_b200_ctx_set_math says; reproducible numbers
 * are what reranking, filtering and quality estimation need.
 * Errors, each reported before any GPU work (the model stays usable): offsets that decrease; a target word >= the
 * vocabulary size; a source or target longer than the smallest slimt_b200_model_max_length current over the replicas;
 * an output capacity too small.
 * Device workspace: about 25 * E bytes per target position of a batch (the longest target times the batch's sentences),
 * plus 4 * source width per position with alignments. */
typedef struct slimt_b200_score_io {
  const uint32_t* tokens;          /* sources, ragged like slimt_b200_translate_io */
  const uint64_t* offsets;         /* [n_sentences + 1] */
  size_t n_sentences;
  const uint32_t* targets;         /* targets, ragged */
  const uint64_t* target_offsets;  /* [n_sentences + 1] */
  size_t max_words;                /* Config::max_words: batches are formed over the source lengths */
  const void* shortlist_bin;       /* as in slimt_b200_translate_io */
  size_t shortlist_bytes;
  int32_t shortlist_check;
  int32_t shortlist_shared;
  /* outputs */
  float* out_scores;               /* ragged by target_offsets (rebased to 0) */
  size_t out_capacity;             /* floats; at least the total number of target tokens */
  /* optional (NULL = not wanted): head 0 of the last decoder layer's cross-attention, [target_len_i][source_len_i]
   * floats for sentence i at out_alignments[out_align_offsets[i] ..), as in slimt_b200_translate_io */
  float* out_alignments;
  size_t align_capacity;           /* floats */
  uint64_t* out_align_offsets;     /* [n_sentences + 1] */
  uint64_t batches;                /* out */
  double device_ms;                /* out: CUDA-event time of the passes (the longest replica's) */
  uint64_t kernel_launches;        /* out */
  uint64_t h2d_bytes;              /* out */
  uint64_t d2h_bytes;              /* out */
} slimt_b200_score_io;

/* Scores io's targets with one or more replicas of one model (as slimt_b200_translate_multi serves a request). */
int slimt_b200_score(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_score_io* io);

/* ---- beam search: K hypotheses per sentence instead of one (marian's --beam-size, --n-best, --normalize) ----
 * The batches are slimt_b200_translate's (the Batcher over the source lengths), so the shortlist unions and the step
 * limit max_steps = max(1, (size_t)(limit_factor * width)) are greedy's.  Sentence b's slots are its decoder rows
 * b * K + k; it starts with one live slot (slot 0) holding the empty hypothesis with cumulative score cum = 0, and a
 * width w = K of hypotheses still to finish.  At step s, for each live slot with exact logits y over the output columns:
 *  - its candidates are its first K columns ordered by (y descending, column ascending) -- for K = 1 the greedy choice;
 *  - a candidate's token score is sc = (float)((double)y[c] - LSE(y)), LSE formed exactly as token_scores forms it,
 *    and its total t = fl32(cum + sc);
 *  - the sentence takes the first w candidates over its live slots, ordered by (t descending, slot ascending,
 *    candidate rank ascending).  A chosen candidate whose word (through the shortlist) is EOS becomes a finished
 *    hypothesis, EOS included; the others become the live slots 0, 1, ... in the order they were chosen, and w drops
 *    by the number of EOS choices (marian's shrinking beam).  At step max_steps - 1 every chosen candidate finishes as
 *    it stands.  A sentence is done when w reaches 0; decoding stops when every sentence is done.
 * Every sentence so ends with exactly K finished hypotheses.  Each is ranked by normalized = (double)total /
 * pow(len, length_penalty), len counting EOS; ties go to the earlier finishing step, then the earlier choice.  total
 * is the float sum of the token scores in order.  So K = 1 is greedy decoding, bit for bit (tokens, scores,
 * alignments), and slimt_b200_score of a returned hypothesis reproduces its token scores bit for bit.
 * Arithmetic: beam search always runs the bit-exact arithmetic, whatever slimt_b200_ctx_set_math says.
 * Errors, each reported before any GPU work (the model stays usable): beam_size outside 1..8, nbest outside
 * 1..beam_size, a length penalty that is negative or not finite, an n-best capacity below n_sentences * nbest *
 * max_steps of the sentence's batch.
 * Device workspace: greedy's with K rows per sentence, plus 12 * K bytes per sentence and step of step records (and
 * 4 * K * source width per sentence and step with alignments). */
typedef struct slimt_b200_beam {
  int32_t beam_size;          /* K, 1..8 */
  int32_t nbest;              /* 1..K hypotheses per sentence in the n-best outputs */
  float length_penalty;       /* alpha: finite, >= 0 */
  /* optional (NULL = not wanted): hypothesis h of sentence i is entry i * nbest + h, best first */
  uint32_t* nbest_tokens;     /* ragged by nbest_offsets, EOS included */
  float* nbest_token_scores;  /* ragged like nbest_tokens */
  size_t nbest_capacity;      /* tokens */
  uint64_t* nbest_offsets;    /* [n_sentences * nbest + 1] */
  float* nbest_totals;        /* [n_sentences * nbest] */
  double* nbest_normalized;   /* [n_sentences * nbest] */
  uint64_t steps;             /* out: decoder steps executed, summed over the batches */
} slimt_b200_beam;
/* Beam search over a request: io's out_tokens, out_scores and out_alignments receive each sentence's best hypothesis
 * (as slimt_b200_translate_multi returns the greedy one), beam's n-best outputs the first nbest hypotheses. */
int slimt_b200_translate_beam(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io,
                              slimt_b200_beam* beam);

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
