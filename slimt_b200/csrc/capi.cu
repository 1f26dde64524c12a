// extern "C" surface declared in include/slimt_b200.h.
#include <string.h>

#include <new>
#include <string>
#include <vector>

#include "../../include/slimt_b200.h"
#include "engine.cuh"
#include "service.cuh"

struct slimt_b200_ctx {
  sb::Context c;
};
struct slimt_b200_model {
  sb::Model m;
};

extern "C" {

const char* slimt_b200_last_error(void) { return sb::last_error(); }
const char* slimt_b200_version(void) { return "slimt_b200 0.1 (sm_100a, tcgen05 kind::i8)"; }

int slimt_b200_ctx_create(int device, slimt_b200_ctx** out) {
  auto* ctx = new (std::nothrow) slimt_b200_ctx();
  if (!ctx) return 1;
  if (ctx->c.init(device)) {
    delete ctx;
    return 1;
  }
  *out = ctx;
  return 0;
}

void slimt_b200_ctx_destroy(slimt_b200_ctx* ctx) {
  if (!ctx) return;
  ctx->c.destroy();
  delete ctx;
}

int slimt_b200_ctx_synchronize(slimt_b200_ctx* ctx) {
  SB_CUDA(cudaSetDevice(ctx->c.device));
  SB_CUDA(cudaStreamSynchronize(ctx->c.stream));
  return 0;
}

int slimt_b200_ctx_set_math(slimt_b200_ctx* ctx, int fast) {
  std::lock_guard<std::recursive_mutex> g(ctx->c.mu);
  ctx->c.fast = fast != 0;
  return 0;
}
int slimt_b200_ctx_get_math(const slimt_b200_ctx* ctx) { return ctx->c.fast ? 1 : 0; }

void* slimt_b200_dev_alloc(slimt_b200_ctx* ctx, size_t bytes) {
  cudaSetDevice(ctx->c.device);
  void* p = nullptr;
  if (cudaMalloc(&p, bytes) != cudaSuccess) {
    sb::set_error("cudaMalloc failed for " + std::to_string(bytes) + " bytes");
    return nullptr;
  }
  return p;
}
void slimt_b200_dev_free(slimt_b200_ctx* ctx, void* p) {
  cudaSetDevice(ctx->c.device);
  cudaFree(p);
}
int slimt_b200_memcpy_h2d(slimt_b200_ctx* ctx, void* dst, const void* src, size_t bytes) {
  SB_CUDA(cudaSetDevice(ctx->c.device));
  SB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->c.stream));
  SB_CUDA(cudaStreamSynchronize(ctx->c.stream));
  ctx->c.h2d_bytes += bytes;
  return 0;
}
int slimt_b200_memcpy_d2h(slimt_b200_ctx* ctx, void* dst, const void* src, size_t bytes) {
  SB_CUDA(cudaSetDevice(ctx->c.device));
  SB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->c.stream));
  SB_CUDA(cudaStreamSynchronize(ctx->c.stream));
  ctx->c.d2h_bytes += bytes;
  return 0;
}
int slimt_b200_timer_start(slimt_b200_ctx* ctx) {
  SB_CUDA(cudaSetDevice(ctx->c.device));
  SB_CUDA(cudaEventRecord(ctx->c.ev0, ctx->c.stream));
  return 0;
}
int slimt_b200_timer_stop(slimt_b200_ctx* ctx, double* ms) {
  SB_CUDA(cudaSetDevice(ctx->c.device));
  SB_CUDA(cudaEventRecord(ctx->c.ev1, ctx->c.stream));
  SB_CUDA(cudaEventSynchronize(ctx->c.ev1));
  float t = 0;
  SB_CUDA(cudaEventElapsedTime(&t, ctx->c.ev0, ctx->c.ev1));
  *ms = t;
  return 0;
}
int slimt_b200_flush_l2(slimt_b200_ctx* ctx, size_t bytes) {
  sb::Context& c = ctx->c;
  SB_CUDA(cudaSetDevice(c.device));
  if (bytes > c.flush_bytes) {
    if (c.flush_buf) SB_CUDA(cudaFree(c.flush_buf));
    c.flush_buf = nullptr;
    SB_CUDA(cudaMalloc(&c.flush_buf, bytes));
    c.flush_bytes = bytes;
  }
  SB_CUDA(cudaMemsetAsync(c.flush_buf, 1, bytes, c.stream));
  return 0;
}

void slimt_b200_qmm_prepare_weight_quantized_transposed(const int8_t* input, int8_t* output, size_t rows, size_t cols) {
  // Already B^T row-major [cols][rows]: tcgen05 consumes it as a K-major operand unchanged.
  memcpy(output, input, rows * cols);
}

void slimt_b200_qmm_prepare_weight_transposed(const float* weights, int8_t* prepared, float quantization_multiplier,
                                              size_t cols, size_t rows) {
  sb::host_quantize(weights, prepared, quantization_multiplier, cols * rows);
}

int slimt_b200_qmm_affine(slimt_b200_ctx* ctx, const float* x, size_t M, size_t K, const int8_t* W, size_t N,
                          const float* bias, float a_quant, float b_quant, const uint32_t* indices, size_t n_indices,
                          float* y) {
  return sb::qmm_affine_host(ctx->c, x, M, K, W, N, bias, a_quant, b_quant, indices, n_indices, y, nullptr, nullptr);
}

int slimt_b200_qmm_affine_debug(slimt_b200_ctx* ctx, const float* x, size_t M, size_t K, const int8_t* W, size_t N,
                                const float* bias, float a_quant, float b_quant, const uint32_t* indices,
                                size_t n_indices, float* y, int8_t* qa_out, int32_t* acc_out) {
  return sb::qmm_affine_host(ctx->c, x, M, K, W, N, bias, a_quant, b_quant, indices, n_indices, y, qa_out, acc_out);
}

int slimt_b200_model_create(slimt_b200_ctx* ctx, const void* model_bin, size_t bytes,
                            const slimt_b200_model_config* config, slimt_b200_model** out) {
  if (config->feed_forward_depth != 2) {
    sb::set_error("feed_forward_depth must be 2");
    return 1;
  }
  auto* m = new (std::nothrow) slimt_b200_model();
  if (!m) return 1;
  m->m.eos_id = config->eos_id, m->m.pad_id = config->pad_id;
  if (m->m.load(&ctx->c, model_bin, bytes, config->encoder_layers, config->decoder_layers, config->num_heads)) {
    m->m.destroy();
    delete m;
    return 1;
  }
  *out = m;
  return 0;
}

void slimt_b200_model_destroy(slimt_b200_model* model) {
  if (!model) return;
  model->m.destroy();
  delete model;
}

int slimt_b200_model_dims(const slimt_b200_model* model, int32_t* emb, int32_t* ffn, int32_t* vocab) {
  *emb = model->m.E, *ffn = model->m.F, *vocab = model->m.V;
  return 0;
}

int slimt_b200_model_set_max_length(slimt_b200_model* model, int32_t n) {
  if (n < 1 || n > model->m.max_pos) {
    sb::set_error("max length " + std::to_string(n) + " is outside [1, " + std::to_string(model->m.max_pos) +
                  "] (the positional table's rows)");
    return 1;
  }
  model->m.len_bound = n;
  return 0;
}

int slimt_b200_model_max_length(const slimt_b200_model* model, int32_t* current, int32_t* supported) {
  *current = model->m.max_len(), *supported = model->m.max_pos;
  return 0;
}

int slimt_b200_model_forward(slimt_b200_model* model, slimt_b200_forward_io* io) {
  return slimt_b200_model_forward_sampled(model, io, nullptr);
}

int slimt_b200_model_forward_sampled(slimt_b200_model* model, slimt_b200_forward_io* io,
                                     const slimt_b200_sampling* sampling) {
  return slimt_b200_model_forward_topk(model, io, sampling, 0);
}

int slimt_b200_model_forward_topk(slimt_b200_model* model, slimt_b200_forward_io* io,
                                  const slimt_b200_sampling* sampling, int32_t top_k) {
  if (sb::check_sampling(sampling) || sb::check_top_k(sampling, top_k)) return 1;
  if (sampling && io->forced) {
    sb::set_error("sampling: teacher forcing (forced) and sampling exclude each other");
    return 1;
  }
  sb::ForwardArgs a;
  a.tokens = io->tokens, a.lengths = io->lengths, a.B = io->batch, a.T = io->seq;
  a.limit_factor = io->limit_factor;
  a.shortlist = io->shortlist, a.n_shortlist = io->n_shortlist;
  a.forced = io->forced, a.device_io = io->device_io != 0;
  a.step_tokens = io->step_tokens;
  a.encoder_out = io->encoder_out, a.logits = io->logits, a.alignment = io->alignment;
  a.scores = io->token_scores;
  if (sampling) a.sample = true, a.inv_t = sb::sampling_inv_t(sampling->temperature), a.seed = sampling->seed, a.keys = sampling->keys;
  a.top_k = top_k;
  int rc = sb::model_forward(model->m, a);
  io->steps = a.steps;
  io->target_tokens = a.target_tokens;
  return rc;
}

int slimt_b200_translate(slimt_b200_model* model, slimt_b200_translate_io* io) {
  sb::Model* m = &model->m;
  return sb::translate_multi(&m, 1, io, nullptr);
}

int slimt_b200_translate_multi(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io) {
  return slimt_b200_translate_sampled(replicas, n_replicas, io, nullptr);
}

int slimt_b200_translate_sampled(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io,
                                 const slimt_b200_sampling* sampling) {
  return slimt_b200_translate_topk(replicas, n_replicas, io, sampling, 0);
}

int slimt_b200_translate_topk(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io,
                              const slimt_b200_sampling* sampling, int32_t top_k) {
  if (sb::check_sampling(sampling) || sb::check_top_k(sampling, top_k)) return 1;
  std::vector<sb::Model*> ms(n_replicas);
  for (size_t i = 0; i < n_replicas; i++) ms[i] = replicas && replicas[i] ? &replicas[i]->m : nullptr;
  return sb::translate_multi(ms.data(), n_replicas, io, sampling, nullptr, top_k);
}

int slimt_b200_translate_beam(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_translate_io* io,
                              slimt_b200_beam* beam) {
  if (beam == nullptr) {
    sb::set_error("translate_beam: beam is NULL");
    return 1;
  }
  std::vector<sb::Model*> ms(n_replicas);
  for (size_t i = 0; i < n_replicas; i++) ms[i] = replicas && replicas[i] ? &replicas[i]->m : nullptr;
  return sb::translate_multi(ms.data(), n_replicas, io, nullptr, beam);
}

int slimt_b200_score(slimt_b200_model* const* replicas, size_t n_replicas, slimt_b200_score_io* io) {
  if (io == nullptr) {
    sb::set_error("score: io is NULL");
    return 1;
  }
  std::vector<sb::Model*> ms(n_replicas);
  for (size_t i = 0; i < n_replicas; i++) ms[i] = replicas && replicas[i] ? &replicas[i]->m : nullptr;
  return sb::score_multi(ms.data(), n_replicas, io);
}

uint64_t slimt_b200_kernel_launches(const slimt_b200_ctx* ctx) { return ctx->c.launches; }

int slimt_b200_shortlist_generate(const void* shortlist_bin, size_t shortlist_bytes, const uint32_t* words,
                                  size_t n_words, size_t vocab, uint32_t* out, size_t out_capacity, size_t* n_out) {
  sb::ShortlistGenerator gen;
  if (gen.load(shortlist_bin, shortlist_bytes, vocab, false)) return 1;
  std::vector<uint32_t> r;
  if (gen.generate(words, n_words, vocab, &r)) return 1;
  *n_out = r.size();
  if (r.size() > out_capacity) {
    sb::set_error("shortlist output capacity too small");
    return 1;
  }
  memcpy(out, r.data(), 4 * r.size());
  return 0;
}

int slimt_b200_shortlist_check(const void* shortlist_bin, size_t shortlist_bytes, size_t vocab) {
  sb::ShortlistGenerator gen;
  return gen.load(shortlist_bin, shortlist_bytes, vocab, true);
}

int slimt_b200_batcher_plan(const uint64_t* lengths, size_t n, size_t max_words, uint64_t* batch_ids,
                            uint64_t* batch_offsets, uint64_t* widths, size_t* n_batches) {
  sb::Batcher batcher(max_words);
  for (size_t i = 0; i < n; i++) batcher.enqueue(i, lengths[i]);
  size_t nb = 0, pos = 0;
  batch_offsets[0] = 0;
  for (;;) {
    size_t width = 0;
    std::vector<size_t> b = batcher.generate(&width);
    if (b.empty()) break;
    for (size_t id : b) batch_ids[pos++] = id;
    widths[nb] = width;
    batch_offsets[++nb] = pos;
  }
  *n_batches = nb;
  return 0;
}

int slimt_b200_profile_enable(slimt_b200_ctx* ctx, int on) {
  sb::Context& c = ctx->c;
  SB_CUDA(cudaSetDevice(c.device));
  SB_CUDA(cudaStreamSynchronize(c.stream));
  for (auto& r : c.prof) c.event_pool.push_back(r.e0), c.event_pool.push_back(r.e1);
  c.prof.clear();
  c.profiling = on != 0;
  return 0;
}

int slimt_b200_profile_read(slimt_b200_ctx* ctx, slimt_b200_kernel_stat* out, size_t capacity, size_t* n_out) {
  sb::Context& c = ctx->c;
  SB_CUDA(cudaSetDevice(c.device));
  SB_CUDA(cudaStreamSynchronize(c.stream));
  std::vector<slimt_b200_kernel_stat> agg;
  for (auto& r : c.prof) {
    float ms = 0;
    SB_CUDA(cudaEventElapsedTime(&ms, r.e0, r.e1));
    size_t i = 0;
    for (; i < agg.size(); i++)
      if (strcmp(agg[i].name, r.tag) == 0) break;
    if (i == agg.size()) {
      slimt_b200_kernel_stat st;
      memset(&st, 0, sizeof(st));
      strncpy(st.name, r.tag, sizeof(st.name) - 1);
      agg.push_back(st);
    }
    agg[i].launches += 1, agg[i].ms += ms, agg[i].ops += r.ops, agg[i].bytes += r.bytes;
    c.event_pool.push_back(r.e0), c.event_pool.push_back(r.e1);
  }
  c.prof.clear();
  *n_out = agg.size();
  for (size_t i = 0; i < agg.size() && i < capacity; i++) out[i] = agg[i];
  return 0;
}

}  // extern "C"
