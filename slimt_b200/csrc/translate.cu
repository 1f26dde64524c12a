// The service half of the path: one request -> Batcher -> batches -> replicas -> ragged targets.
//
// Reference: exhaust() (slimt/Frontend.cc:42-60) inside Blocking::translate (:91-145), and Async's worker threads
// pulling batches from one batcher queue (Frontend.cc:207-227, Batcher.hh:203-259).  Here one host thread per *lane*
// (a stream + workspace + pinned staging block on some replica's GPU) takes the next unserved batch as soon as it is
// free, so N replicas on N GPUs are fed from ONE process by ONE Batcher; two lanes per replica let batch i + 1's
// packing, shortlist generation and H2D copy overlap batch i on the GPU.  Sentences are independent and batch
// composition is decided by the Batcher alone, so the result does not depend on which lane served which batch.
#include <string.h>

#include <algorithm>
#include <atomic>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/slimt_b200.h"
#include "engine.cuh"
#include "service.cuh"

namespace sb {

namespace {

struct Plan {
  std::vector<size_t> ids;
  size_t width = 0;
};

struct LazyShortlist {
  const ShortlistGenerator* gen;
  const std::vector<uint32_t>* words;
  size_t vocab;
  std::vector<uint32_t> out;
};
int lazy_shortlist_cb(void* user, const uint32_t** words, size_t* n) {
  auto* l = static_cast<LazyShortlist*>(user);
  if (l->gen->generate(l->words->data(), l->words->size(), l->vocab, &l->out)) return 1;
  *words = l->out.data();
  *n = l->out.size();
  return 0;
}

// what one batch leaves behind: its sentences' kept tokens back to back in batch row order (record(), Model.cc:127-137)
struct Done {
  std::vector<uint32_t> kept;
  std::vector<float> align;  // per sentence [target_len][source_len], back to back (only when asked for)
};

struct LaneStats {
  double device_ms = 0;
  uint64_t launches = 0, h2d = 0, d2h = 0, target_tokens = 0;
  std::string error;
};

}  // namespace

// Extra lanes of a model's device: created on first use, owned by the model.
Context* Model::lane(size_t i) {
  if (i == 0) return ctx;
  std::lock_guard<std::mutex> g(lanes_mu);
  while (lanes.size() < i) {
    std::unique_ptr<Context> c(new Context());
    if (c->init(ctx->device)) return nullptr;
    lanes.push_back(std::move(c));
  }
  lanes[i - 1]->fast = ctx->fast;  // lanes compute in the arithmetic mode of the model's own context
  return lanes[i - 1].get();
}

int translate_multi(Model* const* models, size_t n_rep, slimt_b200_translate_io* io) {
  if (n_rep == 0 || models == nullptr || models[0] == nullptr) {
    set_error("translate: no model replica given");
    return 1;
  }
  Model& m0 = *models[0];
  for (size_t r = 1; r < n_rep; r++) {
    if (models[r] == nullptr || models[r]->V != m0.V || models[r]->E != m0.E || models[r]->F != m0.F ||
        models[r]->eos_id != m0.eos_id || models[r]->pad_id != m0.pad_id) {
      set_error("translate: replicas must be copies of one model");
      return 1;
    }
  }
  io->target_tokens = 0, io->batches = 0, io->device_ms = 0;
  io->kernel_launches = 0, io->h2d_bytes = 0, io->d2h_bytes = 0;
  const size_t n_sent = io->n_sentences;
  const bool want_align = io->out_alignments != nullptr;

  ShortlistGenerator gen;
  const bool use_sl = io->shortlist_bin != nullptr && io->shortlist_bytes > 0;
  if (use_sl) {
    if (gen.load(io->shortlist_bin, io->shortlist_bytes, static_cast<size_t>(m0.V), io->shortlist_check != 0)) return 1;
    gen.shared_vocabulary = io->shortlist_shared != 0;
  }

  // ---- the Batcher's batches, in the order it forms them (Batcher::generate, Batcher.cc:95-120)
  std::vector<Plan> plan;
  {
    Batcher batcher(io->max_words);
    for (size_t i = 0; i < n_sent; i++) {
      if (io->offsets[i + 1] < io->offsets[i]) {
        set_error("translate: offsets must be non-decreasing");
        return 1;
      }
      if (io->offsets[i + 1] == io->offsets[i]) {
        set_error("translate: empty sentences are not valid input (every segment ends in EOS, TextProcessor.cc:132-143)");
        return 1;
      }
      batcher.enqueue(i, io->offsets[i + 1] - io->offsets[i]);
    }
    for (;;) {
      Plan p;
      p.ids = batcher.generate(&p.width);
      if (p.ids.empty()) break;
      plan.push_back(std::move(p));
    }
  }
  // nothing has touched a GPU yet: a sentence no kernel can take fails the request as a whole, before any batch ran.
  // Any replica may serve any batch, so the smallest bound of them all applies.
  int max_len = m0.max_len();
  for (size_t r = 1; r < n_rep; r++) max_len = std::min(max_len, models[r]->max_len());
  for (const Plan& p : plan) {
    if (p.width > static_cast<size_t>(max_len)) {
      set_error("translate: a sentence of " + std::to_string(p.width) + " tokens exceeds the supported maximum of " +
                std::to_string(max_len) + " (wrap longer input first: TextProcessor's wrap_length)");
      return 1;
    }
  }

  std::vector<Done> done(plan.size());
  std::vector<uint32_t> out_len(n_sent, 0);

  // ---- lanes
  size_t lanes_per = 1;
  if (const char* e = getenv("SLIMT_B200_LANES")) lanes_per = std::max(1, atoi(e));
  else if (plan.size() >= 2 * n_rep) lanes_per = 2;
  struct Lane {
    Model* m;
    Context* c;
  };
  std::vector<Lane> lanes;
  for (size_t l = 0; l < lanes_per; l++)
    for (size_t r = 0; r < n_rep; r++) {
      Context* c = models[r]->lane(l);
      if (!c) return 1;
      lanes.push_back(Lane{models[r], c});
    }
  if (lanes.size() > plan.size()) lanes.resize(std::max<size_t>(1, plan.size()));
  std::vector<LaneStats> stats(lanes.size());
  std::atomic<size_t> next{0};
  std::atomic<bool> failed{false};

  auto serve = [&](size_t li) {
    Lane& lane = lanes[li];
    Context& c = *lane.c;
    Model& m = *lane.m;
    LaneStats& st = stats[li];
    std::lock_guard<std::recursive_mutex> ctx_lock(c.mu);  // the lane's staging block is ours for the whole request
    const uint64_t l0 = c.launches, h0 = c.h2d_bytes, d0 = c.d2h_bytes;
    cudaSetDevice(c.device);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    bool timed = false;
    std::vector<uint32_t> words;
    for (;;) {
      const size_t bi = next.fetch_add(1);
      if (bi >= plan.size() || failed.load()) break;
      const Plan& p = plan[bi];
      const size_t B = p.ids.size(), width = p.width;
      const size_t stride = static_cast<size_t>(forward_max_steps(io->limit_factor, width));
      // staging: [padded tokens][lengths] | [sentence-major step tokens][recorded lengths] | [alignment rows]
      const size_t in_bytes = (4 * (B * width + B) + 255) & ~size_t(255);
      const size_t tok_bytes = (4 * (stride + 1) * B + 255) & ~size_t(255);
      const size_t al_bytes = want_align ? 4 * stride * B * width : 0;
      char* stage = c.staging_reserve(in_bytes + tok_bytes + al_bytes + 256);
      if (!stage) {
        st.error = last_error();
        failed = true;
        break;
      }
      // convert(): Batch -> padded Input (Frontend.cc:30-40; Input.cc:20-47)
      uint32_t* tokens = reinterpret_cast<uint32_t*>(stage);
      uint32_t* lengths = tokens + B * width;
      words.clear();
      words.reserve(B * width);
      for (size_t r = 0; r < B; r++) {
        const size_t s = p.ids[r];
        const size_t len = io->offsets[s + 1] - io->offsets[s];
        memcpy(tokens + r * width, io->tokens + io->offsets[s], 4 * len);
        for (size_t t = len; t < width; t++) tokens[r * width + t] = m.pad_id;
        lengths[r] = static_cast<uint32_t>(len);
        words.insert(words.end(), io->tokens + io->offsets[s], io->tokens + io->offsets[s + 1]);
      }
      // Model::decode builds the candidate set before its first step (Model.cc:116-120); here the host does it
      // while the GPU runs the encoder (the callback fires once the encoder kernels are queued)
      LazyShortlist lazy{&gen, &words, static_cast<size_t>(m.V), {}};
      uint32_t* rows = reinterpret_cast<uint32_t*>(stage + in_bytes);
      uint32_t* lens = rows + stride * B;
      float* align = want_align ? reinterpret_cast<float*>(stage + in_bytes + tok_bytes) : nullptr;
      ForwardArgs a;
      a.tokens = tokens, a.lengths = lengths, a.B = B, a.T = width;
      a.limit_factor = io->limit_factor;
      if (use_sl) a.shortlist_cb = lazy_shortlist_cb, a.shortlist_user = &lazy;
      a.sentence_tokens = rows, a.row_stride = stride, a.target_lengths = lens;
      a.alignment = align;
      if (!timed) {
        cudaEventCreate(&e0), cudaEventCreate(&e1);
        cudaEventRecord(e0, c.stream);
        timed = true;
      }
      if (model_forward_on(m, c, a)) {
        st.error = last_error();
        failed = true;
        break;
      }
      Done& d = done[bi];
      size_t kept_total = 0, align_total = 0;
      for (size_t r = 0; r < B; r++) {
        out_len[p.ids[r]] = lens[r];
        kept_total += lens[r];
        align_total += static_cast<size_t>(lens[r]) * lengths[r];
      }
      d.kept.resize(kept_total);
      size_t pos = 0;
      for (size_t r = 0; r < B; r++) {
        memcpy(d.kept.data() + pos, rows + r * stride, 4ul * lens[r]);
        pos += lens[r];
      }
      if (want_align) {  // update_alignment (Model.cc:84-108): one distribution over the sentence's own source tokens per target token
        d.align.resize(align_total);
        size_t ap = 0;
        for (size_t r = 0; r < B; r++)
          for (size_t s = 0; s < lens[r]; s++) {
            memcpy(d.align.data() + ap, align + (s * B + r) * width, 4ul * lengths[r]);
            ap += lengths[r];
          }
      }
      st.target_tokens += a.target_tokens;
    }
    if (timed) {
      cudaEventRecord(e1, c.stream);
      cudaEventSynchronize(e1);
      float ms = 0;
      cudaEventElapsedTime(&ms, e0, e1);
      st.device_ms = ms;
      cudaEventDestroy(e0), cudaEventDestroy(e1);
    }
    st.launches = c.launches - l0, st.h2d = c.h2d_bytes - h0, st.d2h = c.d2h_bytes - d0;
  };

  if (lanes.size() == 1) {
    serve(0);
  } else {
    std::vector<std::thread> threads;
    for (size_t li = 0; li < lanes.size(); li++) threads.emplace_back(serve, li);
    for (std::thread& t : threads) t.join();
  }
  for (const LaneStats& st : stats) {
    if (!st.error.empty()) {
      set_error(st.error);  // the worker's message, re-raised on the calling thread
      return 1;
    }
    io->device_ms = std::max(io->device_ms, st.device_ms);
    io->kernel_launches += st.launches, io->h2d_bytes += st.h2d, io->d2h_bytes += st.d2h;
    io->target_tokens += st.target_tokens;
  }
  io->batches = plan.size();

  // ---- ragged outputs
  std::vector<uint64_t> out_off(n_sent + 1, 0);
  for (size_t i = 0; i < n_sent; i++) out_off[i + 1] = out_off[i] + out_len[i];
  if (io->out_tokens && out_off[n_sent] > io->out_capacity) {
    set_error("out_tokens capacity too small");
    return 1;
  }
  if (io->out_offsets) memcpy(io->out_offsets, out_off.data(), 8 * (n_sent + 1));
  if (io->out_tokens) {
    for (size_t bi = 0; bi < plan.size(); bi++) {
      size_t pos = 0;
      for (size_t s : plan[bi].ids) {
        memcpy(io->out_tokens + out_off[s], done[bi].kept.data() + pos, 4ul * out_len[s]);
        pos += out_len[s];
      }
    }
  }
  if (want_align) {
    std::vector<uint64_t> al_off(n_sent + 1, 0);
    for (size_t i = 0; i < n_sent; i++) al_off[i + 1] = al_off[i] + static_cast<uint64_t>(out_len[i]) * (io->offsets[i + 1] - io->offsets[i]);
    if (al_off[n_sent] > io->align_capacity) {
      set_error("out_alignments capacity too small");
      return 1;
    }
    if (io->out_align_offsets) memcpy(io->out_align_offsets, al_off.data(), 8 * (n_sent + 1));
    for (size_t bi = 0; bi < plan.size(); bi++) {
      size_t pos = 0;
      for (size_t s : plan[bi].ids) {
        const size_t n = static_cast<size_t>(al_off[s + 1] - al_off[s]);
        memcpy(io->out_alignments + al_off[s], done[bi].align.data() + pos, 4ul * n);
        pos += n;
      }
    }
  }
  return 0;
}

}  // namespace sb
