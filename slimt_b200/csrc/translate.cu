// The service half of the path: one request -> Batcher -> batches -> replicas -> ragged targets (translate_multi) or
// ragged scores of given targets (score_multi); both share the batching and the lanes (Service).
//
// Reference: exhaust() (slimt/Frontend.cc:42-60) inside Blocking::translate (:91-145), and Async's worker threads
// pulling batches from one batcher queue (Frontend.cc:207-227, Batcher.hh:203-259).  Here one host thread per *lane*
// (a stream + workspace + pinned staging block on some replica's GPU) takes the next unserved batch as soon as it is
// free, so N replicas on N GPUs are fed from ONE process by ONE Batcher; two lanes per replica let batch i + 1's
// packing, shortlist generation and H2D copy overlap batch i on the GPU.  Sentences are independent and batch
// composition is decided by the Batcher alone, so the result does not depend on which lane served which batch.
#include <math.h>
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
  std::vector<uint32_t> words;
  size_t vocab;
  std::vector<uint32_t> out;
};
int lazy_shortlist_cb(void* user, const uint32_t** words, size_t* n) {
  auto* l = static_cast<LazyShortlist*>(user);
  if (l->gen->generate(l->words.data(), l->words.size(), l->vocab, &l->out)) return 1;
  *words = l->out.data();
  *n = l->out.size();
  return 0;
}

// what one batch leaves behind: its sentences' kept tokens back to back in batch row order (record(), Model.cc:127-137)
struct Done {
  std::vector<uint32_t> kept;
  std::vector<float> align;  // per sentence [target_len][source_len], back to back (only when asked for)
  std::vector<float> scores;  // like kept (only when asked for)
};

// One batch on its lane: its ForwardArgs and the shortlist that is built from its source words during the call.
struct Batch {
  ForwardArgs a;
  LazyShortlist sl;
};

struct LaneStats {
  double device_ms = 0;
  uint64_t launches = 0, h2d = 0, d2h = 0;
  std::string error;
};

// What translate_multi and score_multi share: one request's replicas, its shortlist generator, the Batcher's batches
// over the source lengths, and the lanes that serve them.
struct Service {
  Model* const* models;
  size_t n_rep;
  const char* what;  // the entry point, for error messages
  ShortlistGenerator gen;
  bool use_sl = false;
  std::vector<Plan> plan;
  // counters of run(): device_ms is the longest lane's time
  double device_ms = 0;
  uint64_t launches = 0, h2d = 0, d2h = 0;

  int check_replicas() const {
    if (n_rep == 0 || models == nullptr || models[0] == nullptr) {
      set_error(std::string(what) + ": no model replica given");
      return 1;
    }
    const Model& m0 = *models[0];
    for (size_t r = 1; r < n_rep; r++) {
      if (models[r] == nullptr || models[r]->V != m0.V || models[r]->E != m0.E || models[r]->F != m0.F ||
          models[r]->eos_id != m0.eos_id || models[r]->pad_id != m0.pad_id) {
        set_error(std::string(what) + ": replicas must be copies of one model");
        return 1;
      }
    }
    return 0;
  }
  // The smallest length bound over the replicas: any replica may serve any batch.
  int max_len() const {
    int n = models[0]->max_len();
    for (size_t r = 1; r < n_rep; r++) n = std::min(n, models[r]->max_len());
    return n;
  }
  int load_shortlist(const void* bin, size_t bytes, int32_t check, int32_t shared) {
    use_sl = bin != nullptr && bytes > 0;
    if (!use_sl) return 0;
    if (gen.load(bin, bytes, static_cast<size_t>(models[0]->V), check != 0)) return 1;
    gen.shared_vocabulary = shared != 0;
    return 0;
  }
  // The Batcher's batches, in the order it forms them (Batcher::generate, Batcher.cc:95-120).  Nothing has touched a
  // GPU yet: a sentence no kernel can take fails the request as a whole, before any batch ran.
  int make_plan(const uint64_t* offsets, size_t n, size_t max_words) {
    Batcher batcher(max_words);
    for (size_t i = 0; i < n; i++) {
      if (offsets[i + 1] < offsets[i]) {
        set_error(std::string(what) + ": offsets must be non-decreasing");
        return 1;
      }
      if (offsets[i + 1] == offsets[i]) {
        set_error(std::string(what) +
                  ": empty sentences are not valid input (every segment ends in EOS, TextProcessor.cc:132-143)");
        return 1;
      }
      batcher.enqueue(i, offsets[i + 1] - offsets[i]);
    }
    for (;;) {
      Plan p;
      p.ids = batcher.generate(&p.width);
      if (p.ids.empty()) break;
      plan.push_back(std::move(p));
    }
    const int bound = max_len();
    for (const Plan& p : plan) {
      if (p.width > static_cast<size_t>(bound)) {
        set_error(std::string(what) + ": a sentence of " + std::to_string(p.width) +
                  " tokens exceeds the supported maximum of " + std::to_string(bound) +
                  " (wrap longer input first: TextProcessor's wrap_length)");
        return 1;
      }
    }
    return 0;
  }
  // Sets up batch p on lane c: cuts the lane's staging block into the buffers the caller listed in `staging` and the
  // padded sources, packs the sources (convert(), Frontend.cc:30-40; Input.cc:20-47) and fills the ForwardArgs fields
  // every mode shares.  Model::decode builds the candidate set before its first step (Model.cc:116-120); here the host
  // does it from the batch's words while the GPU runs the encoder (the callback fires once the encoder kernels are
  // queued).
  int stage(const Model& m, Context& c, const Plan& p, const uint32_t* src, const uint64_t* offsets, Workspace& staging,
            Batch& b) const {
    const size_t B = p.ids.size(), width = p.width;
    uint32_t *tokens = nullptr, *lengths = nullptr;
    staging.add(tokens, B * width), staging.add(lengths, B);
    if (staging.carve(c, true)) return 1;
    b.sl = LazyShortlist{&gen, {}, static_cast<size_t>(m.V), {}};
    b.sl.words.reserve(B * width);
    for (size_t r = 0; r < B; r++) {
      const size_t s = p.ids[r];
      const size_t len = offsets[s + 1] - offsets[s];
      memcpy(tokens + r * width, src + offsets[s], 4 * len);
      for (size_t t = len; t < width; t++) tokens[r * width + t] = m.pad_id;
      lengths[r] = static_cast<uint32_t>(len);
      b.sl.words.insert(b.sl.words.end(), src + offsets[s], src + offsets[s + 1]);
    }
    b.a.tokens = tokens, b.a.lengths = lengths, b.a.B = B, b.a.T = width;
    if (use_sl) b.a.shortlist_cb = lazy_shortlist_cb, b.a.shortlist_user = &b.sl;
    return 0;
  }
  // Deals the batches to the lanes: one host thread per lane takes the next unserved batch as soon as it is free.
  // serve(m, c, bi) runs batch bi on lane context c (whose lock is held) and returns nonzero with the error set.
  template <class Serve>
  int run(Serve serve) {
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

    auto lane_loop = [&](size_t li) {
      Lane& lane = lanes[li];
      Context& c = *lane.c;
      LaneStats& st = stats[li];
      std::lock_guard<std::recursive_mutex> ctx_lock(c.mu);  // the lane's staging block is ours for the whole request
      const uint64_t l0 = c.launches, h0 = c.h2d_bytes, d0 = c.d2h_bytes;
      cudaSetDevice(c.device);
      cudaEvent_t e0 = nullptr, e1 = nullptr;
      bool timed = false;
      for (;;) {
        const size_t bi = next.fetch_add(1);
        if (bi >= plan.size() || failed.load()) break;
        if (!timed) {
          cudaEventCreate(&e0), cudaEventCreate(&e1);
          cudaEventRecord(e0, c.stream);
          timed = true;
        }
        if (serve(*lane.m, c, bi)) {
          st.error = last_error();
          failed = true;
          break;
        }
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
      lane_loop(0);
    } else {
      std::vector<std::thread> threads;
      for (size_t li = 0; li < lanes.size(); li++) threads.emplace_back(lane_loop, li);
      for (std::thread& t : threads) t.join();
    }
    for (const LaneStats& st : stats) {
      if (!st.error.empty()) {
        set_error(st.error);  // the worker's message, re-raised on the calling thread
        return 1;
      }
      device_ms = std::max(device_ms, st.device_ms);
      launches += st.launches, h2d += st.h2d, d2h += st.d2h;
    }
    return 0;
  }
};

// One hypothesis of beam search, rebuilt on the host from the step records: its words and their scores, and for each
// word the slot whose row computed it (where its alignment row is).
struct Hyp {
  std::vector<uint32_t> tokens;
  std::vector<float> scores;
  std::vector<uint32_t> slots;
  float total = 0;
  double normalized = 0;
};

// Sentence r's K finished hypotheses (fin[r * K ..], in the order they finished), ranked by normalized score; ties keep
// the finishing order.  rec: [steps][B * K].
std::vector<Hyp> beam_hypotheses(const BeamRec* rec, const BeamFin* fin, size_t r, size_t B, int K, float alpha) {
  std::vector<Hyp> hs(K);
  for (int f = 0; f < K; f++) {
    const BeamFin& e = fin[r * K + f];
    const size_t len = e.step + 1;
    Hyp& h = hs[f];
    h.tokens.resize(len), h.scores.resize(len), h.slots.resize(len);
    h.tokens[e.step] = e.word, h.scores[e.step] = e.score, h.slots[e.step] = e.parent;
    uint32_t p = e.parent;
    for (size_t st = e.step; st-- > 0;) {
      const BeamRec& x = rec[st * B * K + r * K + p];
      h.tokens[st] = x.word, h.scores[st] = x.score;
      p = x.parent;
      h.slots[st] = p;
    }
    h.total = e.total;
    h.normalized = static_cast<double>(e.total) / std::pow(static_cast<double>(len), static_cast<double>(alpha));
  }
  std::stable_sort(hs.begin(), hs.end(), [](const Hyp& x, const Hyp& y) { return x.normalized > y.normalized; });
  return hs;
}

// The offsets of a ragged output whose sentence i holds n(i) values.
template <class N>
std::vector<uint64_t> ragged_offsets(size_t n_sent, N n) {
  std::vector<uint64_t> off(n_sent + 1, 0);
  for (size_t i = 0; i < n_sent; i++) off[i + 1] = off[i] + n(i);
  return off;
}

// Copies one field of each batch's Done (per-sentence results back to back in batch row order) to the sentences'
// places in the request's ragged output: sentence s's off[s + 1] - off[s] values go to out + off[s].
template <class T>
void scatter(const std::vector<Plan>& plan, const std::vector<Done>& done, std::vector<T> Done::*field,
             const std::vector<uint64_t>& off, T* out) {
  for (size_t bi = 0; bi < plan.size(); bi++) {
    const T* src = (done[bi].*field).data();
    for (size_t s : plan[bi].ids) {
      memcpy(out + off[s], src, sizeof(T) * (off[s + 1] - off[s]));
      src += off[s + 1] - off[s];
    }
  }
}

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

int check_sampling(const slimt_b200_sampling* sampling) {
  if (sampling == nullptr) return 0;
  const float t = sampling->temperature;
  if (!(t >= 1e-3f && t <= 1e3f)) {  // also NaN
    set_error("sampling: temperature must be finite and in [1e-3, 1e3], got " + std::to_string(t));
    return 1;
  }
  return 0;
}

int check_top_k(const slimt_b200_sampling* sampling, int top_k) {
  if (top_k < 0 || top_k > kMaxTopK) {
    set_error("top-k sampling: top_k must be in 0 .. " + std::to_string(kMaxTopK) + ", got " + std::to_string(top_k));
    return 1;
  }
  if (top_k > 0 && sampling == nullptr) {
    set_error("top-k sampling: top_k > 0 needs sampling parameters (temperature, seed, keys)");
    return 1;
  }
  return 0;
}

int check_beam(const slimt_b200_beam* beam) {
  if (beam == nullptr) return 0;
  if (beam->beam_size < 1 || beam->beam_size > kMaxBeam) {
    set_error("beam: beam_size must be in 1 .. " + std::to_string(kMaxBeam) + ", got " + std::to_string(beam->beam_size));
    return 1;
  }
  if (beam->nbest < 1 || beam->nbest > beam->beam_size) {
    set_error("beam: nbest must be in 1 .. beam_size, got " + std::to_string(beam->nbest));
    return 1;
  }
  if (!(beam->length_penalty >= 0.0f && beam->length_penalty <= 3.402823466e38f)) {  // also NaN
    set_error("beam: length_penalty must be finite and >= 0, got " + std::to_string(beam->length_penalty));
    return 1;
  }
  return 0;
}

int translate_multi(Model* const* models, size_t n_rep, slimt_b200_translate_io* io, const slimt_b200_sampling* sampling,
                    slimt_b200_beam* beam, int top_k) {
  if (check_beam(beam)) return 1;
  Service sv{models, n_rep, beam ? "translate_beam" : "translate"};
  if (sv.check_replicas()) return 1;
  io->target_tokens = 0, io->batches = 0, io->device_ms = 0;
  io->kernel_launches = 0, io->h2d_bytes = 0, io->d2h_bytes = 0;
  const size_t n_sent = io->n_sentences;
  const bool want_align = io->out_alignments != nullptr;
  const bool want_scores = io->out_scores != nullptr;
  if (sv.load_shortlist(io->shortlist_bin, io->shortlist_bytes, io->shortlist_check, io->shortlist_shared)) return 1;
  if (sv.make_plan(io->offsets, n_sent, io->max_words)) return 1;
  const std::vector<Plan>& plan = sv.plan;
  const int K = beam ? beam->beam_size : 0;
  const bool want_nbest = beam && (beam->nbest_tokens || beam->nbest_token_scores);
  if (want_nbest) {  // every hypothesis has at most its batch's max_steps tokens
    uint64_t bound = 0;
    for (const Plan& p : plan)
      bound += static_cast<uint64_t>(p.ids.size()) * beam->nbest * forward_max_steps(io->limit_factor, p.width);
    if (beam->nbest_capacity < bound) {
      set_error("translate_beam: nbest_capacity of " + std::to_string(beam->nbest_capacity) + " tokens is below the " +
                std::to_string(bound) + " that nbest hypotheses of max_steps tokens per sentence can take");
      return 1;
    }
  }

  std::vector<Done> done(plan.size());
  std::vector<uint32_t> out_len(n_sent, 0);
  std::vector<std::vector<Hyp>> nbest(beam ? n_sent : 0);  // each sentence's first nbest hypotheses
  std::atomic<uint64_t> beam_steps{0};
  auto serve_beam = [&](Model& m, Context& c, size_t bi) -> int {
    const Plan& p = plan[bi];
    const size_t B = p.ids.size(), width = p.width, M = B * K;
    const size_t stride = static_cast<size_t>(forward_max_steps(io->limit_factor, width));
    // staging: step records, finished hypotheses, alignment rows
    Workspace staging;
    BeamRec* rec = nullptr;
    BeamFin* fin = nullptr;
    float* align = nullptr;
    staging.add(rec, stride * M), staging.add(fin, M);
    if (want_align) staging.add(align, stride * M * width);
    Batch b;
    if (sv.stage(m, c, p, io->tokens, io->offsets, staging, b)) return 1;
    ForwardArgs& a = b.a;
    a.limit_factor = io->limit_factor;
    a.beam = K, a.beam_steps = rec, a.beam_finished = fin, a.alignment = align;
    if (model_beam_on(m, c, a)) return 1;
    beam_steps += a.steps;
    Done& d = done[bi];
    for (size_t r = 0; r < B; r++) {
      std::vector<Hyp> hs = beam_hypotheses(rec, fin, r, B, K, beam->length_penalty);
      const Hyp& h = hs[0];
      out_len[p.ids[r]] = static_cast<uint32_t>(h.tokens.size());
      d.kept.insert(d.kept.end(), h.tokens.begin(), h.tokens.end());
      if (want_scores) d.scores.insert(d.scores.end(), h.scores.begin(), h.scores.end());
      if (want_align)  // the row that computed word s: slot h.slots[s] of step s
        for (size_t st = 0; st < h.tokens.size(); st++) {
          const float* row = align + (st * M + r * K + h.slots[st]) * width;
          d.align.insert(d.align.end(), row, row + a.lengths[r]);
        }
      hs.resize(beam->nbest);
      nbest[p.ids[r]] = std::move(hs);
    }
    return 0;
  };
  auto serve = [&](Model& m, Context& c, size_t bi) -> int {
    if (beam) return serve_beam(m, c, bi);
    const Plan& p = plan[bi];
    const size_t B = p.ids.size(), width = p.width;
    const size_t stride = static_cast<size_t>(forward_max_steps(io->limit_factor, width));
    // staging: sentence-major step tokens, recorded lengths, alignment rows, step-major scores, sampling keys
    Workspace staging;
    uint32_t *rows = nullptr, *lens = nullptr;
    float *align = nullptr, *scores = nullptr;
    uint64_t* keys = nullptr;
    staging.add(rows, stride * B), staging.add(lens, B);
    if (want_align) staging.add(align, stride * B * width);
    if (want_scores) staging.add(scores, stride * B);
    if (sampling) staging.add(keys, B);
    Batch b;
    if (sv.stage(m, c, p, io->tokens, io->offsets, staging, b)) return 1;
    ForwardArgs& a = b.a;
    a.limit_factor = io->limit_factor;
    a.sentence_tokens = rows, a.row_stride = stride, a.target_lengths = lens;
    a.alignment = align;
    a.scores = scores;
    if (sampling) {
      // each sentence's own key (default: its index in the request), wherever the Batcher put it
      for (size_t r = 0; r < B; r++) keys[r] = sampling->keys ? sampling->keys[p.ids[r]] : static_cast<uint64_t>(p.ids[r]);
      a.sample = true, a.inv_t = sampling_inv_t(sampling->temperature), a.seed = sampling->seed, a.keys = keys;
      a.top_k = top_k;
    }
    if (model_forward_on(m, c, a)) return 1;
    Done& d = done[bi];
    size_t kept_total = 0, align_total = 0;
    for (size_t r = 0; r < B; r++) {
      out_len[p.ids[r]] = lens[r];
      kept_total += lens[r];
      align_total += static_cast<size_t>(lens[r]) * a.lengths[r];
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
          memcpy(d.align.data() + ap, align + (s * B + r) * width, 4ul * a.lengths[r]);
          ap += a.lengths[r];
        }
    }
    if (want_scores) {  // the scores of the recorded steps, sentence by sentence in batch row order like kept
      d.scores.resize(kept_total);
      size_t sp = 0;
      for (size_t r = 0; r < B; r++)
        for (size_t s = 0; s < lens[r]; s++) d.scores[sp++] = scores[s * B + r];
    }
    return 0;
  };
  if (sv.run(serve)) return 1;
  io->device_ms = sv.device_ms;
  io->kernel_launches = sv.launches, io->h2d_bytes = sv.h2d, io->d2h_bytes = sv.d2h;
  io->batches = plan.size();

  // ---- ragged outputs
  const std::vector<uint64_t> out_off = ragged_offsets(n_sent, [&](size_t i) { return out_len[i]; });
  io->target_tokens = out_off[n_sent];
  if ((io->out_tokens || want_scores) && out_off[n_sent] > io->out_capacity) {
    set_error(io->out_tokens ? "out_tokens capacity too small" : "out_scores capacity too small");
    return 1;
  }
  if (io->out_offsets) memcpy(io->out_offsets, out_off.data(), 8 * (n_sent + 1));
  if (io->out_tokens) scatter(plan, done, &Done::kept, out_off, io->out_tokens);
  if (want_scores) scatter(plan, done, &Done::scores, out_off, io->out_scores);
  if (want_align) {
    const std::vector<uint64_t> al_off = ragged_offsets(
        n_sent, [&](size_t i) { return static_cast<uint64_t>(out_len[i]) * (io->offsets[i + 1] - io->offsets[i]); });
    if (al_off[n_sent] > io->align_capacity) {
      set_error("out_alignments capacity too small");
      return 1;
    }
    if (io->out_align_offsets) memcpy(io->out_align_offsets, al_off.data(), 8 * (n_sent + 1));
    scatter(plan, done, &Done::align, al_off, io->out_alignments);
  }
  if (beam) {
    beam->steps = beam_steps.load();
    const size_t nb = static_cast<size_t>(beam->nbest);
    uint64_t pos = 0;
    for (size_t i = 0; i < n_sent; i++)
      for (size_t h = 0; h < nb; h++) {
        const Hyp& x = nbest[i][h];
        const size_t e = i * nb + h;
        if (beam->nbest_offsets) beam->nbest_offsets[e] = pos;
        if (beam->nbest_tokens) memcpy(beam->nbest_tokens + pos, x.tokens.data(), 4 * x.tokens.size());
        if (beam->nbest_token_scores) memcpy(beam->nbest_token_scores + pos, x.scores.data(), 4 * x.scores.size());
        if (beam->nbest_totals) beam->nbest_totals[e] = x.total;
        if (beam->nbest_normalized) beam->nbest_normalized[e] = x.normalized;
        pos += x.tokens.size();
      }
    if (beam->nbest_offsets) beam->nbest_offsets[n_sent * nb] = pos;
  }
  return 0;
}

int score_multi(Model* const* models, size_t n_rep, slimt_b200_score_io* io) {
  io->batches = 0, io->device_ms = 0, io->kernel_launches = 0, io->h2d_bytes = 0, io->d2h_bytes = 0;
  const size_t n_sent = io->n_sentences;
  const uint64_t* so = io->offsets;
  const uint64_t* to = io->target_offsets;
  const bool want_align = io->out_alignments != nullptr;
  // the request's shape, checked before anything else (no model is needed for it)
  if (n_sent > 0 && (so == nullptr || to == nullptr || io->tokens == nullptr)) {
    set_error("score: tokens, offsets and target_offsets are required");
    return 1;
  }
  for (size_t i = 0; i < n_sent; i++) {
    if (so[i + 1] < so[i] || to[i + 1] < to[i]) {
      set_error("score: offsets must be non-decreasing");
      return 1;
    }
  }
  const uint64_t n_tgt = n_sent ? to[n_sent] - to[0] : 0;
  if (n_tgt > 0 && (io->targets == nullptr || io->out_scores == nullptr)) {
    set_error("score: targets and out_scores are required");
    return 1;
  }
  if (n_tgt > io->out_capacity) {
    set_error("score: out_scores capacity too small (" + std::to_string(n_tgt) + " target tokens)");
    return 1;
  }
  const std::vector<uint64_t> al_off =
      ragged_offsets(n_sent, [&](size_t i) { return (to[i + 1] - to[i]) * (so[i + 1] - so[i]); });
  if (want_align && al_off[n_sent] > io->align_capacity) {
    set_error("score: out_alignments capacity too small");
    return 1;
  }
  Service sv{models, n_rep, "score"};
  if (sv.check_replicas()) return 1;
  const int bound = sv.max_len();
  const uint32_t V = static_cast<uint32_t>(models[0]->V);
  for (size_t i = 0; i < n_sent; i++) {
    if (to[i + 1] - to[i] > static_cast<uint64_t>(bound)) {
      set_error("score: target " + std::to_string(i) + " of " + std::to_string(to[i + 1] - to[i]) +
                " tokens exceeds the supported maximum of " + std::to_string(bound));
      return 1;
    }
    for (uint64_t k = to[i]; k < to[i + 1]; k++)
      if (io->targets[k] >= V) {
        set_error("score: target word " + std::to_string(io->targets[k]) + " is outside the vocabulary of " +
                  std::to_string(V));
        return 1;
      }
  }
  if (sv.load_shortlist(io->shortlist_bin, io->shortlist_bytes, io->shortlist_check, io->shortlist_shared)) return 1;
  if (sv.make_plan(so, n_sent, io->max_words)) return 1;
  const std::vector<Plan>& plan = sv.plan;

  std::vector<Done> done(plan.size());
  auto serve = [&](Model& m, Context& c, size_t bi) -> int {
    const Plan& p = plan[bi];
    const size_t B = p.ids.size(), width = p.width;
    size_t Tt = 0, n_scores = 0, n_align = 0;
    for (size_t s : p.ids) {
      const size_t tl = to[s + 1] - to[s];
      Tt = std::max(Tt, tl), n_scores += tl, n_align += tl * (so[s + 1] - so[s]);
    }
    if (Tt == 0) return 0;  // every target of the batch is empty: nothing to score
    // staging: padded targets, scores, alignments
    Workspace staging;
    uint32_t* targets = nullptr;
    float *sc = nullptr, *al = nullptr;
    staging.add(targets, B * Tt), staging.add(sc, B * Tt);
    if (want_align) staging.add(al, B * Tt * width);
    Batch b;
    if (sv.stage(m, c, p, io->tokens, so, staging, b)) return 1;
    for (size_t r = 0; r < B; r++) {
      const size_t s = p.ids[r], tl = to[s + 1] - to[s];
      memcpy(targets + r * Tt, io->targets + to[s], 4 * tl);
      for (size_t j = tl; j < Tt; j++) targets[r * Tt + j] = m.pad_id;  // computed and discarded
    }
    ForwardArgs& a = b.a;
    a.targets = targets, a.target_T = Tt, a.scores = sc, a.alignment = al;
    if (model_score_on(m, c, a)) return 1;
    // each sentence's valid positions, back to back in batch row order
    Done& d = done[bi];
    d.scores.resize(n_scores);
    size_t sp = 0;
    for (size_t r = 0; r < B; r++) {
      const size_t tl = to[p.ids[r] + 1] - to[p.ids[r]];
      memcpy(d.scores.data() + sp, sc + r * Tt, 4 * tl);
      sp += tl;
    }
    if (want_align) {
      d.align.resize(n_align);
      size_t ap = 0;
      for (size_t r = 0; r < B; r++) {
        const size_t tl = to[p.ids[r] + 1] - to[p.ids[r]];
        for (size_t j = 0; j < tl; j++) {
          memcpy(d.align.data() + ap, al + (r * Tt + j) * width, 4ul * a.lengths[r]);
          ap += a.lengths[r];
        }
      }
    }
    return 0;
  };
  if (sv.run(serve)) return 1;
  io->device_ms = sv.device_ms;
  io->kernel_launches = sv.launches, io->h2d_bytes = sv.h2d, io->d2h_bytes = sv.d2h;
  io->batches = plan.size();

  const std::vector<uint64_t> out_off = ragged_offsets(n_sent, [&](size_t i) { return to[i + 1] - to[i]; });
  if (n_tgt > 0) scatter(plan, done, &Done::scores, out_off, io->out_scores);
  if (want_align) {
    if (io->out_align_offsets) memcpy(io->out_align_offsets, al_off.data(), 8 * (n_sent + 1));
    scatter(plan, done, &Done::align, al_off, io->out_alignments);
  }
  return 0;
}

}  // namespace sb
