// The slice of slimt's service layer that sits on the hot path: batch formation
// (Batcher::generate, reference slimt/Batcher.cc:95-120), batch -> Input
// (convert(), slimt/Frontend.cc:30-40), the per-batch shortlist union
// (ShortlistGenerator::generate, slimt/Shortlist.cc:115-175) and the worker loop
// exhaust() (slimt/Frontend.cc:42-60).  Plain host C++.
#pragma once
#include <stddef.h>
#include <stdint.h>

#include <vector>

namespace sb {

struct Model;

// Binary lexical shortlist image (slimt/Shortlist.hh:78-85; Shortlist.cc:41-98).
struct ShortlistGenerator {
  uint64_t frequent = 0, best = 0;
  const uint64_t* word_to_offset = nullptr;
  uint64_t word_to_offset_size = 0;
  const uint32_t* shortlist = nullptr;
  uint64_t shortlist_size = 0;
  bool shared_vocabulary = false;  // `shared_` of the reference (Shortlist.cc:132-134): source words are candidates too
  // check = the reference loader's `check` argument (checksum + content_check, Shortlist.cc:30-37, 68-98); whatever
  // its value, generate() never reads outside the image.  Nonzero return: see last_error().
  int load(const void* data, size_t bytes, size_t vocab, bool check);
  // words: all source tokens of the batch; vocab: target vocabulary size.  Sorted ids, size % 8 == 0.
  int generate(const uint32_t* words, size_t n, size_t vocab, std::vector<uint32_t>* out) const;
};

// Length-bucketed greedy batching over one request's sentences.
struct Batcher {
  explicit Batcher(size_t max_words) : max_words_(max_words) {}
  void enqueue(size_t sentence, size_t length);
  // Next batch of sentence indices (empty when drained); max_length receives the padded width.
  std::vector<size_t> generate(size_t* max_length);

 private:
  size_t max_words_;
  std::vector<std::vector<size_t>> bucket_;  // per length: sentence ids in ascending order
  std::vector<size_t> head_;                 // per length: first unconsumed position
  size_t running_max_ = 0;
};

}  // namespace sb

struct slimt_b200_translate_io;
struct slimt_b200_score_io;
struct slimt_b200_sampling;
struct slimt_b200_beam;
namespace sb {
// exhaust() over one request with the batches dealt to the replicas' lanes (translate.cu); with beam set, each batch
// runs beam search (engine.cu: model_beam_on) and io receives every sentence's best hypothesis
// run beam search; with sampling and top_k > 0, each batch samples from the top_k columns of every step
int translate_multi(Model* const* models, size_t n_replicas, slimt_b200_translate_io* io,
                    const slimt_b200_sampling* sampling, slimt_b200_beam* beam = nullptr, int top_k = 0);
// The same batches and lanes scoring given targets with the time-parallel pass (engine.cu: model_score_on)
int score_multi(Model* const* models, size_t n_replicas, slimt_b200_score_io* io);

// Sampling arguments of the C ABI: nonzero (and the error set) for a temperature that is not finite or lies outside
// [1e-3, 1e3]; sampling = null (greedy) passes.
int check_sampling(const slimt_b200_sampling* sampling);
// Top-k arguments of the C ABI: nonzero (and the error set) for top_k outside 0 .. 256, or top_k > 0 without sampling.
int check_top_k(const slimt_b200_sampling* sampling, int top_k);
// inv_t = (float)(1.0 / (double)temperature)
inline float sampling_inv_t(float temperature) { return static_cast<float>(1.0 / static_cast<double>(temperature)); }
}  // namespace sb
