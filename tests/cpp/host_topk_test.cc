// Top-k sampling through the C++ host layer (Options::top_k): Blocking and Async on word ids, Async requests pooled only
// with equal top_k, the invalid_argument cases, the pivot, and one text-level Blocking::translate.
// Usage: host_topk_test <model.bin> <shortlist.bin|-> <sentences.u32> <out.bin> [<text model.bin> <vocab.spm> <text>]
//   sentences.u32: u32 n, then per sentence u32 len + words.
//   out.bin: Blocking's top-10 targets and scores (temperature 0.8, seed 7): u32 n, then per sentence u32 len + words
//   + len floats.
#include <algorithm>
#include <cstdio>
#include <fstream>
#include <iostream>
#include <iterator>

#include "slimt_b200.hh"

static std::vector<char> slurp(const char *path) {
  std::ifstream f(path, std::ios::binary);
  return std::vector<char>((std::istreambuf_iterator<char>(f)), std::istreambuf_iterator<char>());
}
static void put(std::ofstream &o, const void *p, size_t n) { o.write(static_cast<const char *>(p), n); }
static void expect(bool ok, const char *what) {
  if (!ok) throw std::runtime_error(what);
}

int main(int argc, char **argv) {
  if (argc < 5) return 2;
  try {
    std::vector<char> raw = slurp(argv[3]);
    if (raw.size() < 4) throw std::runtime_error("cannot read the sentences file");
    const uint32_t *p = reinterpret_cast<const uint32_t *>(raw.data());
    slimt::Sentences sources(*p++);
    for (auto &s : sources) {
      uint32_t len = *p++;
      s.assign(p, p + len);
      p += len;
    }
    slimt::Package<std::string> paths{argv[1], "", std::string(argv[2]) == "-" ? "" : argv[2]};
    auto model = std::make_shared<slimt::Model>(slimt::preset::tiny(), paths);
    slimt::Options topk;
    topk.sample = true, topk.temperature = 0.8f, topk.seed = 7, topk.scores = true, topk.top_k = 10;
    slimt::Options full = topk;
    full.top_k = 0;

    // 1. Blocking: the top-k answer (compared with the C ABI by the caller); the same call again gives the same
    slimt::Config config;
    config.max_words = 96;
    config.cache_size = 0;
    slimt::Blocking blocking(config);
    slimt::WordsResponse with = blocking.translate(model, sources, topk);
    expect(with.scores.size() == with.target.size(), "Blocking: scores per sentence");
    expect(blocking.translate(model, sources, topk).target == with.target, "Blocking: not reproducible");
    std::ofstream out(argv[4], std::ios::binary);
    uint32_t n = with.target.size();
    put(out, &n, 4);
    for (size_t i = 0; i < with.target.size(); i++) {
      uint32_t len = with.target[i].size();
      put(out, &len, 4);
      put(out, with.target[i].data(), 4 * len);
      put(out, with.scores[i].data(), 4 * len);
    }

    // 2. Async over two replicas on one device: the same answer
    slimt::Config workers = config;
    workers.workers = 2;
    {
      auto two = std::make_shared<slimt::Model>(slimt::preset::tiny(), paths, std::vector<int>{0, 0});
      slimt::Async async(workers);
      slimt::WordsResponse a = async.translate(two, sources, topk).get();
      expect(a.target == with.target && a.scores == with.scores, "Async answer differs from Blocking's");
    }

    // 3. Async requests queued together are pooled only with equal top_k: each equals the same request served alone.
    // Without a shortlist (a pooled batch's candidate set is the union over the pool); a pooled batch may be wider than
    // the request's own and so decode more steps: the shorter answer must be the beginning of the longer.
    {
      auto open = std::make_shared<slimt::Model>(slimt::preset::tiny(), slimt::Package<std::string>{argv[1], "", ""});
      slimt::Options five = topk;
      five.top_k = 5;
      const slimt::Options opts[4] = {topk, full, five, topk};
      slimt::Config one = config;
      one.workers = 1;
      slimt::Async async(one);
      std::future<slimt::WordsResponse> f[4];
      for (int k = 0; k < 4; k++) f[k] = async.translate(open, sources, opts[k]);
      for (int k = 0; k < 4; k++) {
        slimt::WordsResponse pooled = f[k].get(), alone = blocking.translate(open, sources, opts[k]);
        expect(pooled.target.size() == alone.target.size(), "pooled Async: segment count");
        for (size_t i = 0; i < alone.target.size(); i++) {
          const size_t len = std::min(pooled.target[i].size(), alone.target[i].size());
          expect(std::equal(alone.target[i].begin(), alone.target[i].begin() + len, pooled.target[i].begin()) &&
                     std::equal(alone.scores[i].begin(), alone.scores[i].begin() + len, pooled.scores[i].begin()),
                 "pooled Async: an answer differs from the request served alone");
        }
      }
    }

    // 4. invalid arguments
    {
      auto refused = [&](slimt::Options o) {
        try {
          blocking.translate(model, sources, o);
        } catch (const std::invalid_argument &) {
          return true;
        }
        return false;
      };
      slimt::Options o = topk;
      o.top_k = -1;
      expect(refused(o), "top_k = -1 accepted");
      o.top_k = 257;
      expect(refused(o), "top_k = 257 accepted");
      o = topk;
      o.sample = false;
      expect(refused(o), "top_k without sample accepted");
      o = topk;
      o.beam_size = 4;
      expect(refused(o), "top_k with beam_size 4 accepted");
      expect(blocking.translate(model, sources, topk).target == with.target, "the service is unusable after a refusal");
    }

    // 5. pivot: both legs restricted with the same options
    {
      slimt::WordsResponse pivoted = blocking.pivot(model, model, sources, topk);
      slimt::WordsResponse second = blocking.translate(model, with.target, topk);
      expect(pivoted.target == second.target && pivoted.scores == second.scores, "pivot: not the top-k second leg");
    }

    // 6. text level: one top-k request
    if (argc >= 8) {
      slimt::Model::Config mc = slimt::preset::tiny();
      auto text_model = std::make_shared<slimt::Model>(mc, slimt::Package<std::string>{argv[5], argv[6], "", ""});
      slimt::Blocking service(config);
      std::vector<slimt::Response> r = service.translate(text_model, std::vector<std::string>{argv[7]}, topk);
      auto [annotated, segments] = text_model->processor().process(std::string(argv[7]), config.wrap_length);
      slimt::WordsResponse words = service.translate(text_model, segments, topk);
      expect(r.size() == 1 && r[0].scores.size() == segments.size(), "text: one score list per sentence");
      for (size_t s = 0; s < segments.size(); s++) expect(r[0].scores[s] == words.scores[s], "text: not the word-level answer");
      std::printf("text sentences %zu\n", segments.size());
    }
    std::printf("host_topk_test ok\n");
    return 0;
  } catch (const std::exception &e) {
    std::fprintf(stderr, "host_topk_test: %s\n", e.what());
    return 1;
  }
}
