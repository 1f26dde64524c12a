// Sampling through the C++ host layer (Options::sample): Blocking and Async on word ids, pooled Async requests, the
// cache bypass, the pivot, and one text-level Blocking::translate.
// Usage: host_sampling_test <model.bin> <shortlist.bin|-> <sentences.u32> <out.bin> [<text model.bin> <vocab.spm> <text>]
//   sentences.u32: u32 n, then per sentence u32 len + words.
//   out.bin: Blocking's sampled targets and scores (temperature 0.8, seed 7): u32 n, then per sentence u32 len + words
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
    slimt::Options sampled;
    sampled.sample = true, sampled.temperature = 0.8f, sampled.seed = 7, sampled.scores = true;

    // 1. Blocking: the sampled answer (compared with the C ABI by the caller); the same call again gives the same
    slimt::Config config;
    config.max_words = 96;
    config.cache_size = 0;
    slimt::Blocking blocking(config);
    slimt::WordsResponse with = blocking.translate(model, sources, sampled);
    expect(with.scores.size() == with.target.size(), "Blocking: scores per sentence");
    expect(blocking.translate(model, sources, sampled).target == with.target, "Blocking: not reproducible");
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
      slimt::WordsResponse a = async.translate(two, sources, sampled).get();
      expect(a.target == with.target && a.scores == with.scores, "Async answer differs from Blocking's");
    }

    // 3. pooled Async requests: each equals the same request served alone.  Without a shortlist (a pooled batch's
    // candidate set is the union over the pool); a pooled batch may be wider than the request's own and so decode more
    // steps: the shorter answer must be the beginning of the longer.
    {
      auto open = std::make_shared<slimt::Model>(slimt::preset::tiny(), slimt::Package<std::string>{argv[1], "", ""});
      const size_t half = sources.size() / 2;
      const slimt::Sentences parts[2] = {slimt::Sentences(sources.begin(), sources.begin() + half),
                                         slimt::Sentences(sources.rbegin(), sources.rend())};
      slimt::Async async(workers);
      std::future<slimt::WordsResponse> f[2] = {async.translate(open, parts[0], sampled), async.translate(open, parts[1], sampled)};
      for (int k = 0; k < 2; k++) {
        slimt::WordsResponse pooled = f[k].get(), alone = blocking.translate(open, parts[k], sampled);
        expect(pooled.target.size() == alone.target.size(), "pooled Async: segment count");
        for (size_t i = 0; i < alone.target.size(); i++) {
          const size_t n = std::min(pooled.target[i].size(), alone.target[i].size());
          expect(std::equal(alone.target[i].begin(), alone.target[i].begin() + n, pooled.target[i].begin()) &&
                     std::equal(alone.scores[i].begin(), alone.scores[i].begin() + n, pooled.scores[i].begin()),
                 "pooled Async: an answer differs from the request served alone");
        }
      }
    }

    // 4. the cache: sampled segments are neither answered from it nor stored; a later greedy request is greedy
    {
      slimt::Config cached = config;
      cached.cache_size = 1024;
      slimt::Blocking service(cached);
      slimt::WordsResponse s1 = service.translate(model, sources, sampled);
      slimt::WordsResponse s2 = service.translate(model, sources, sampled);
      expect(service.cache_hits() == 0, "cache: a sampled request was answered from the cache");
      expect(s1.target == with.target && s2.target == with.target, "cache: sampled answers differ");
      slimt::WordsResponse greedy = service.translate(model, sources);
      expect(service.cache_hits() == 0, "cache: a sampled history was stored");
      expect(greedy.target == blocking.translate(model, sources).target, "cache: greedy request got another answer");
    }

    // 5. pivot: both legs sampled with the same options
    {
      slimt::WordsResponse pivoted = blocking.pivot(model, model, sources, sampled);
      slimt::WordsResponse second = blocking.translate(model, with.target, sampled);
      expect(pivoted.target == second.target && pivoted.scores == second.scores, "pivot: not the sampled second leg");
    }

    // 6. text level: one sampled request
    if (argc >= 8) {
      slimt::Model::Config mc = slimt::preset::tiny();
      auto text_model = std::make_shared<slimt::Model>(mc, slimt::Package<std::string>{argv[5], argv[6], "", ""});
      slimt::Blocking service(config);
      std::vector<slimt::Response> r = service.translate(text_model, std::vector<std::string>{argv[7]}, sampled);
      auto [annotated, segments] = text_model->processor().process(std::string(argv[7]), config.wrap_length);
      slimt::WordsResponse words = service.translate(text_model, segments, sampled);
      expect(r.size() == 1 && r[0].scores.size() == segments.size(), "text: one score list per sentence");
      for (size_t s = 0; s < segments.size(); s++) expect(r[0].scores[s] == words.scores[s], "text: not the word-level answer");
      std::printf("text sentences %zu\n", segments.size());
    }
    std::printf("host_sampling_test ok\n");
    return 0;
  } catch (const std::exception &e) {
    std::fprintf(stderr, "host_sampling_test: %s\n", e.what());
    return 1;
  }
}
