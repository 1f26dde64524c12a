// Per-token scores through the C++ host layer (Options::scores): Blocking and Async on word ids, the cache rule, the
// pivot, and one text-level Blocking::translate.
// Usage: host_scores_test <model.bin> <shortlist.bin|-> <sentences.u32> <out.bin> [<text model.bin> <vocab.spm> <text>]
//   sentences.u32: u32 n, then per sentence u32 len + words.
//   out.bin: Blocking's targets and scores: u32 n, then per sentence u32 len + words + len floats.
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
static void one_per_token(const slimt::WordsResponse &r, const char *what) {
  expect(r.scores.size() == r.target.size(), what);
  for (size_t i = 0; i < r.target.size(); i++) expect(r.scores[i].size() == r.target[i].size(), what);
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
    slimt::Options scored;
    scored.scores = true;

    // 1. Blocking: one score per target token; without Options::scores none
    slimt::Config config;
    config.max_words = 96;
    config.cache_size = 0;
    slimt::Blocking blocking(config);
    slimt::WordsResponse plain = blocking.translate(model, sources);
    expect(plain.scores.empty(), "scores without Options::scores");
    slimt::WordsResponse with = blocking.translate(model, sources, scored);
    expect(with.target == plain.target, "scores changed the translation");
    one_per_token(with, "Blocking: one score per target token");
    std::ofstream out(argv[4], std::ios::binary);
    uint32_t n = with.target.size();
    put(out, &n, 4);
    for (size_t i = 0; i < with.target.size(); i++) {
      uint32_t len = with.target[i].size();
      put(out, &len, 4);
      put(out, with.target[i].data(), 4 * len);
      put(out, with.scores[i].data(), 4 * len);
    }

    // 2. Async over two replicas on one device: the same scores
    {
      auto two = std::make_shared<slimt::Model>(slimt::preset::tiny(), paths, std::vector<int>{0, 0});
      slimt::Config workers = config;
      workers.workers = 2;
      slimt::Async async(workers);
      std::future<slimt::WordsResponse> f = async.translate(two, sources, scored);
      slimt::WordsResponse a = f.get();
      expect(a.target == with.target && a.scores == with.scores, "Async scores differ from Blocking's");
    }

    // 3. the cache: a history stored without scores is translated again for a request that wants them
    {
      slimt::Config cached = config;
      cached.cache_size = 1024;
      slimt::Blocking service(cached);
      service.translate(model, sources);
      expect(service.cache_hits() == 0, "cache: hit on first sight");
      slimt::WordsResponse again = service.translate(model, sources, scored);
      expect(service.cache_hits() == 0, "cache: a history without scores answered a request for them");
      expect(again.scores == with.scores, "cache: re-run scores differ");
      slimt::WordsResponse third = service.translate(model, sources, scored);
      expect(service.cache_hits() == sources.size(), "cache: stored scores not reused");
      expect(third.scores == with.scores, "cache: cached scores differ");
    }

    // 4. pivot: the second leg's scores, which score the returned target tokens
    {
      slimt::WordsResponse pivoted = blocking.pivot(model, model, sources, scored);
      slimt::WordsResponse second = blocking.translate(model, with.target, scored);
      one_per_token(pivoted, "pivot: one score per target token");
      expect(pivoted.target == second.target && pivoted.scores == second.scores, "pivot: not the second leg's scores");
    }

    // 5. text level: Response::scores[s] has one score per token of sentence s's translation
    if (argc >= 8) {
      slimt::Model::Config mc = slimt::preset::tiny();
      auto text_model = std::make_shared<slimt::Model>(mc, slimt::Package<std::string>{argv[5], argv[6], "", ""});
      slimt::Blocking service(config);
      std::vector<slimt::Response> r = service.translate(text_model, std::vector<std::string>{argv[7]}, scored);
      auto [annotated, segments] = text_model->processor().process(std::string(argv[7]), config.wrap_length);
      slimt::WordsResponse words = service.translate(text_model, segments, scored);
      expect(r.size() == 1 && r[0].scores.size() == segments.size(), "text: one score list per sentence");
      for (size_t s = 0; s < segments.size(); s++)
        expect(r[0].scores[s].size() == words.target[s].size() && r[0].scores[s] == words.scores[s],
               "text: one score per token of the sentence");
      std::printf("text sentences %zu\n", segments.size());
    }
    std::printf("host_scores_test ok\n");
    return 0;
  } catch (const std::exception &e) {
    std::fprintf(stderr, "host_scores_test: %s\n", e.what());
    return 1;
  }
}
