// Scoring through the C++ host layer: Blocking::score on word ids, with alignments, its refusals and the cache bypass.
// Usage: host_score_test <model.bin> <shortlist.bin|-> <pairs.u32> <out.bin>
//   pairs.u32: u32 n, then per pair u32 source len + words, u32 target len + words.
//   out.bin: per pair u32 target len, then len scores, then len * source len alignment floats.
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
    if (raw.size() < 4) throw std::runtime_error("cannot read the pairs file");
    const uint32_t *p = reinterpret_cast<const uint32_t *>(raw.data());
    const uint32_t n = *p++;
    slimt::Sentences sources(n), targets(n);
    for (uint32_t i = 0; i < n; i++) {
      uint32_t len = *p++;
      sources[i].assign(p, p + len);
      p += len;
      len = *p++;
      targets[i].assign(p, p + len);
      p += len;
    }
    slimt::Package<std::string> paths{argv[1], "", std::string(argv[2]) == "-" ? "" : argv[2]};
    auto model = std::make_shared<slimt::Model>(slimt::preset::tiny(), paths);
    slimt::Config config;
    config.max_words = 96;
    slimt::Blocking blocking(config);
    slimt::Options options;
    options.alignment = true;
    slimt::WordsResponse r = blocking.score(model, sources, targets, options);
    expect(r.size() == n && r.target == targets && r.scores.size() == n && r.alignments.size() == n, "score: shape");
    for (uint32_t i = 0; i < n; i++)
      expect(r.scores[i].size() == targets[i].size() && r.alignments[i].size() == targets[i].size(), "score: ragged");
    // scoring twice gives the same answer and never consults the translation cache
    slimt::WordsResponse again = blocking.score(model, sources, targets, slimt::Options());
    expect(again.scores == r.scores && again.alignments.empty(), "score: not reproducible");
    expect(blocking.cache_hits() == 0, "score: went through the cache");
    bool refused = false;
    slimt::Options sampled;
    sampled.sample = true;
    try {
      blocking.score(model, sources, targets, sampled);
    } catch (const std::invalid_argument &) {
      refused = true;
    }
    expect(refused, "score: Options::sample accepted");
    std::ofstream out(argv[4], std::ios::binary);
    for (uint32_t i = 0; i < n; i++) {
      uint32_t len = r.scores[i].size();
      put(out, &len, 4);
      put(out, r.scores[i].data(), 4 * len);
      for (const auto &row : r.alignments[i]) put(out, row.data(), 4 * row.size());
    }
  } catch (const std::exception &e) {
    std::cerr << e.what() << "\n";
    return 1;
  }
  return 0;
}
