// Beam search through the C++ host layer (Options::beam_size): Blocking with beam_size 4 and 1, the cache bypass,
// and sample together with a beam refused.
// Usage: host_beam_test <model.bin> <shortlist.bin|-> <sentences.u32> <out.bin>
//   sentences.u32: u32 n, then per sentence u32 len + words.
//   out.bin: for beam_size 4 (length penalty 1), then for beam_size 1: u32 n, then per sentence u32 len, u32 source
//   len + words + len floats of scores + len * source len floats of alignments.
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

static void write(std::ofstream &out, const slimt::Sentences &sources, const slimt::WordsResponse &r) {
  uint32_t n = r.target.size();
  put(out, &n, 4);
  for (size_t i = 0; i < r.target.size(); i++) {
    uint32_t len = r.target[i].size(), src = sources[i].size();
    put(out, &len, 4);
    put(out, &src, 4);
    put(out, r.target[i].data(), 4 * len);
    put(out, r.scores[i].data(), 4 * len);
    for (const auto &row : r.alignments[i]) put(out, row.data(), 4 * row.size());
  }
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
    slimt::Options beam;
    beam.beam_size = 4, beam.length_penalty = 1.0f, beam.scores = true, beam.alignment = true;
    slimt::Options greedy;
    greedy.scores = true, greedy.alignment = true;

    // 1. Blocking with beam_size 4 and with 1: compared with the C ABI by the caller
    slimt::Config config;
    config.max_words = 96;
    config.cache_size = 1024;
    slimt::Blocking blocking(config);
    slimt::WordsResponse b4 = blocking.translate(model, sources, beam);
    expect(b4.scores.size() == b4.target.size() && b4.alignments.size() == b4.target.size(), "beam: per sentence");
    // 2. the cache: beam segments are neither answered from it nor stored
    slimt::WordsResponse again = blocking.translate(model, sources, beam);
    expect(blocking.cache_hits() == 0, "cache: a beam request was answered from the cache");
    expect(again.target == b4.target && again.scores == b4.scores, "beam: not reproducible");
    slimt::WordsResponse b1 = blocking.translate(model, sources, greedy);
    expect(blocking.cache_hits() == 0, "cache: a beam history was stored");
    std::ofstream out(argv[4], std::ios::binary);
    write(out, sources, b4);
    write(out, sources, b1);

    // 3. sample together with a beam is refused
    slimt::Options both = beam;
    both.sample = true;
    bool refused = false;
    try {
      blocking.translate(model, sources, both);
    } catch (const std::invalid_argument &) {
      refused = true;
    }
    expect(refused, "sample with beam_size > 1 was not refused");
    std::cout << "host_beam_test ok" << std::endl;
    return 0;
  } catch (const std::exception &e) {
    std::cerr << "host_beam_test: " << e.what() << std::endl;
    return 1;
  }
}
