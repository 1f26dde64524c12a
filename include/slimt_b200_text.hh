// slimt_b200_text.hh -- the text front half of slimt's services (SURVEY.md section 8 f4): what sits between a blob
// of text and the word ids Model::forward takes, and between the decoder's word ids and the translated text.
// Host-only C++17, header only, no CUDA and no dependency on libslimt_b200 (link with -ldl for the sentence
// splitter's PCRE2).  slimt_b200.hh includes this file and builds the text-level Blocking / Async services on it.
//
//   slimt::Range, Encoding, Views, Segment(s)        slimt/Types.hh:14-74
//   slimt::Annotation / AnnotatedText                slimt/Annotation.hh:15-284, Annotation.cc:14-217
//   slimt::Vocabulary                                slimt/Vocabulary.hh:13-29, Vocabulary.cc:24-104
//   slimt::spm::Processor                            the part of sentencepiece 0.2.00 (3rd-party/sentencepiece, an
//                                                    un-modified vendored dependency of the reference) that Vocabulary
//                                                    calls: model load, Normalize, unigram Encode, Decode -- restated
//                                                    from the library's published algorithm (see the class comment)
//   slimt::Regex / Match                             slimt/Regex.hh:15-62 (PCRE2, bound at run time with dlopen)
//   slimt::Splitter / SentenceStream                 slimt/Splitter.hh:14-73, Splitter.cc:21-375
//   slimt::TextProcessor                             slimt/TextProcessor.hh:17-58, TextProcessor.cc:65-199
//   slimt::Response (text level), Options            slimt/Response.hh:20-48
//   slimt::remap_alignments / combine                slimt/Response.cc:16-175
//
// Not carried: HTML (HTML.cc, XHScanner.cc: markup handling above the services, SURVEY.md section 8 marks it out of
// scope; Options::html is accepted and must be false), BPE / word / char sentencepiece models (the browsermt
// vocabularies slimt loads are unigram; another model type fails at load with a message).
//
// Error convention: loaders throw std::runtime_error (the reference's MmapFile does; sentencepiece reports a Status
// that slimt ignores, which then fails later -- failing at load is the deliberate difference).
#pragma once
#include <algorithm>
#include <array>
#include <cassert>
#include <cfloat>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <map>
#include <memory>
#include <set>
#include <sstream>
#include <stdexcept>
#include <string>
#include <string_view>
#include <tuple>
#include <unordered_map>
#include <utility>
#include <vector>

#include <dlfcn.h>

namespace slimt {

// ---------------------------------------------------------------- Types.hh
using Word = uint32_t;
using Words = std::vector<Word>;
using Segment = Words;
using Segments = std::vector<Segment>;
using Sentences = std::vector<Words>;
using Views = std::vector<std::string_view>;
template <class T>
using Ptr = std::shared_ptr<T>;
using Distribution = std::vector<float>;
using Alignment = std::vector<Distribution>;
using Alignments = std::vector<Alignment>;
struct View {
  void *data = nullptr;
  size_t size = 0;
};
struct Hypothesis {
  Words target;
  Alignment alignment;
  std::vector<float> scores;  // log-probability of each target token (Options::scores), empty otherwise
};
using History = Ptr<Hypothesis>;
using Histories = std::vector<History>;

// half-open interval [begin, end) of a string: a sentence, a word (Types.hh:14-20)
struct Range {
  size_t begin = 0;
  size_t end = 0;
  size_t size() const { return end - begin; }
};
inline bool operator==(const Range &a, const Range &b) { return a.begin == b.begin && a.end == b.end; }
enum class Encoding { Byte, UTF8 };

// ---------------------------------------------------------------- sentencepiece (unigram) as Vocabulary uses it
namespace spm {

// UTF-8 helpers with sentencepiece's semantics (src/util.h:151-176, util.cc:48-81): a lead byte decides the length,
// a malformed sequence is ONE byte, U+FFFD itself (three bytes) is valid.
inline size_t one_char_len(const char *s) { return "\1\1\1\1\1\1\1\1\1\1\1\1\2\2\3\4"[(static_cast<uint8_t>(*s)) >> 4]; }
inline bool is_trail(char c) { return static_cast<signed char>(c) < -0x40; }
inline bool valid_codepoint(uint32_t c) { return c < 0xD800 || (c >= 0xE000 && c <= 0x10FFFF); }
constexpr uint32_t kUnicodeError = 0xFFFD;
inline uint32_t decode_utf8(const char *b, const char *e, size_t *mblen) {
  const size_t len = static_cast<size_t>(e - b);
  const uint8_t c0 = static_cast<uint8_t>(b[0]);
  if (c0 < 0x80) {
    *mblen = 1;
    return c0;
  }
  if (len >= 2 && (c0 & 0xE0) == 0xC0) {
    const uint32_t cp = ((c0 & 0x1Fu) << 6) | (static_cast<uint8_t>(b[1]) & 0x3Fu);
    if (is_trail(b[1]) && cp >= 0x80 && valid_codepoint(cp)) {
      *mblen = 2;
      return cp;
    }
  } else if (len >= 3 && (c0 & 0xF0) == 0xE0) {
    const uint32_t cp = ((c0 & 0x0Fu) << 12) | ((static_cast<uint8_t>(b[1]) & 0x3Fu) << 6) | (static_cast<uint8_t>(b[2]) & 0x3Fu);
    if (is_trail(b[1]) && is_trail(b[2]) && cp >= 0x800 && valid_codepoint(cp)) {
      *mblen = 3;
      return cp;
    }
  } else if (len >= 4 && (c0 & 0xF8) == 0xF0) {
    const uint32_t cp = ((c0 & 0x07u) << 18) | ((static_cast<uint8_t>(b[1]) & 0x3Fu) << 12) |
                        ((static_cast<uint8_t>(b[2]) & 0x3Fu) << 6) | (static_cast<uint8_t>(b[3]) & 0x3Fu);
    if (is_trail(b[1]) && is_trail(b[2]) && is_trail(b[3]) && cp >= 0x10000 && valid_codepoint(cp)) {
      *mblen = 4;
      return cp;
    }
  }
  *mblen = 1;
  return kUnicodeError;
}
inline bool valid_decode_utf8(std::string_view in, size_t *mblen) {
  const uint32_t c = decode_utf8(in.data(), in.data() + in.size(), mblen);
  return c != kUnicodeError || *mblen == 3;
}

// protobuf wire format, as much as ModelProto needs (varint, 64-bit, length-delimited, 32-bit)
class Wire {
 public:
  Wire(const uint8_t *p, size_t n) : p_(p), end_(p + n) {}
  bool more() const { return p_ < end_; }
  uint64_t varint() {
    uint64_t v = 0;
    for (int shift = 0; shift < 64; shift += 7) {
      if (p_ >= end_) throw std::runtime_error("sentencepiece model: truncated varint");
      const uint8_t b = *p_++;
      v |= static_cast<uint64_t>(b & 0x7F) << shift;
      if (!(b & 0x80)) return v;
    }
    throw std::runtime_error("sentencepiece model: varint too long");
  }
  // reads one key; for length-delimited fields `bytes` is the payload, for the others `value` holds the number
  void field(uint32_t *number, uint32_t *wire, uint64_t *value, std::string_view *bytes) {
    const uint64_t key = varint();
    *number = static_cast<uint32_t>(key >> 3), *wire = static_cast<uint32_t>(key & 7);
    *value = 0, *bytes = std::string_view();
    switch (*wire) {
      case 0: *value = varint(); break;
      case 1: *value = fixed(8); break;
      case 5: *value = fixed(4); break;
      case 2: {
        const uint64_t n = varint();
        if (n > static_cast<uint64_t>(end_ - p_)) throw std::runtime_error("sentencepiece model: truncated field");
        *bytes = std::string_view(reinterpret_cast<const char *>(p_), static_cast<size_t>(n));
        p_ += n;
        break;
      }
      default: throw std::runtime_error("sentencepiece model: unsupported wire type");
    }
  }

 private:
  uint64_t fixed(int n) {
    if (end_ - p_ < n) throw std::runtime_error("sentencepiece model: truncated fixed field");
    uint64_t v = 0;
    std::memcpy(&v, p_, static_cast<size_t>(n));  // little endian host (x86-64)
    p_ += n;
    return v;
  }
  const uint8_t *p_, *end_;
};

// A byte trie over a set of keys with one int per key: what sentencepiece builds as a Darts double array
// (unigram_model.cc BuildTrie, normalizer.cc PrefixMatcher).  Only the set of matches and their order by length
// matter to the callers, not the array layout, so this is a flat child table.
class ByteTrie {
 public:
  void build(const std::vector<std::pair<std::string_view, int>> &keys) {
    std::vector<std::map<uint8_t, int>> kids(1);
    std::vector<int> val(1, -1);
    for (const auto &[key, value] : keys) {
      int node = 0;
      for (char ch : key) {
        const uint8_t c = static_cast<uint8_t>(ch);
        auto it = kids[node].find(c);
        if (it == kids[node].end()) {
          kids.emplace_back();
          val.push_back(-1);
          it = kids[node].emplace(c, static_cast<int>(kids.size()) - 1).first;
        }
        node = it->second;
      }
      val[node] = value;
    }
    first_.assign(kids.size() + 1, 0);
    value_ = std::move(val);
    for (size_t n = 0; n < kids.size(); n++) first_[n + 1] = first_[n] + static_cast<int>(kids[n].size());
    label_.resize(first_.back()), child_.resize(first_.back());
    for (size_t n = 0; n < kids.size(); n++) {
      int k = first_[n];
      for (const auto &[c, to] : kids[n]) label_[k] = c, child_[k] = to, k++;
    }
    // nodes with many children (the root, the node behind U+2581, ...) get a direct 256-entry table
    dense_of_.assign(kids.size(), -1);
    dense_.clear();
    for (size_t n = 0; n < kids.size(); n++) {
      if (n != 0 && kids[n].size() <= kDenseFrom) continue;
      dense_of_[n] = static_cast<int>(dense_.size() / 256);
      dense_.resize(dense_.size() + 256, -1);
      for (const auto &[c, to] : kids[n]) dense_[dense_.size() - 256 + c] = to;
    }
  }
  bool empty() const { return value_.size() <= 1; }
  size_t dense_nodes() const { return dense_.size() / 256; }
  // one step from `node` along byte c: the child or -1
  int step(int node, uint8_t c) const {
    const int d = dense_of_[node];
    if (d >= 0) return dense_[static_cast<size_t>(d) * 256 + c];
    for (int k = first_[node], e = first_[node + 1]; k < e; k++)  // at most kDenseFrom sorted labels
      if (label_[k] >= c) return label_[k] == c ? child_[k] : -1;
    return -1;
  }
  int value(int node) const { return value_[node]; }
  // length of the longest key that is a prefix of s (0: none)
  size_t longest_prefix(std::string_view s) const {
    size_t best = 0;
    int node = 0;
    for (size_t i = 0; i < s.size() && !empty(); i++) {
      node = step(node, static_cast<uint8_t>(s[i]));
      if (node < 0) break;
      if (value_[node] >= 0) best = i + 1;
    }
    return best;
  }

 private:
  static constexpr size_t kDenseFrom = 6;
  std::vector<int> first_, child_, value_, dense_of_, dense_;
  std::vector<uint8_t> label_;
};

// The slice of sentencepiece::SentencePieceProcessor that slimt::Vocabulary calls (Vocabulary.cc:24-104): Load /
// LoadFromSerializedProto, Encode(line, SentencePieceText*), Decode(ids, SentencePieceText*), eos_id, pad_id,
// GetPieceSize.  The library is a vendored third-party dependency of the reference (3rd-party/sentencepiece, version
// 0.2.00); its algorithm is restated here, each function naming the library function it follows, and pinned against the
// sentencepiece Python wheel of this image on a committed fixture model (tests/test_text_front.py).
class Processor {
 public:
  enum Type { NORMAL = 1, UNKNOWN = 2, CONTROL = 3, USER_DEFINED = 4, UNUSED = 5, BYTE = 6 };  // sentencepiece_model.proto:290-299
  struct Piece {
    std::string piece;
    float score = 0.0F;
    int type = NORMAL;
  };
  // one entry of SentencePieceText.pieces (sentencepiece.proto): [begin, end) are byte offsets into the ORIGINAL input
  // (Encode) or into the decoded text (Decode)
  struct Span {
    int id = 0;
    std::string piece;
    std::string surface;
    size_t begin = 0, end = 0;
  };

  Processor() = default;
  void load(const std::string &path) {
    std::ifstream in(path, std::ios::binary);
    if (!in) throw std::runtime_error("sentencepiece model: cannot open " + path);
    std::string blob((std::istreambuf_iterator<char>(in)), std::istreambuf_iterator<char>());
    load(blob.data(), blob.size());
  }
  // ModelProto (sentencepiece_model.proto:309-324): pieces = 1, trainer_spec = 2, normalizer_spec = 3, denormalizer_spec = 5
  void load(const void *data, size_t size) {
    *this = Processor();
    Wire top(static_cast<const uint8_t *>(data), size);
    uint32_t num, wire;
    uint64_t value;
    std::string_view bytes;
    while (top.more()) {
      top.field(&num, &wire, &value, &bytes);
      if (num == 1 && wire == 2) {
        Piece piece;
        Wire w(reinterpret_cast<const uint8_t *>(bytes.data()), bytes.size());
        while (w.more()) {
          uint32_t n, t;
          uint64_t v;
          std::string_view b;
          w.field(&n, &t, &v, &b);
          if (n == 1 && t == 2) piece.piece.assign(b);
          if (n == 2 && t == 5) {
            const uint32_t bits = static_cast<uint32_t>(v);
            std::memcpy(&piece.score, &bits, 4);
          }
          if (n == 3 && t == 0) piece.type = static_cast<int>(v);
        }
        pieces_.push_back(std::move(piece));
      } else if (num == 2 && wire == 2) {
        Wire w(reinterpret_cast<const uint8_t *>(bytes.data()), bytes.size());
        while (w.more()) {
          uint32_t n, t;
          uint64_t v;
          std::string_view b;
          w.field(&n, &t, &v, &b);
          if (n == 3 && t == 0) model_type_ = static_cast<int>(v);          // TrainerSpec.model_type (UNIGRAM = 1)
          if (n == 24 && t == 0) whitespace_as_suffix_ = v != 0;           // treat_whitespace_as_suffix
          if (n == 35 && t == 0) byte_fallback_ = v != 0;                  // byte_fallback
          if (n == 44 && t == 2) unk_surface_.assign(b);                   // unk_surface
          if (n == 45 && t == 2) unk_piece_.assign(b);
          if (n == 46 && t == 2) bos_piece_.assign(b);
          if (n == 47 && t == 2) eos_piece_.assign(b);
          if (n == 48 && t == 2) pad_piece_.assign(b);
        }
      } else if ((num == 3 || num == 5) && wire == 2) {
        Wire w(reinterpret_cast<const uint8_t *>(bytes.data()), bytes.size());
        while (w.more()) {
          uint32_t n, t;
          uint64_t v;
          std::string_view b;
          w.field(&n, &t, &v, &b);
          if (num == 5) {  // denormalizer_spec: only an empty one is supported
            if (n == 2 && t == 2 && !b.empty()) throw std::runtime_error("sentencepiece model: denormalizer rules are not supported");
            continue;
          }
          if (n == 2 && t == 2) charsmap_.assign(b);        // NormalizerSpec.precompiled_charsmap
          if (n == 3 && t == 0) add_dummy_prefix_ = v != 0;
          if (n == 4 && t == 0) remove_extra_whitespaces_ = v != 0;
          if (n == 5 && t == 0) escape_whitespaces_ = v != 0;
        }
      }
    }
    initialize();
  }

  int size() const { return static_cast<int>(pieces_.size()); }  // GetPieceSize
  const Piece &piece(int id) const { return pieces_.at(static_cast<size_t>(id)); }
  bool is_control(int id) const { return in_range(id) && pieces_[id].type == CONTROL; }
  bool is_unknown(int id) const { return in_range(id) && pieces_[id].type == UNKNOWN; }
  bool is_byte(int id) const { return in_range(id) && pieces_[id].type == BYTE; }
  // ModelInterface::PieceToId (model_interface.cc:51-61)
  int piece_to_id(std::string_view piece) const {
    auto it = ids_.find(std::string(piece));
    return it == ids_.end() ? unk_id_ : it->second;
  }
  // sentencepiece_processor.cc:962-984: looked up by the trainer's piece names, and only if of the right type
  int unk_id() const {
    const int id = piece_to_id(unk_piece_);
    return is_unknown(id) ? id : -1;
  }
  int eos_id() const {
    const int id = piece_to_id(eos_piece_);
    return is_control(id) ? id : -1;
  }
  int bos_id() const {
    const int id = piece_to_id(bos_piece_);
    return is_control(id) ? id : -1;
  }
  int pad_id() const {
    const int id = piece_to_id(pad_piece_);
    return is_control(id) ? id : -1;
  }

  // Normalizer::Normalize (normalizer.cc:72-197): NFKC-style rewriting through the precompiled character map, leading /
  // trailing / repeated whitespace removed, the dummy prefix added, blanks escaped to U+2581; norm_to_orig[i] = offset in
  // the input of the character normalized byte i came from, plus one closing entry.
  void normalize(std::string_view input, std::string *normalized, std::vector<size_t> *norm_to_orig) const {
    normalized->clear(), norm_to_orig->clear();
    if (input.empty()) return;
    int consumed = 0;
    if (remove_extra_whitespaces_) {
      while (!input.empty()) {
        const auto p = normalize_prefix(input);
        if (p.first != " ") break;
        input.remove_prefix(static_cast<size_t>(p.second));
        consumed += p.second;
      }
    }
    if (input.empty()) return;
    static constexpr std::string_view kSpace = "\xe2\x96\x81";
    auto add_ws = [&]() {
      if (escape_whitespaces_) {
        normalized->append(kSpace);
        norm_to_orig->insert(norm_to_orig->end(), kSpace.size(), static_cast<size_t>(consumed));
      } else {
        normalized->push_back(' ');
        norm_to_orig->push_back(static_cast<size_t>(consumed));
      }
    };
    if (!whitespace_as_suffix_ && add_dummy_prefix_) add_ws();
    bool prev_space = remove_extra_whitespaces_;
    while (!input.empty()) {
      // an ASCII byte that starts no rule and no user-defined symbol maps to itself: the common case, without the walk
      const uint8_t c0 = static_cast<uint8_t>(input.front());
      if (c0 != ' ' && plain_ascii_[c0]) {
        normalized->push_back(static_cast<char>(c0));
        norm_to_orig->push_back(static_cast<size_t>(consumed));
        prev_space = false;
        consumed += 1;
        input.remove_prefix(1);
        continue;
      }
      const auto p = normalize_prefix(input);
      std::string_view sp = p.first;
      while (prev_space && !sp.empty() && sp.front() == ' ') sp.remove_prefix(1);
      if (!sp.empty()) {
        for (char c : sp) {
          if (escape_whitespaces_ && c == ' ') {
            normalized->append(kSpace);
            norm_to_orig->insert(norm_to_orig->end(), kSpace.size(), static_cast<size_t>(consumed));
          } else {
            normalized->push_back(c);
            norm_to_orig->push_back(static_cast<size_t>(consumed));
          }
        }
        prev_space = sp.back() == ' ';
      }
      consumed += p.second;
      input.remove_prefix(static_cast<size_t>(p.second));
      if (!remove_extra_whitespaces_) prev_space = false;
    }
    if (remove_extra_whitespaces_) {
      const std::string_view space = escape_whitespaces_ ? kSpace : std::string_view(" ");
      while (normalized->size() >= space.size() &&
             normalized->compare(normalized->size() - space.size(), space.size(), space) == 0) {
        const size_t length = normalized->size() - space.size();
        consumed = static_cast<int>((*norm_to_orig)[length]);
        normalized->resize(length), norm_to_orig->resize(length);
      }
    }
    if (whitespace_as_suffix_ && add_dummy_prefix_) add_ws();
    norm_to_orig->push_back(static_cast<size_t>(consumed));
  }

  // SentencePieceProcessor::Encode(input, SentencePieceText*) (sentencepiece_processor.cc:633-646): Normalize, the
  // model's Encode, PopulateSentencePieceText (:542-631: offsets mapped back to the input, runs of unknown pieces
  // merged, byte fallback).
  std::vector<Span> encode(std::string_view input) const {
    std::vector<Span> out;
    encode_walk(input, [&](int id, std::string_view w, size_t ob, size_t oe, bool merge, bool has_surface) {
      const std::string_view surface = has_surface ? input.substr(ob, oe - ob) : std::string_view();
      if (merge) {
        Span &s = out.back();
        s.piece.append(w), s.surface.append(surface), s.end = oe;
      } else {
        Span s;
        s.id = id, s.piece.assign(w), s.surface.assign(surface), s.begin = ob, s.end = oe;
        out.push_back(std::move(s));
      }
    });
    return out;
  }
  // the same walk for callers that only want what slimt::Vocabulary keeps: the ids and each piece's byte range
  void encode(std::string_view input, std::vector<uint32_t> *ids, std::vector<std::pair<size_t, size_t>> *ranges) const {
    ids->clear(), ranges->clear();
    encode_walk(input, [&](int id, std::string_view, size_t ob, size_t oe, bool merge, bool) {
      if (merge) {
        ranges->back().second = oe;
      } else {
        ids->push_back(static_cast<uint32_t>(id)), ranges->emplace_back(ob, oe);
      }
    });
  }

 private:
  // PopulateSentencePieceText (sentencepiece_processor.cc:542-631) as a walk: emit(id, piece, begin, end, merge, has_surface)
  // once per output piece; merge = a run of unknown pieces continues (the previous piece grows, no new one)
  template <class Emit>
  void encode_walk(std::string_view input, Emit &&emit) const {
    thread_local std::string normalized;
    thread_local std::vector<size_t> n2o;
    thread_local std::vector<std::pair<std::string_view, int>> result;
    normalize(input, &normalized, &n2o);
    encode_unigram(normalized, &result);
    size_t consumed = 0;
    bool prev_unk = false;
    for (const auto &[w, id] : result) {
      const bool unk = is_unknown(id);
      const size_t begin = consumed, end = consumed + w.size();
      if (end >= n2o.size()) throw std::runtime_error("sentencepiece: piece outside the normalized text");
      const size_t ob = n2o[begin], oe = n2o[end];
      if (ob > input.size() || oe > input.size() || ob > oe) throw std::runtime_error("sentencepiece: inconsistent offsets");
      if (unk && byte_fallback_) {
        for (size_t i = 0; i < w.size(); i++) {
          const std::string piece = byte_to_piece(static_cast<uint8_t>(w[i]));
          const bool last = i + 1 == w.size();
          emit(piece_to_id(piece), std::string_view(piece), ob, last ? oe : ob, false, last);
        }
      } else {
        emit(id, w, ob, oe, prev_unk && unk, true);
      }
      consumed += w.size();
      prev_unk = unk;
    }
    if (consumed != normalized.size()) throw std::runtime_error("sentencepiece: all normalized characters are not consumed");
  }

 public:

  // SentencePieceProcessor::Decode(ids, SentencePieceText*) (sentencepiece_processor.cc:754-917).  Returns false for an id
  // outside the vocabulary (the library returns an OUT_OF_RANGE status and leaves the text empty).
  bool decode(const std::vector<int> &ids, std::string *text, std::vector<Span> *spans) const {
    std::vector<std::pair<size_t, size_t>> ranges;
    spans->clear();
    if (!decode(ids, text, &ranges)) return false;
    for (size_t i = 0; i < ids.size(); i++) {
      Span s;
      s.id = ids[i], s.piece = pieces_[ids[i]].piece, s.begin = ranges[i].first, s.end = ranges[i].second;
      s.surface = text->substr(s.begin, s.end - s.begin);
      spans->push_back(std::move(s));
    }
    return true;
  }
  // the text and, per id, the byte range of its surface in it.  (Decode goes id -> piece -> id; pieces are unique --
  // checked at load -- so the round trip is the identity and is not made.)
  template <class Id>
  bool decode(const std::vector<Id> &ids, std::string *text, std::vector<std::pair<size_t, size_t>> *ranges) const {
    text->clear();
    ranges->assign(ids.size(), {0, 0});
    for (Id id : ids)
      if (!in_range(static_cast<int>(id))) {
        ranges->clear();
        return false;
      }
    static constexpr std::string_view kSpace = "\xe2\x96\x81";
    auto set_surface = [&](size_t i, std::string_view surface) {
      (*ranges)[i] = {text->size(), text->size() + surface.size()};
      text->append(surface);
    };
    auto byte_run = [&](size_t from, size_t to) {  // a run of byte pieces: one surface per UTF-8 character, on its last byte
      if (from >= to) return;
      std::string bytes;
      for (size_t i = from; i < to; i++) bytes.push_back(static_cast<char>(piece_to_byte(pieces_[ids[i]].piece)));
      size_t offset = 0;
      while (offset < bytes.size()) {
        size_t used = 0;
        const bool ok = valid_decode_utf8(std::string_view(bytes).substr(offset), &used);
        if (!ok) {
          set_surface(from + offset, "\xEF\xBF\xBD");
        } else {
          for (size_t j = 0; j < used; j++)
            set_surface(from + offset + j, j + 1 == used ? std::string_view(bytes).substr(offset, used) : std::string_view());
        }
        offset += used;
      }
    };
    size_t byte_start = 0;
    bool is_bos_ws = true, bos_ws_seen = false;
    for (size_t i = 0; i < ids.size(); i++) {
      const Piece &p = pieces_[ids[i]];
      if (p.type == BYTE) continue;
      byte_run(byte_start, i);
      if (bos_ws_seen || !text->empty()) is_bos_ws = false;
      byte_start = i + 1;
      bos_ws_seen = false;
      const size_t begin = text->size();
      if (p.type == CONTROL) {
        // invisible
      } else if (p.type == UNKNOWN) {
        text->append(unk_surface_);
      } else {
        std::string_view piece = p.piece;
        if (is_bos_ws && (add_dummy_prefix_ || remove_extra_whitespaces_)) {
          if (piece.substr(0, kSpace.size()) == kSpace) piece.remove_prefix(kSpace.size()), bos_ws_seen = true;
          if (remove_extra_whitespaces_) bos_ws_seen = false;
        }
        for (size_t k = 0; k < piece.size();) {
          if (piece[k] == kSpace[0] && piece.compare(k, kSpace.size(), kSpace) == 0) {
            text->push_back(' ');
            k += kSpace.size();
          } else {
            text->push_back(piece[k++]);
          }
        }
      }
      (*ranges)[i] = {begin, text->size()};
    }
    byte_run(byte_start, ids.size());
    return true;
  }

 private:
  bool in_range(int id) const { return id >= 0 && id < static_cast<int>(pieces_.size()); }
  static std::string byte_to_piece(uint8_t c) {  // model_interface.cc:193-195
    char buf[8];
    std::snprintf(buf, sizeof(buf), "<0x%02X>", c);
    return buf;
  }
  static int piece_to_byte(std::string_view piece) {  // model_interface.cc:197-212
    if (piece.size() != 6 || piece.substr(0, 3) != "<0x" || piece[5] != '>') return -1;
    auto hex = [](char c) { return c >= '0' && c <= '9' ? c - '0' : (c >= 'A' && c <= 'F' ? c - 'A' + 10 : -1); };
    const int hi = hex(piece[3]), lo = hex(piece[4]);
    return (hi < 0 || lo < 0) ? -1 : hi * 16 + lo;
  }

  // ModelInterface::InitializePieces (model_interface.cc:63-137), unigram Model::Model (unigram_model.cc:653-671),
  // Normalizer::Init (normalizer.cc:42-70)
  void initialize() {
    if (model_type_ != 1) throw std::runtime_error("sentencepiece model: only unigram models are supported (model_type " + std::to_string(model_type_) + ")");
    unk_id_ = -1;
    min_score_ = FLT_MAX, max_score_ = FLT_MIN;
    std::vector<std::pair<std::string_view, int>> normal, user;
    std::array<bool, 256> byte_found{};
    for (int i = 0; i < static_cast<int>(pieces_.size()); i++) {
      const Piece &p = pieces_[i];
      if (p.piece.empty()) throw std::runtime_error("sentencepiece model: piece must not be empty");
      if (!ids_.emplace(p.piece, i).second) throw std::runtime_error("sentencepiece model: " + p.piece + " is already defined");
      if (p.type == NORMAL || p.type == USER_DEFINED || p.type == UNUSED) normal.emplace_back(p.piece, i);
      if (p.type == USER_DEFINED) user.emplace_back(p.piece, i);
      if (p.type == UNKNOWN) {
        if (unk_id_ >= 0) throw std::runtime_error("sentencepiece model: unk is already defined");
        unk_id_ = i;
      }
      if (p.type == BYTE) {
        const int b = piece_to_byte(p.piece);
        if (!byte_fallback_ || b < 0) throw std::runtime_error("sentencepiece model: unexpected byte piece " + p.piece);
        byte_found[static_cast<size_t>(b)] = true;
      }
      if (p.type == NORMAL) min_score_ = std::min(min_score_, p.score), max_score_ = std::max(max_score_, p.score);
    }
    if (unk_id_ < 0) throw std::runtime_error("sentencepiece model: unk is not defined");
    if (byte_fallback_ && std::find(byte_found.begin(), byte_found.end(), false) != byte_found.end())
      throw std::runtime_error("sentencepiece model: byte_fallback without 256 byte pieces");
    trie_.build(normal);
    user_.build(user);
    score_.clear(), type_.clear();
    for (const Piece &p : pieces_) score_.push_back(p.score), type_.push_back(static_cast<uint8_t>(p.type));
    // precompiled_charsmap = u32 size of the trie blob, the Darts double array (u32 units), the replacement strings
    // (NUL-terminated, indexed by the trie's values)  (normalizer.cc:275-309)
    if (!charsmap_.empty()) {
      uint32_t trie_bytes = 0;
      if (charsmap_.size() <= 4) throw std::runtime_error("sentencepiece model: blob for normalization rule is broken");
      std::memcpy(&trie_bytes, charsmap_.data(), 4);
      if (trie_bytes >= charsmap_.size() || 4 + static_cast<size_t>(trie_bytes) > charsmap_.size() || trie_bytes % 4 != 0)
        throw std::runtime_error("sentencepiece model: trie data size exceeds the input blob size");
      darts_.resize(trie_bytes / 4);
      std::memcpy(darts_.data(), charsmap_.data() + 4, trie_bytes);
      replacements_at_ = 4 + static_cast<size_t>(trie_bytes);
    }
    // bytes below 0x80 for which NormalizePrefix is the identity: no rule of the character map and no user-defined
    // symbol starts with them
    for (int c = 0; c < 256; c++) {
      const char ch = static_cast<char>(c);
      size_t length = 0;
      uint32_t value = 0;
      plain_ascii_[c] = c < 0x80 && !darts_has_prefix(ch) && user_.step(0, static_cast<uint8_t>(c)) < 0 &&
                        !darts_longest(std::string_view(&ch, 1), &length, &value);
    }
  }

  // Darts::DoubleArray::commonPrefixSearch restricted to what NormalizePrefix keeps: the LONGEST key that is a prefix of
  // the input and its value (darts.h: unit = u32; has_leaf bit 8, value low 31 bits, label = unit & (1u<<31 | 0xFF),
  // offset = (unit >> 10) << ((unit & 512) >> 6)).
  bool darts_longest(std::string_view s, size_t *length, uint32_t *value) const {
    if (darts_.empty()) return false;
    auto offset = [](uint32_t u) { return (u >> 10) << ((u & (1u << 9)) >> 6); };
    size_t pos = 0;
    uint32_t unit = darts_[pos];
    pos ^= offset(unit);
    bool found = false;
    for (size_t i = 0; i < s.size(); i++) {
      const uint8_t c = static_cast<uint8_t>(s[i]);
      pos ^= c;
      if (pos >= darts_.size()) break;
      unit = darts_[pos];
      if ((unit & ((1u << 31) | 0xFFu)) != c) break;
      pos ^= offset(unit);
      if (pos >= darts_.size()) break;
      if ((unit >> 8) & 1u) {
        *length = i + 1, *value = darts_[pos] & ((1u << 31) - 1);
        found = true;
      }
    }
    return found;
  }

  // does any key of the character map start with byte c?
  bool darts_has_prefix(char ch) const {
    if (darts_.empty()) return false;
    auto offset = [](uint32_t u) { return (u >> 10) << ((u & (1u << 9)) >> 6); };
    const uint8_t c = static_cast<uint8_t>(ch);
    size_t pos = offset(darts_[0]) ^ c;
    return pos < darts_.size() && (darts_[pos] & ((1u << 31) | 0xFFu)) == c;
  }

  // Normalizer::NormalizePrefix (normalizer.cc:195-254): (replacement text, input bytes consumed)
  std::pair<std::string_view, int> normalize_prefix(std::string_view input) const {
    if (input.empty()) return {std::string_view(), 0};
    if (!user_.empty()) {  // user-defined symbols pass through untouched (PrefixMatcher::PrefixMatch)
      const size_t n = user_.longest_prefix(input);
      if (n > 0) return {input.substr(0, n), static_cast<int>(n)};
    }
    size_t length = 0;
    uint32_t value = 0;
    if (darts_longest(input, &length, &value)) {
      const std::string_view table = std::string_view(charsmap_).substr(replacements_at_);
      if (value >= table.size()) throw std::runtime_error("sentencepiece model: normalization rule outside its table");
      const char *s = table.data() + value;
      const void *nul = std::memchr(s, 0, table.size() - value);
      const size_t n = nul ? static_cast<size_t>(static_cast<const char *>(nul) - s) : table.size() - value;
      return {std::string_view(s, n), static_cast<int>(length)};
    }
    size_t mblen = 0;
    if (!valid_decode_utf8(input, &mblen)) return {std::string_view("\xEF\xBF\xBD"), 1};
    return {input.substr(0, mblen), static_cast<int>(mblen)};
  }

  // unigram Model::EncodeOptimized (unigram_model.cc:529-640): Viterbi over the piece trie without a lattice; an
  // unknown character costs min_score - 10; a user-defined piece scores length * max_score - 0.1; the first of
  // equally good paths is kept (strict >).  The arithmetic types follow the library's (float scores, the candidate sum
  // formed in double when a user-defined piece is involved, stored back as float).
  struct ViterbiNode {
    int id = -1;
    float score = 0.0F;
    int starts_at = -1;
  };
  void encode_unigram(std::string_view normalized, std::vector<std::pair<std::string_view, int>> *out) const {
    std::vector<std::pair<std::string_view, int>> &results = *out;
    results.clear();
    if (normalized.empty()) return;
    using Node = ViterbiNode;
    const int size = static_cast<int>(normalized.size());
    const float unk_score = min_score_ - 10.0F;
    thread_local std::vector<Node> best;
    best.assign(static_cast<size_t>(size) + 1, Node());
    int starts_at = 0;
    while (starts_at < size) {
      const float till_here = best[starts_at].score;
      bool has_single = false;
      const int mblen = std::min<int>(static_cast<int>(one_char_len(normalized.data() + starts_at)), size - starts_at);
      int node = 0;
      for (int key_pos = starts_at; key_pos < size;) {
        node = trie_.step(node, static_cast<uint8_t>(normalized[key_pos]));
        key_pos++;
        if (node < 0) break;
        const int ret = trie_.value(node);
        if (ret < 0) continue;
        const uint8_t type = type_[ret];
        if (type == UNUSED) continue;
        Node &target = best[key_pos];
        const size_t length = static_cast<size_t>(key_pos - starts_at);
        bool better;
        float stored;
        if (type == USER_DEFINED) {
          const double cand = (static_cast<float>(length) * max_score_ - 0.1) + static_cast<double>(till_here);
          better = target.starts_at == -1 || cand > static_cast<double>(target.score);
          stored = static_cast<float>(cand);
        } else {
          // GetScoreInlined is a float, but the ternary it sits in has type double: the sum is formed in double
          const double cand = static_cast<double>(score_[ret]) + static_cast<double>(till_here);
          better = target.starts_at == -1 || cand > static_cast<double>(target.score);
          stored = static_cast<float>(cand);
        }
        if (better) target.score = stored, target.starts_at = starts_at, target.id = ret;
        if (!has_single && length == static_cast<size_t>(mblen)) has_single = true;
      }
      if (!has_single) {
        Node &target = best[starts_at + mblen];
        const float cand = unk_score + till_here;
        if (target.starts_at == -1 || cand > target.score) target.score = cand, target.starts_at = starts_at, target.id = unk_id_;
      }
      starts_at += mblen;
    }
    for (int ends_at = size; ends_at > 0;) {
      const Node &n = best[ends_at];
      results.emplace_back(normalized.substr(static_cast<size_t>(n.starts_at), static_cast<size_t>(ends_at - n.starts_at)), n.id);
      ends_at = n.starts_at;
    }
    std::reverse(results.begin(), results.end());
  }

  std::vector<Piece> pieces_;
  std::array<bool, 256> plain_ascii_{};
  std::vector<float> score_;   // pieces_[i].score / .type once more, packed for the Viterbi loop
  std::vector<uint8_t> type_;
  std::unordered_map<std::string, int> ids_;
  ByteTrie trie_, user_;
  int unk_id_ = -1;
  float min_score_ = FLT_MAX, max_score_ = FLT_MIN;
  int model_type_ = 1;
  bool byte_fallback_ = false, whitespace_as_suffix_ = false;
  bool add_dummy_prefix_ = true, remove_extra_whitespaces_ = true, escape_whitespaces_ = true;
  std::string unk_surface_ = " \xE2\x81\x87 ", unk_piece_ = "<unk>", bos_piece_ = "<s>", eos_piece_ = "</s>", pad_piece_ = "<pad>";
  std::string charsmap_;
  std::vector<uint32_t> darts_;
  size_t replacements_at_ = 0;  // where the replacement strings start in charsmap_
};

}  // namespace spm

// ---------------------------------------------------------------- Vocabulary (slimt/Vocabulary.hh, Vocabulary.cc)
class Vocabulary {
 public:
  explicit Vocabulary(const std::string &fpath) { processor_.load(fpath); }
  explicit Vocabulary(View view) { processor_.load(view.data, view.size); }
  Vocabulary(const Vocabulary &other) = delete;  // (the processor's tables hold views into its own strings)
  Vocabulary &operator=(const Vocabulary &) = delete;

  // Vocabulary.cc:35-79: word ids of `line` and, for each, the bytes of `line` it came from (views INTO line)
  std::tuple<Words, Views> encode(const std::string_view &line, bool add_eos = false) const {
    Words words;
    thread_local std::vector<std::pair<size_t, size_t>> ranges;
    processor_.encode(line, &words, &ranges);
    Views views;
    views.reserve(ranges.size());
    for (const auto &[b, e] : ranges) views.push_back(line.substr(b, e - b));
    if (add_eos) words.push_back(eos_id());
    return {std::move(words), std::move(views)};
  }
  // Vocabulary.cc:81-104: the text of `words` in `decoded` and one view into it per word; with ignore_eos the last
  // view (the EOS the decoder closed the sentence with) is dropped
  Views decode(const Words &words, std::string &decoded, bool ignore_eos = true) const {
    thread_local std::vector<std::pair<size_t, size_t>> ranges;
    Views views;
    processor_.decode(words, &decoded, &ranges);  // (an id outside the vocabulary: empty text, no views)
    views.reserve(ranges.size());
    for (const auto &[b, e] : ranges) views.emplace_back(decoded.data() + b, e - b);
    if (ignore_eos && !views.empty()) views.pop_back();
    return views;
  }
  Word pad_id() const { return static_cast<Word>(std::max(0, processor_.pad_id())); }
  Word eos_id() const { return static_cast<Word>(processor_.eos_id()); }
  size_t size() const { return static_cast<size_t>(processor_.size()); }
  const spm::Processor &processor() const { return processor_; }

 private:
  spm::Processor processor_;
};

// ---------------------------------------------------------------- Regex (slimt/Regex.hh) over the system's PCRE2
// The reference links libpcre2-8; this image carries the run-time library without its header, so the handful of entry
// points Regex.cc uses are bound with dlopen (prototypes from PCRE2's published API, 8-bit code unit width).
namespace pcre2 {
constexpr uint32_t ANCHORED = 0x80000000u, NO_UTF_CHECK = 0x40000000u, DOTALL = 0x00000020u, UTF = 0x00080000u;
constexpr uint32_t NEWLINE_ANY = 4;  // Splitter.cc ORs this newline CODE into the compile options (:134, :160); kept as written
constexpr uint32_t JIT_COMPLETE = 1, CONFIG_JIT = 1;
struct Api {
  void *(*compile)(const uint8_t *, size_t, uint32_t, int *, size_t *, void *) = nullptr;
  int (*jit_compile)(void *, uint32_t) = nullptr;
  int (*config)(uint32_t, void *) = nullptr;
  void *(*match_data_create_from_pattern)(const void *, void *) = nullptr;
  int (*match)(const void *, const uint8_t *, size_t, size_t, uint32_t, void *, void *) = nullptr;
  size_t *(*get_ovector_pointer)(void *) = nullptr;
  size_t (*get_startchar)(void *) = nullptr;
  int (*get_error_message)(int, uint8_t *, size_t) = nullptr;
  void (*match_data_free)(void *) = nullptr;
  void (*code_free)(void *) = nullptr;
  static const Api &get() {
    static const Api api = []() {
      Api a;
      void *lib = nullptr;
      for (const char *name : {"libpcre2-8.so.0", "libpcre2-8.so"})
        if ((lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL)) != nullptr) break;
      if (lib == nullptr) throw std::runtime_error("sentence splitter: libpcre2-8 not found (dlopen)");
      auto bind = [lib](auto &fn, const char *sym) {
        void *p = dlsym(lib, sym);
        if (p == nullptr) throw std::runtime_error(std::string("sentence splitter: libpcre2-8 lacks ") + sym);
        fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(p);
      };
      bind(a.compile, "pcre2_compile_8"), bind(a.jit_compile, "pcre2_jit_compile_8"), bind(a.config, "pcre2_config_8");
      bind(a.match_data_create_from_pattern, "pcre2_match_data_create_from_pattern_8"), bind(a.match, "pcre2_match_8");
      bind(a.get_ovector_pointer, "pcre2_get_ovector_pointer_8"), bind(a.get_startchar, "pcre2_get_startchar_8");
      bind(a.get_error_message, "pcre2_get_error_message_8");
      bind(a.match_data_free, "pcre2_match_data_free_8"), bind(a.code_free, "pcre2_code_free_8");
      return a;
    }();
    return api;
  }
};
}  // namespace pcre2

class Regex;
class Match {  // Regex.hh:51-60
 public:
  explicit Match(const Regex &re);
  ~Match() { pcre2::Api::get().match_data_free(match_data); }
  Match(const Match &) = delete;
  Match &operator=(const Match &) = delete;
  std::string_view operator[](int i) const {
    const size_t *o = pcre2::Api::get().get_ovector_pointer(match_data);
    return std::string_view(data + o[2 * i], o[2 * i + 1] - o[2 * i]);
  }
  void *const match_data;
  const char *data = nullptr;
  int num_matched_groups = 0;
};

class Regex {  // Regex.hh:15-49, Regex.cc:14-77
 public:
  Regex(const std::string &pattern, uint32_t options, uint32_t jit_options = pcre2::JIT_COMPLETE)
      : pattern_(pattern),
        re_(pcre2::Api::get().compile(reinterpret_cast<const uint8_t *>(pattern.c_str()), ~static_cast<size_t>(0), options,
                                      &error_number_, &error_offset_, nullptr)) {
    if (re_ == nullptr) throw std::runtime_error(get_error_message());
    uint32_t have_jit = 0;
    pcre2::Api::get().config(pcre2::CONFIG_JIT, &have_jit);
    if (have_jit) pcre2::Api::get().jit_compile(re_, jit_options);
  }
  ~Regex() { pcre2::Api::get().code_free(re_); }
  Regex(const Regex &) = delete;
  Regex &operator=(const Regex &) = delete;
  // number of matched groups (> 0) or a PCRE2 error code (< 0; -1 = no match)
  int find(std::string_view subj, Match *m, size_t start = 0, uint32_t options = 0) const {
    const int rc = pcre2::Api::get().match(re_, reinterpret_cast<const uint8_t *>(subj.data()), subj.size(), start, options,
                                           m->match_data, nullptr);
    m->data = rc > 0 ? subj.data() : nullptr;
    m->num_matched_groups = rc;
    return rc;
  }
  // an anchored find that, on success, removes the match from the front of *subj
  int consume(std::string_view *subj, Match *m, uint32_t options = 0) const {
    const int rc = find(*subj, m, 0, options | pcre2::ANCHORED);
    if (rc > 0) subj->remove_prefix((*m)[0].size());
    return rc;
  }
  const void *get_pcre2_code() const { return re_; }
  bool ok() const { return re_ != nullptr; }
  std::string get_error_message() const {
    uint8_t buffer[256] = {0};
    pcre2::Api::get().get_error_message(error_number_, buffer, sizeof(buffer));
    std::ostringstream msg;
    msg << "PCRE2 compilation failed at offset " << error_offset_ << ": " << reinterpret_cast<const char *>(buffer);
    return msg.str();
  }

 private:
  std::string pattern_;
  size_t error_offset_ = 0;
  int error_number_ = 0;
  void *const re_;
};
inline Match::Match(const Regex &re) : match_data(pcre2::Api::get().match_data_create_from_pattern(re.get_pcre2_code(), nullptr)) {}

// ---------------------------------------------------------------- Splitter / SentenceStream (slimt/Splitter.hh, Splitter.cc)
namespace detail {
// the line at *start without its end-of-line ('\n', any '\r' before it); data() == nullptr once the buffer is used up
// (Splitter.cc:274-288)
inline std::string_view read_line(const char **start, const char *stop) {
  if (*start == stop) return std::string_view();
  const char *nl = *start;
  while (nl < stop && *nl != '\n') ++nl;
  const char *end = nl;
  while (end > *start && end[-1] == '\r') --end;
  std::string_view line(*start, static_cast<size_t>(end - *start));
  *start = nl == stop ? nl : nl + 1;
  return line;
}
// lines up to the first line break that is followed by another '\n' or '\r': single line breaks are wraps inside a
// paragraph (Splitter.cc:293-314)
inline std::string_view read_paragraph(const char **start, const char *stop) {
  if (*start == stop) return std::string_view();
  const char *nl = *start, *run = nullptr;
  for (;;) {
    while (nl < stop && *nl != '\n') ++nl;
    run = nl;
    while (run < stop && (*run == '\n' || *run == '\r')) ++run;
    if (run < stop && run == nl + 1) {
      ++nl;
      continue;
    }
    break;
  }
  const char *end = nl;
  while (end > *start && end[-1] == '\r') --end;
  std::string_view par(*start, static_cast<size_t>(end - *start));
  *start = run < stop ? run : stop;
  return par;
}
}  // namespace detail

class Splitter {
 public:
  Splitter() = default;
  explicit Splitter(const std::string &prefix_file) {
    if (!prefix_file.empty()) load(prefix_file);
  }
  void load(const std::string &fname) {  // Splitter.cc:21-31
    std::ifstream pfile(fname);
    std::string line;
    while (std::getline(pfile, line)) declare_prefix(line);
  }
  void load_from_serialized(std::string_view buffer) {  // Splitter.cc:49-56
    const char *start = buffer.data(), *stop = buffer.data() + buffer.size();
    for (std::string_view line = detail::read_line(&start, stop); line.data() != nullptr; line = detail::read_line(&start, stop))
      declare_prefix(line);
  }

  // The next sentence of *rest; *rest advances past it (Splitter.cc:126-263).  No UTF-8 validation here (the stream
  // validates once up front).  `limit` is the end of the storage *rest lies in: the reference tests the byte just past the
  // paragraph (Splitter.cc:233), which exists there because the text is a NUL-terminated std::string.
  std::string_view operator()(std::string_view *rest, const char *limit = nullptr) const {
    using namespace pcre2;
    // the patterns are the reference's, verbatim: they ARE the specification of where a sentence may end
    static const Regex whitespace_re("\\s*", UTF | DOTALL | NEWLINE_ANY);
    static const Regex chunker_re(
        "\\s*"
        "[^.?!։。？！]*?"
        "([\\p{L}\\p{Lo}\\p{N}]*)"
        "([.?!։。？！]++)"
        "("
        "['\")\\]’”\\p{Pf}]*"
        "(?:\\[[\\p{Nd}]+[\\p{Nd},\\s]*[\\p{Nd}]\\])?"
        "['\")\\]’”\\p{Pf}]*"
        ")"
        "(\\s*)"
        "(?="
        "([^\\s\\p{L}\\p{Lo}\\p{N}\\p{M}\\p{S}]*)"
        "\\s*"
        "([\\p{L}\\p{Lo}\\p{M}\\p{N}]*)"
        ")",
        UTF | DOTALL | NEWLINE_ANY);
    static const Regex lowercase("\\p{M}*\\p{Ll}", NO_UTF_CHECK);
    static const Regex uppercase("\\p{M}*[\\p{Lu}\\p{Lt}]", NO_UTF_CHECK);
    static const Regex digit("[\\p{Nd}\\p{Nl}]", NO_UTF_CHECK);
    static const Regex letterother("\\p{M}*[\\p{Lo}]", NO_UTF_CHECK | UTF);
    static const Regex rtrim("(.*[^\\s])\\s*", NO_UTF_CHECK | DOTALL);
    thread_local Match whitespace_m(whitespace_re), chunker_m(chunker_re), lowercase_m(lowercase), uppercase_m(uppercase),
        digit_m(digit), letterother_m(letterother), rtrim_m(rtrim);

    whitespace_re.consume(rest, &whitespace_m, NO_UTF_CHECK);
    const char *snt_start = rest->data();
    const char *snt_end = rest->data() + rest->size();
    const char past = (limit != nullptr && snt_end < limit) ? *snt_end : '\0';
    int success;
    while ((success = chunker_re.consume(rest, &chunker_m, NO_UTF_CHECK)) > 0) {
      const std::string_view whole = chunker_m[0], prefix = chunker_m[1], punct = chunker_m[2], tail = chunker_m[3];
      const std::string_view whitespace_after = chunker_m[4], following = chunker_m[6];
      // a full-width ideographic stop needs no blank after it; anything else does
      if (whitespace_after.empty() && !(punct == "。" || punct == "！" || punct == "？")) continue;
      if (letterother.find(following, &letterother_m, 0, ANCHORED) > 0) {
        // a caseless letter follows: no reason not to break
      } else if (lowercase.find(following, &lowercase_m, 0, ANCHORED) > 0) {
        continue;
      } else if (uppercase.find(following, &uppercase_m, 0, ANCHORED) > 0) {
        if (punct == "." && get_prefix_class(prefix) != 0) continue;  // a protected prefix ("Dr.")
        if (punct.size() == 1 && past == '.') continue;
      } else if (digit.find(following, &digit_m, 0, ANCHORED) > 0) {
        if (punct == "." && get_prefix_class(prefix) == 2) continue;  // a prefix protected in front of numbers ("No.")
      } else {
        // an ellipsis in brackets inside the text: "[...]"
        if (punct == "..." && punct.data() - whole.data() > 1 && tail == "]" && punct.data()[-1] == '[') continue;
      }
      snt_end = whitespace_after.data();
      break;
    }
    std::string_view snt(snt_start, static_cast<size_t>(snt_end - snt_start));
    if (success < 1) {  // the chunker ran out: the remainder, without its trailing whitespace, is the last sentence
      if (rtrim.consume(&snt, &rtrim_m, NO_UTF_CHECK) > 0) snt = rtrim_m[1];
      *rest = std::string_view();
    }
    return snt;
  }

 private:
  // 0: not a prefix, 1: prefix, 2: prefix only in front of numbers (Splitter.cc:112-124)
  int get_prefix_class(std::string_view piece) const {
    static const Regex last_word(".*\\s([^\\s]*)", pcre2::DOTALL);
    thread_local Match m(last_word);
    if (last_word.consume(&piece, &m, pcre2::NO_UTF_CHECK) > 0) piece = m[1];
    auto it = prefix_type_.find(piece);
    return it == prefix_type_.end() ? 0 : it->second;
  }
  void declare_prefix(std::string_view buffer) {  // Splitter.cc:33-47: "<prefix> [#NUMERIC_ONLY#]", '#' starts a comment
    static const Regex pat("([^#\\s]*)\\s*(?:(#\\s*NUMERIC_ONLY\\s*#))?", pcre2::UTF);
    thread_local Match m(pat);
    if (pat.find(buffer, &m) > 0) {
      const std::string_view m1 = m[1];
      if (!m1.empty()) prefix_type_[std::string(m1)] = !m[2].empty() ? 2 : 1;
    }
  }
  std::map<std::string, int, std::less<>> prefix_type_;
};

class SentenceStream {  // Splitter.hh:42-73, Splitter.cc:316-373
 public:
  enum class splitmode { OneSentencePerLine, OneParagraphPerLine, WrappedText };
  SentenceStream(std::string_view text, const Splitter &splitter, splitmode mode, bool verify_utf8 = true)
      : SentenceStream(text.data(), text.size(), splitter, mode, verify_utf8) {}
  SentenceStream(const char *data, size_t size, const Splitter &splitter, splitmode mode, bool verify_utf8 = true)
      : cursor_(data), stop_(data + size), mode_(mode), splitter_(splitter) {
    if (verify_utf8) {  // pre-flight: a text that is not well-formed UTF-8 yields no sentences and an error message
      static const Regex any(".*", pcre2::UTF);
      thread_local Match m(any);
      const int rc = any.find(std::string_view(data, size), &m);
      if (rc < 0) {
        uint8_t buffer[256] = {0};
        pcre2::Api::get().get_error_message(rc, buffer, sizeof(buffer));
        std::ostringstream msg;
        msg << "Invalid UTF at position " << pcre2::Api::get().get_startchar(m.match_data) << ": " << reinterpret_cast<const char *>(buffer);
        error_message_ = msg.str();
        status_ = rc;
      }
    }
    if (mode == splitmode::OneParagraphPerLine) paragraph_ = detail::read_line(&cursor_, stop_);
    if (mode == splitmode::WrappedText) paragraph_ = detail::read_paragraph(&cursor_, stop_);
  }
  int status() const { return status_; }
  const std::string &error_message() const { return error_message_; }
  // In the paragraph modes an EMPTY view separates the sentences of consecutive paragraphs.
  bool operator>>(std::string_view &snt) {
    if (!error_message_.empty()) return false;
    if (paragraph_.empty() && cursor_ == stop_) return false;
    if (mode_ == splitmode::OneSentencePerLine) {
      snt = detail::read_line(&cursor_, stop_);
    } else if (paragraph_.empty()) {
      snt = std::string_view();
      paragraph_ = mode_ == splitmode::OneParagraphPerLine ? detail::read_line(&cursor_, stop_) : detail::read_paragraph(&cursor_, stop_);
    } else {
      snt = splitter_(&paragraph_, stop_);
    }
    return true;
  }

 private:
  const char *cursor_;
  const char *const stop_;
  std::string_view paragraph_;
  splitmode mode_;
  const Splitter &splitter_;
  std::string error_message_;
  int status_ = 0;
};

// ---------------------------------------------------------------- Annotation / AnnotatedText (slimt/Annotation.hh, .cc)
inline int utf8_sequence_length(char c) {  // Annotation.cc:168-186
  if ((c & 0x80) == 0) return 1;
  if ((c & 0xE0) == 0xC0) return 2;
  if ((c & 0xF0) == 0xE0) return 3;
  if ((c & 0xF8) == 0xF0) return 4;
  return 0;
}

// Sentences and their (sub)words as offsets into one text.  token_begin_ holds the start of every token, where the
// whitespace BETWEEN sentences counts as a token too ("gap"); gap_[i] is the index of the gap in front of sentence i,
// and one more gap closes the text.  (Annotation.hh:15-110)
class Annotation {
 public:
  Annotation() : token_begin_{0, 0}, gap_{0} {}
  size_t sentence_count() const { return gap_.size() - 1; }
  size_t word_count(size_t s) const { return gap_[s + 1] - gap_[s] - 1; }
  Range word(size_t s, size_t w) const {
    const size_t t = gap_[s] + 1 + w;
    return Range{token_begin_[t], token_begin_[t + 1]};
  }
  Range sentence(size_t s) const { return Range{token_begin_[gap_[s] + 1], token_begin_[gap_[s + 1]]}; }
  Range gap(size_t g) const { return Range{token_begin_[gap_[g]], token_begin_[gap_[g] + 1]}; }
  void update(const std::vector<size_t> &token_begin) {
    assert(token_begin_.size() == token_begin.size());
    token_begin_ = token_begin;
  }
  const std::vector<size_t> &token_begin() const { return token_begin_; }

 private:
  friend class AnnotatedText;
  std::vector<size_t> token_begin_;
  std::vector<size_t> gap_;
};

class AnnotatedText {
 public:
  std::string text;
  Annotation annotation;

  AnnotatedText() = default;
  explicit AnnotatedText(std::string &&t) : text(std::move(t)) { annotation.token_begin_.back() = text.size(); }

  // Annotation.cc:21-42: `prefix` is the whitespace in front of the sentence, the tokens are contiguous views of some
  // other string whose bytes are appended
  void append_sentence(std::string_view prefix, Views::iterator begin, Views::iterator end) {
    append_ending_whitespace(prefix);
    size_t offset = text.size();
    for (auto token = begin; token != end; ++token) {
      offset += token->size();
      annotation.token_begin_.push_back(offset);
    }
    if (begin != end) text.append(begin->data(), static_cast<size_t>((end - 1)->data() + (end - 1)->size() - begin->data()));
    annotation.gap_.push_back(annotation.token_begin_.size() - 1);
    annotation.token_begin_.push_back(offset);
  }
  void append_ending_whitespace(std::string_view whitespace) {  // Annotation.cc:44-47
    text.append(whitespace.data(), whitespace.size());
    annotation.token_begin_.back() = text.size();
  }
  // Annotation.cc:52-78: the tokens are views INTO text; the bytes since the previous sentence become its gap
  void record_existing_sentence(Views::iterator begin, Views::iterator end, const char *sentence_begin) {
    annotation.token_begin_.pop_back();
    for (auto i = begin; i != end; ++i) annotation.token_begin_.push_back(static_cast<size_t>(i->data() - text.data()));
    annotation.gap_.push_back(annotation.token_begin_.size());
    if (begin != end) {
      annotation.token_begin_.push_back(static_cast<size_t>((end - 1)->data() + (end - 1)->size() - text.data()));
    } else {
      annotation.token_begin_.push_back(static_cast<size_t>(sentence_begin - text.data()));
    }
    annotation.token_begin_.push_back(text.size());
  }
  void update(const std::vector<size_t> &token_begin) { annotation.update(token_begin); }

  // byte offsets <-> code point offsets (Annotation.cc:80-166)
  void to(Encoding encoding) {
    if (encoding == encoding_) return;
    const std::vector<size_t> &from = annotation.token_begin_;
    std::vector<size_t> out;
    out.reserve(from.size());
    size_t byte = 0, point = 0, k = 0;
    const bool to_bytes = encoding == Encoding::Byte;
    auto flush = [&]() {
      while (k < from.size() && from[k] == (to_bytes ? point : byte)) out.push_back(to_bytes ? byte : point), k++;
    };
    flush();
    while (byte < text.size()) {
      const int n = utf8_sequence_length(text[byte]);
      if (to_bytes) {
        point += 1, byte += static_cast<size_t>(n);
        if (n == 0) break;  // (the reference would not advance on a stray continuation byte)
      } else if (n > 0) {
        point += 1, byte += static_cast<size_t>(n);
      } else {
        byte += 1;
      }
      flush();
    }
    annotation.update(out);
    encoding_ = encoding;
  }

  size_t sentence_count() const { return annotation.sentence_count(); }
  size_t word_count(size_t s) const { return annotation.word_count(s); }
  std::string_view word(size_t s, size_t w) const { return as_view(annotation.word(s, w)); }
  std::string_view sentence(size_t s) const { return as_view(annotation.sentence(s)); }
  std::string_view gap(size_t s) const { return as_view(annotation.gap(s)); }
  Range word_as_range(size_t s, size_t w) const { return annotation.word(s, w); }
  Range sentence_as_range(size_t s) const { return annotation.sentence(s); }

 private:
  std::string_view as_view(const Range &r) const { return std::string_view(text.data() + r.begin, r.size()); }
  Encoding encoding_ = Encoding::Byte;
};

// ---------------------------------------------------------------- TextProcessor (slimt/TextProcessor.hh, .cc)
class TextProcessor {
 public:
  // `prefixes`: the contents of an ssplit prefix file, may be empty (Model.cc:58, 69 always pass an empty blob)
  TextProcessor(const std::string &mode, const Vocabulary &vocabulary, std::string_view prefixes = std::string_view())
      : ssplit_mode_(string2splitmode(mode)), vocabulary_(vocabulary) {
    if (!prefixes.empty()) ssplit_.load_from_serialized(prefixes);
  }

  // TextProcessor.cc:96-121: split into sentences, tokenise each, hard-wrap at wrap_length tokens (EOS included)
  std::tuple<AnnotatedText, Segments> process(std::string &&input, size_t wrap_length) const {
    AnnotatedText source(std::move(input));
    Segments segments;
    SentenceStream stream(std::string_view(source.text.data(), source.text.size()), ssplit_, ssplit_mode_);
    std::string_view sentence;
    while (stream >> sentence) {
      auto [words, ranges] = vocabulary_.encode(sentence, /*add_eos=*/false);
      // a sentence may normalise to nothing: it leaves no segment (TextProcessor.cc:113-117)
      if (!words.empty()) wrap(words, ranges, segments, source, wrap_length);
    }
    return {std::move(source), std::move(segments)};
  }

  // TextProcessor.cc:159-199: re-tokenise an already split text (the pivot of a two-model translation); no wrapping
  std::tuple<AnnotatedText, Segments> process(AnnotatedText &source) const {
    Segments segments;
    std::string text = source.text;
    AnnotatedText replacement(std::move(text));
    for (size_t s = 0; s < source.sentence_count(); s++) {
      const Range range = source.sentence_as_range(s);
      const std::string_view sentence(replacement.text.data() + range.begin, range.size());
      auto [words, ranges] = vocabulary_.encode(sentence, /*add_eos=*/false);
      words.push_back(vocabulary_.eos_id());
      const char *end = ranges.empty() ? sentence.data() + sentence.size() : ranges.back().data() + ranges.back().size();
      ranges.emplace_back(end, 0);
      segments.push_back(std::move(words));
      replacement.record_existing_sentence(ranges.begin(), ranges.end(), ranges.begin()->data());
    }
    return {std::move(replacement), std::move(segments)};
  }

 private:
  static SentenceStream::splitmode string2splitmode(const std::string &m) {  // TextProcessor.cc:21-37
    if (m == "sentence") return SentenceStream::splitmode::OneSentencePerLine;
    if (m == "paragraph") return SentenceStream::splitmode::OneParagraphPerLine;
    if (m == "wrapped_text") return SentenceStream::splitmode::WrappedText;
    throw std::runtime_error("Unknown ssplitmode " + m + ", Please choose one of {sentence,paragraph,wrapped_text}");
  }
  // TextProcessor.cc:123-157: pieces of wrap_length - 1 words, each closed by its own EOS whose range is the empty
  // string right behind the piece's last word
  void wrap(const Segment &segment, Views &ranges, Segments &segments, AnnotatedText &source, size_t wrap_length) const {
    const Word eos = vocabulary_.eos_id();
    const size_t step = wrap_length - 1;
    for (size_t offset = 0; offset < segment.size(); offset += step) {
      const size_t diff = std::min(step, segment.size() - offset);
      segments.emplace_back(segment.begin() + offset, segment.begin() + offset + diff);
      segments.back().push_back(eos);
      Views part(ranges.begin() + offset, ranges.begin() + offset + diff);
      part.emplace_back(part.back().data() + part.back().size(), 0);
      source.record_existing_sentence(part.begin(), part.end(), ranges[offset].data());
    }
  }
  SentenceStream::splitmode ssplit_mode_;
  const Vocabulary &vocabulary_;
  Splitter ssplit_;
};

// ---------------------------------------------------------------- Response, Options (slimt/Response.hh, Response.cc)
struct Options {
  bool alignment = false;  // include alignments or not
  bool html = false;       // markup handling is not carried (see the header comment): must be false
  bool scores = false;     // include per-token log-probabilities or not (marian's --word-scores)
  // Draw each word from the model's distribution at `temperature` instead of decoding greedily (marian's
  // --output-sampling; slimt_b200_translate_sampled).  A segment's answer depends on (seed, temperature, segment) alone,
  // not on the request or batch that carried it; sampled segments bypass the translation cache.
  bool sample = false;
  float temperature = 1.0f;  // finite, in [1e-3, 1e3]
  uint64_t seed = 0;
  // With sample: draw each word from the top_k most likely words only (marian's --output-sampling topk;
  // slimt_b200_translate_topk).  0 = from every word; 1 .. 256 otherwise.  top_k > 0 without sample, with
  // beam_size > 1, or out of range is std::invalid_argument.
  int top_k = 0;
  // Beam search with beam_size hypotheses per segment (marian's --beam-size / --normalize; slimt_b200_translate_beam):
  // the best hypothesis by total / len^length_penalty is returned, its scores and alignments with it.  beam_size = 1 is
  // the greedy call; beam_size > 1 together with sample is std::invalid_argument.  Beam segments bypass the translation
  // cache.
  int beam_size = 1;  // 1 .. 8
  float length_penalty = 0.0f;  // finite, >= 0
};

struct Response {
  AnnotatedText source;
  AnnotatedText target;
  // alignments[sentence][t][s] = p(source token s | target token t)
  std::vector<Alignment> alignments;
  // scores[sentence][t] = log p(target token t | source, tokens before t) under greedy decoding, EOS included: one per
  // token of the sentence's translation, empty unless Options::scores.  After a pivot: the second leg's scores.
  std::vector<std::vector<float>> scores;
  size_t size() const { return source.sentence_count(); }
  void to(Encoding encoding) { source.to(encoding), target.to(encoding); }
};
using Responses = std::vector<Response>;

// Response.cc:16-124: the two models tokenise the pivot text differently; probability mass moves from the second
// model's pivot tokens to the first's in proportion to the characters they share
inline Alignment transfer_through_characters(const std::vector<Range> &source_side_pivots,
                                             const std::vector<Range> &target_side_pivots, const Alignment &pivot_given_targets) {
  Alignment remapped(pivot_given_targets.size(), Distribution(source_side_pivots.size(), 0.0F));
  size_t sq = 0, qt = 0;
  while (sq < source_side_pivots.size() && qt < target_side_pivots.size()) {
    const Range &s = source_side_pivots[sq], &q = target_side_pivots[qt];
    if (s.begin == q.begin && s.end == q.end) {
      for (size_t t = 0; t < pivot_given_targets.size(); t++) remapped[t][sq] += pivot_given_targets[t][qt];
      sq++, qt++;
      continue;
    }
    const size_t left = std::max(q.begin, s.begin), right = std::min(q.end, s.end);
    // The reference asserts left < right here (Response.cc:49) and, built without assertions, goes on with a wrapped
    // difference.  The case is real -- a piece that decodes to nothing (a lone U+2581 at the start of the pivot
    // sentence) facing a non-empty token of the other tokenisation -- so instead: no shared characters, no mass moved;
    // a zero-width token of the second tokenisation hands its whole mass to the token it falls into.
    const size_t shared = right > left ? right - left : 0, spread = q.size();
    for (size_t t = 0; t < pivot_given_targets.size(); t++)
      remapped[t][sq] += spread == 0 ? pivot_given_targets[t][qt]
                                     : static_cast<float>(shared) * pivot_given_targets[t][qt] / static_cast<float>(spread);
    if (s.end == q.end) {
      sq++, qt++;
    } else if (s.end > q.end) {
      qt++;
    } else {
      sq++;
    }
  }
  // what is left on the second model's side is its EOS: spread evenly
  for (; qt < target_side_pivots.size(); qt++) {
    for (size_t t = 0; t < pivot_given_targets.size(); t++) {
      const float gift = pivot_given_targets[t][qt] / static_cast<float>(source_side_pivots.size());
      for (size_t k = 0; k < source_side_pivots.size(); k++) remapped[t][k] += gift;
    }
  }
  return remapped;
}

inline std::vector<Alignment> remap_alignments(const Response &first, const Response &second) {  // Response.cc:126-163
  std::vector<Alignment> alignments;
  auto word_ranges = [](const AnnotatedText &text, size_t s) {
    std::vector<Range> out;
    for (size_t i = 0; i < text.word_count(s); i++) out.push_back(text.word_as_range(s, i));
    return out;
  };
  for (size_t s = 0; s < first.source.sentence_count(); s++) {
    const Alignment &source_given_pivots = first.alignments[s];
    const std::vector<Range> source_side = word_ranges(first.target, s), target_side = word_ranges(second.source, s);
    const Alignment remapped = transfer_through_characters(source_side, target_side, second.alignments[s]);
    const size_t S = first.source.word_count(s), T = second.target.word_count(s);
    Alignment out(T, Distribution(S, 0.0F));
    for (size_t t = 0; t < T; t++)
      for (size_t q = 0; q < source_side.size(); q++)
        for (size_t k = 0; k < S; k++) out[t][k] += source_given_pivots[q][k] * remapped[t][q];
    alignments.push_back(std::move(out));
  }
  return alignments;
}

// The scores of a pivot are the second leg's: they score the tokens the combined Response returns (the first leg's
// scores are of the pivot text, which the caller does not see).
inline Response combine(Response &&first, Response &&second) {  // Response.cc:165-175
  Response combined;
  if (!first.alignments.empty()) combined.alignments = remap_alignments(first, second);
  combined.scores = std::move(second.scores);
  combined.source = std::move(first.source);
  combined.target = std::move(second.target);
  return combined;
}

// Request::complete (Request.cc:133-169): the target text of a request from its sentences' histories -- every decoded
// sentence behind the whitespace that stood in front of its source sentence
inline Response make_response(AnnotatedText &&source, const Histories &histories, const Vocabulary &vocabulary) {
  if (source.sentence_count() != histories.size()) throw std::runtime_error("Mismatch in source and translated sentences");
  Response response;
  response.source = std::move(source);
  response.target.text.reserve(response.source.text.size());
  for (size_t s = 0; s < histories.size(); s++) {
    std::string decoded;
    Views views = vocabulary.decode(histories[s]->target, decoded, /*ignore_eos=*/false);
    response.target.append_sentence(response.source.gap(s), views.begin(), views.end());
    if (s + 1 == histories.size()) response.target.append_ending_whitespace(response.source.gap(s + 1));
    response.alignments.push_back(histories[s]->alignment);
    response.scores.push_back(histories[s]->scores);
  }
  return response;
}

}  // namespace slimt
