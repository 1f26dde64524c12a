// slimt_b200.hh -- host-side C++ mirror of slimt's API surface for the hot path, over the C ABI in
// slimt_b200.h.  Header only; link with libslimt_b200.so.  Same names, argument meaning and error
// behaviour as the reference for the slice that sits on the path:
//
//   slimt::Tensor / Shape / Type            slimt/Tensor.hh:16-154   (row-major dense, owning or view)
//   slimt::qmm::affine / affine_with_select / dot / prepare_weight_*   slimt/QMM.hh:48-63
//   slimt::Input                            slimt/Input.hh:10-37     (padded batch of word ids)
//   slimt::Model::forward -> Histories      slimt/Model.hh:31-83, Model.cc:187-204
//   slimt::Config, slimt::Blocking, slimt::Async   slimt/Frontend.hh:21-78
//   slimt::Options, slimt::Response, combine()     slimt/Response.hh:20-58, Response.cc:126-175
//
// The text front half above Model::forward (Vocabulary, TextProcessor, sentence splitter, AnnotatedText, Response) is
// slimt_b200_text.hh (host only; included below).  The services therefore come at two levels: on text, with the
// reference's own signatures (Blocking::translate(model, std::vector<std::string>, options) -> std::vector<Response>,
// Async::translate(model, std::string, options) -> Handle), and on word ids (slimt::Sentences in, WordsResponse out),
// which is what the reference hands to Model::forward (Frontend.cc:30-60) and what the benchmarks feed.  HTML markup
// handling (HTML.cc) is not carried.  Not meant to be included together with the reference's own headers: inside the
// slimt tree the same C ABI is bound by the provider file shown in INTEGRATION.md.
//
// Error convention: the reference asserts / aborts on shape violations (qmm/Gemmology.inl.cc:51,141,
// Macros.hh:30-42) and throws std::runtime_error from its loaders (Io.cc:294-309); here every failure of the
// C ABI is a std::runtime_error carrying slimt_b200_last_error().  There is no CPU fallback.
#pragma once
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <functional>
#include <future>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include "slimt_b200.h"
#include "slimt_b200_text.hh"  // Types.hh's aliases (Word, Words, Sentences, Ptr, View, Hypothesis, ...) and the text front half

namespace slimt {

namespace detail {
inline void check(int rc, const char *what) {
  if (rc != 0) throw std::runtime_error(std::string(what) + ": " + slimt_b200_last_error());
}
// one context per device, created on first use and kept for the life of the process.  Every C-ABI call that uses a
// context's stream or workspace takes the context's own lock, so models, services and qmm:: calls that share a device
// serialise on it instead of racing (the reference's callers are re-entrant: Frontend.cc:213-225).
inline slimt_b200_ctx *context(int device = 0) {
  static std::mutex mu;
  static std::vector<slimt_b200_ctx *> ctxs;
  std::lock_guard<std::mutex> lock(mu);
  if (static_cast<size_t>(device) >= ctxs.size()) ctxs.resize(device + 1, nullptr);
  if (ctxs[device] == nullptr) check(slimt_b200_ctx_create(device, &ctxs[device]), "slimt_b200_ctx_create");
  return ctxs[device];
}
}  // namespace detail

// ---------------------------------------------------------------- Tensor (slimt/Tensor.hh)
enum class Type { i8, ig8, i32, u32, f32 };
inline size_t size_in_bytes(Type t) { return (t == Type::i8 || t == Type::ig8) ? 1 : 4; }

class Shape {
 public:
  Shape() = default;
  Shape(std::initializer_list<uint64_t> dims) : dims_(dims) {}
  explicit Shape(std::vector<uint64_t> dims) : dims_(std::move(dims)) {}
  uint64_t dim(int64_t i) const { return dims_[i < 0 ? dims_.size() + i : i]; }  // negative = from the end
  size_t size() const { return dims_.size(); }
  size_t elements() const {
    size_t n = 1;
    for (uint64_t d : dims_) n *= d;
    return n;
  }
  const std::vector<uint64_t> &dims() const { return dims_; }
  void set_dim(int64_t i, uint64_t v) { dims_[i < 0 ? dims_.size() + i : i] = v; }

 private:
  std::vector<uint64_t> dims_;
};

class Tensor {
 public:
  Tensor() = default;
  Tensor(Type type, Shape shape, std::string name = "") : type_(type), shape_(std::move(shape)), name_(std::move(name)) {
    bytes_ = shape_.elements() * size_in_bytes(type_);
    // 64-byte aligned like slimt::Aligned (Aligned.cc:45-52); ig8 weights carry their f32 multiplier after the bytes
    size_t alloc = ((bytes_ + (type_ == Type::ig8 ? 4 : 0) + 63) / 64) * 64;
    own_.reset(static_cast<char *>(std::aligned_alloc(64, alloc ? alloc : 64)), std::free);
    data_ = own_.get();
  }
  // non-owning view (Tensor::load, Tensor.cc:87-93)
  void load(View view, Type type, Shape shape, std::string name) {
    own_.reset();
    data_ = view.data, bytes_ = view.size, type_ = type, shape_ = std::move(shape), name_ = std::move(name);
  }
  template <class T>
  T *data() { return static_cast<T *>(data_); }
  template <class T>
  const T *data() const { return static_cast<const T *>(data_); }
  uint64_t dim(int64_t i) const { return shape_.dim(i); }
  const Shape &shape() const { return shape_; }
  Type type() const { return type_; }
  size_t size() const { return shape_.elements(); }
  const std::string &name() const { return name_; }
  Tensor clone() const {
    Tensor t(type_, shape_, name_);
    std::memcpy(t.data_, data_, bytes_ + (type_ == Type::ig8 ? 4 : 0));
    return t;
  }

 private:
  Type type_ = Type::f32;
  Shape shape_;
  std::string name_;
  std::shared_ptr<char> own_;
  void *data_ = nullptr;
  size_t bytes_ = 0;
};

// ---------------------------------------------------------------- qmm:: (slimt/QMM.hh:48-63)
namespace qmm {
namespace detail {
inline Tensor run(const Tensor &x, const Tensor &W, const float *bias, float a_quant, float b_quant,
                  const std::vector<uint32_t> *indices, const std::string &name) {
  // x [..., K] f32; W prepared int8 of logical shape {K, N} (Io.cc:227-228) stored as B^T [N][K]
  const size_t K = x.dim(-1), M = x.size() / K;
  const size_t N = W.dim(-1);
  if (W.dim(-2) != K) throw std::runtime_error("qmm: inner dimensions of x and W differ");
  Shape out = x.shape();
  out.set_dim(-1, indices ? indices->size() : N);
  Tensor y(Type::f32, out, name);
  ::slimt::detail::check(
      slimt_b200_qmm_affine(::slimt::detail::context(), x.data<float>(), M, K, W.data<int8_t>(), N, bias, a_quant, b_quant,
                            indices ? indices->data() : nullptr, indices ? indices->size() : 0, y.data<float>()),
      "slimt_b200_qmm_affine");
  return y;
}
}  // namespace detail

inline Tensor affine(const Tensor &x, const Tensor &W, const Tensor &b, float a_quant, float b_quant,
                     const std::string &name = "") {
  return detail::run(x, W, b.data<float>(), a_quant, b_quant, nullptr, name);
}
inline Tensor affine_with_select(const Tensor &x, const Tensor &W, const Tensor &b, float a_quant, float b_quant,
                                 const std::vector<uint32_t> &indices, const std::string &name = "") {
  return detail::run(x, W, b.data<float>(), a_quant, b_quant, &indices, name);
}
inline Tensor dot(const Tensor &x, const Tensor &W, float a_quant, float b_quant, const std::string &name = "") {
  return detail::run(x, W, nullptr, a_quant, b_quant, nullptr, name);
}
inline void prepare_weight_transposed(const float *weights, int8_t *prepared, float quantization_multiplier, size_t cols,
                                      size_t rows) {
  slimt_b200_qmm_prepare_weight_transposed(weights, prepared, quantization_multiplier, cols, rows);
}
inline void prepare_weight_quantized_transposed(const int8_t *input, int8_t *output, size_t rows, size_t cols) {
  slimt_b200_qmm_prepare_weight_quantized_transposed(input, output, rows, cols);
}
}  // namespace qmm

// ---------------------------------------------------------------- Input (slimt/Input.hh)
class Input {
 public:
  Input(size_t batch_size, size_t sequence_length, uint32_t pad_id, float limit_factor)
      : batch_(Type::u32, Shape({batch_size, sequence_length}), "batch"), pad_id_(pad_id), limit_factor_(limit_factor) {
    std::fill(batch_.data<uint32_t>(), batch_.data<uint32_t>() + batch_.size(), pad_id);
  }
  void add(const std::vector<uint32_t> &words) {
    const size_t T = batch_.dim(-1);
    if (index_ >= batch_.dim(-2) || words.size() > T) throw std::runtime_error("Input::add: batch or sequence overflow");
    std::memcpy(batch_.data<uint32_t>() + index_ * T, words.data(), 4 * words.size());
    words_.insert(words_.end(), words.begin(), words.end());
    lengths_.push_back(words.size());
    ++index_;
  }
  void finalize() {}  // the additive mask (Input.cc:49-63) is implied by lengths() on the device
  const Tensor &indices() const { return batch_; }
  const std::vector<uint32_t> &words() const { return words_; }
  const std::vector<size_t> &lengths() const { return lengths_; }
  size_t index() const { return index_; }
  float limit_factor() const { return limit_factor_; }

 private:
  std::vector<uint32_t> words_;
  std::vector<size_t> lengths_;
  Tensor batch_;
  size_t index_ = 0;
  uint32_t pad_id_ = 0;
  float limit_factor_;
};

// ---------------------------------------------------------------- io::MmapFile (slimt/Io.hh, Io.cc:291-340)
namespace io {
// Read-only private mapping of a file; move-only; throws std::runtime_error exactly where the reference does.
class MmapFile {
 public:
  MmapFile() = default;
  explicit MmapFile(const std::string &filepath) {
    fd_ = open(filepath.c_str(), O_RDONLY);
    if (fd_ == -1) throw std::runtime_error("Failed to open file: " + filepath);
    struct stat st;
    if (fstat(fd_, &st) == -1) {
      close(fd_);
      throw std::runtime_error("Failed to get file size: " + filepath);
    }
    size_ = static_cast<size_t>(st.st_size);
    data_ = mmap(nullptr, size_, PROT_READ, MAP_PRIVATE, fd_, 0);
    if (data_ == MAP_FAILED) {
      close(fd_);
      throw std::runtime_error("Failed to mmap file: " + filepath);
    }
  }
  ~MmapFile() { release(); }
  MmapFile(const MmapFile &) = delete;
  MmapFile &operator=(const MmapFile &) = delete;
  MmapFile(MmapFile &&from) noexcept : fd_(from.fd_), data_(from.data_), size_(from.size_) { from.reset(); }
  MmapFile &operator=(MmapFile &&from) noexcept {
    if (this != &from) {
      release();
      fd_ = from.fd_, data_ = from.data_, size_ = from.size_;
      from.reset();
    }
    return *this;
  }
  void *data() const { return data_; }
  size_t size() const { return size_; }

 private:
  void reset() { fd_ = -1, data_ = nullptr, size_ = 0; }
  void release() {
    if (data_ != nullptr && data_ != MAP_FAILED) munmap(data_, size_);
    if (fd_ != -1) close(fd_);
    reset();
  }
  int fd_ = -1;
  void *data_ = nullptr;
  size_t size_ = 0;
};
}  // namespace io

// ---------------------------------------------------------------- Shortlist / ShortlistGenerator (slimt/Shortlist.hh)
class Shortlist {  // Shortlist.hh:14-33: the sorted candidate word ids of one batch
 public:
  explicit Shortlist(Words words) : words_(std::move(words)) {}
  const std::vector<Word> &words() const { return words_; }
  Word reverse_map(int idx) const { return words_[idx]; }
  int try_forward_map(Word w) const {
    auto first = std::lower_bound(words_.begin(), words_.end(), w);
    return (first != words_.end() && *first == w) ? static_cast<int>(std::distance(words_.begin(), first)) : -1;
  }

 private:
  std::vector<Word> words_;
};

// Shortlist.hh:35-76 over the host-only C-ABI calls (no GPU needed): the binary lex.s2t.bin image stays the caller's
// (a View, as in the reference); `vocabulary_size` is the target vocabulary's size, which bounds the candidate ids.
// check = true runs the reference's header / size / checksum / content_check (Shortlist.cc:16-37, 68-98) at
// construction and throws where the reference aborts.
class ShortlistGenerator {
 public:
  ShortlistGenerator(View view, size_t vocabulary_size, bool check = false) : view_(view), vocab_(vocabulary_size) {
    if (check) detail::check(slimt_b200_shortlist_check(view_.data, view_.size, vocab_), "ShortlistGenerator: check failed");
  }
  ShortlistGenerator(View view, const Vocabulary & /*source*/, const Vocabulary &target, size_t /*source_index*/ = 0,
                     size_t /*target_index*/ = 1, bool /*shared*/ = false, bool check = false)
      : ShortlistGenerator(view, target.size(), check) {}
  // Shortlist.cc:115-175: first `frequent` ids + the targets of every distinct source word, padded to a multiple of 8
  Shortlist generate(const Words &words) const {
    Words out(vocab_ + 8);
    size_t n = 0;
    detail::check(slimt_b200_shortlist_generate(view_.data, view_.size, words.data(), words.size(), vocab_, out.data(), out.size(), &n),
                  "slimt_b200_shortlist_generate");
    out.resize(n);
    return Shortlist(std::move(out));
  }

 private:
  View view_;
  size_t vocab_;
};

// Batcher::generate (Batcher.cc:95-120) as a plan over sentence lengths: batches in ascending length, each as many
// sentences as fit `(n + 1) * longest <= max_words`.  The services run the same planner inside the C-ABI call.
struct BatchPlan {
  std::vector<size_t> ids;  // sentence indices of the batch
  size_t width = 0;         // padded length
};
inline std::vector<BatchPlan> plan_batches(const Sentences &sentences, size_t max_words) {
  std::vector<uint64_t> lengths(sentences.size()), ids(sentences.size()), offsets(sentences.size() + 1), widths(sentences.size() + 1);
  for (size_t i = 0; i < sentences.size(); i++) lengths[i] = sentences[i].size();
  size_t n = 0;
  detail::check(slimt_b200_batcher_plan(lengths.data(), lengths.size(), max_words, ids.data(), offsets.data(), widths.data(), &n),
                "slimt_b200_batcher_plan");
  std::vector<BatchPlan> plan(n);
  for (size_t b = 0; b < n; b++) {
    plan[b].ids.assign(ids.begin() + offsets[b], ids.begin() + offsets[b + 1]);
    plan[b].width = widths[b];
  }
  return plan;
}

// ---------------------------------------------------------------- Model (slimt/Model.hh)
template <class Field>
struct Package {
  Field model;       // marian binary v1 (model.intgemm.alphas.bin)
  Field vocabulary;  // sentencepiece model (vocab.spm); may be empty when only word ids are served
  Field shortlist;   // lex.s2t.bin or empty
  Field ssplit;      // sentence-splitter prefix file or empty (the reference maps it but never reads it, Model.cc:58, 69)
};

class Model {
 public:
  struct Config {  // Model.hh:33-51
    size_t encoder_layers = 6;
    size_t decoder_layers = 2;
    size_t feed_forward_depth = 2;
    size_t num_heads = 8;
    std::string split_mode = "sentence";
    // Vocabulary::eos_id() / pad_id() (Vocabulary.hh:22-23).  With a vocabulary in the package they are taken from it,
    // as in the reference; a model that serves word ids only (no vocabulary) uses the values given here.
    uint32_t eos_id = 0;
    uint32_t pad_id = 0;
  };

  // Model.hh:53: the files are mapped (io::MmapFile) and stay mapped for the model's lifetime, as in the reference
  // (Model.cc:52-66); an empty path leaves the field empty.  Throws std::runtime_error for a missing file.
  // `devices`: one weight replica per listed GPU.  Model::forward uses the first; the services deal batches to all of
  // them (the reference's Async workers share one Model on the CPU, Frontend.cc:213-225).
  Model(const Config &config, const Package<std::string> &package, std::vector<int> devices = {0})
      : Model(config, map_files(package), std::move(devices), 0) {}

  Model(const Config &config, const Package<View> &package, std::vector<int> devices = {0})
      : id_(next_id()), config_(config), devices_(std::move(devices)) {
    create(package);
  }
  ~Model() {
    for (slimt_b200_model *m : replicas_) slimt_b200_model_destroy(m);
  }
  Model(const Model &) = delete;
  Model &operator=(const Model &) = delete;

 private:
  using Mmap = Package<io::MmapFile>;
  static Mmap map_files(const Package<std::string> &p) {
    Mmap m;
    if (!p.model.empty()) m.model = io::MmapFile(p.model);
    if (!p.vocabulary.empty()) m.vocabulary = io::MmapFile(p.vocabulary);
    if (!p.shortlist.empty()) m.shortlist = io::MmapFile(p.shortlist);
    if (!p.ssplit.empty()) m.ssplit = io::MmapFile(p.ssplit);
    return m;
  }
  static size_t next_id() {  // Model.cc:28, 53: every model of the process gets the next id (the cache key's seed)
    static std::atomic<size_t> model_id{0};
    return model_id++;
  }
  Model(const Config &config, Mmap &&files, std::vector<int> devices, int /*tag*/)
      : id_(next_id()), config_(config), devices_(std::move(devices)), mmap_(std::move(files)) {
    create(Package<View>{{mmap_.model.data(), mmap_.model.size()},
                         {mmap_.vocabulary.data(), mmap_.vocabulary.size()},
                         {mmap_.shortlist.data(), mmap_.shortlist.size()},
                         {mmap_.ssplit.data(), mmap_.ssplit.size()}});
  }
  void create(const Package<View> &package) {
    if (devices_.empty()) throw std::runtime_error("Model: at least one device is required");
    // Model.cc:56-58: the vocabulary and, on it, the text processor (always without a prefix file, as in the reference)
    if (package.vocabulary.data != nullptr && package.vocabulary.size > 0) {
      vocabulary_ = std::make_unique<Vocabulary>(package.vocabulary);
      processor_ = std::make_unique<TextProcessor>(config_.split_mode, *vocabulary_);
      config_.eos_id = vocabulary_->eos_id(), config_.pad_id = vocabulary_->pad_id();
    }
    slimt_b200_model_config c{static_cast<int32_t>(config_.encoder_layers), static_cast<int32_t>(config_.decoder_layers),
                              static_cast<int32_t>(config_.feed_forward_depth), static_cast<int32_t>(config_.num_heads),
                              config_.eos_id, config_.pad_id};
    for (int device : devices_) {
      slimt_b200_model *m = nullptr;
      detail::check(slimt_b200_model_create(detail::context(device), package.model.data, package.model.size, &c, &m),
                    "slimt_b200_model_create");
      replicas_.push_back(m);
      // as in the reference, only the caller's wrap_length bounds a segment: admit every length the model can encode
      int32_t current = 0, supported = 0;
      slimt_b200_model_max_length(m, &current, &supported);
      detail::check(slimt_b200_model_set_max_length(m, supported), "slimt_b200_model_set_max_length");
    }
    int32_t e = 0, f = 0, v = 0;
    slimt_b200_model_dims(replicas_[0], &e, &f, &v);
    vocab_ = static_cast<size_t>(v);
    if (vocabulary_ && vocabulary_->size() > vocab_) {
      for (slimt_b200_model *m : replicas_) slimt_b200_model_destroy(m);  // (the destructor does not run for a throwing constructor)
      replicas_.clear();
      throw std::runtime_error("Model: the vocabulary has " + std::to_string(vocabulary_->size()) + " pieces, the model's embedding " +
                               std::to_string(vocab_) + " rows");
    }
    if (package.shortlist.data != nullptr && package.shortlist.size > 0) {
      shortlist_.assign(static_cast<const char *>(package.shortlist.data),
                        static_cast<const char *>(package.shortlist.data) + package.shortlist.size);
    }
  }

 public:
  // Model::forward (Model.cc:187-204): embedding -> encoder -> greedy decode with the per-batch shortlist.
  // Re-entrant like the reference's: concurrent calls serialise on the device context's own lock (one stream and one
  // workspace per context), not on this object.
  Histories forward(const Input &input) const {
    const size_t B = input.index(), T = input.indices().dim(-1);
    std::vector<uint32_t> lengths(input.lengths().begin(), input.lengths().end());
    std::vector<uint32_t> shortlist;
    if (auto generator = shortlist_generator()) shortlist = generator->generate(input.words()).words();  // Model.cc:116-120
    // the first decoder step is unconditional (Model.cc:145-157): at least one step
    const size_t max_steps = std::max<size_t>(1, static_cast<size_t>(input.limit_factor() * static_cast<float>(T)));
    std::vector<uint32_t> steps(max_steps * std::max<size_t>(1, B));
    std::vector<float> align(steps.size() * T);
    slimt_b200_forward_io io;
    std::memset(&io, 0, sizeof(io));
    io.tokens = input.indices().data<uint32_t>(), io.lengths = lengths.data(), io.batch = B, io.seq = T;
    io.limit_factor = input.limit_factor();
    io.shortlist = shortlist.empty() ? nullptr : shortlist.data(), io.n_shortlist = shortlist.size();
    io.step_tokens = steps.data(), io.alignment = align.data();
    detail::check(slimt_b200_model_forward(replicas_[0], &io), "slimt_b200_model_forward");
    Histories histories;
    for (size_t b = 0; b < B; b++) {  // record() + update_alignment (Model.cc:84-137)
      auto h = std::make_shared<Hypothesis>();
      for (size_t s = 0; s < io.steps; s++) {
        const uint32_t w = steps[s * B + b];
        h->target.push_back(w);
        const float *row = align.data() + (s * B + b) * T;
        h->alignment.emplace_back(row, row + lengths[b]);
        if (w == config_.eos_id) break;
      }
      histories.push_back(std::move(h));
    }
    return histories;
  }
  const Config &config() const { return config_; }
  // Model.hh:59-60; a model created without a vocabulary serves word ids only
  bool has_vocabulary() const { return vocabulary_ != nullptr; }
  const Vocabulary &vocabulary() const {
    if (!vocabulary_) throw std::runtime_error("Model: created without a vocabulary (Package::vocabulary is empty)");
    return *vocabulary_;
  }
  const TextProcessor &processor() const {
    if (!processor_) throw std::runtime_error("Model: created without a vocabulary (Package::vocabulary is empty)");
    return *processor_;
  }
  size_t id() const { return id_; }  // Model.hh:62
  // Model.hh:63-65: absent when the package has no shortlist.  The candidate ids are bounded by the vocabulary's size
  // when there is one (Shortlist.cc:116-117), else by the embedding's rows.
  std::optional<ShortlistGenerator> shortlist_generator() const {
    if (shortlist_.empty()) return std::nullopt;
    return ShortlistGenerator(View{const_cast<char *>(shortlist_.data()), shortlist_.size()}, vocabulary_ ? vocabulary_->size() : vocab_);
  }
  size_t vocabulary_size() const { return vocab_; }
  const std::vector<int> &devices() const { return devices_; }
  slimt_b200_model *handle() const { return replicas_[0]; }
  const std::vector<slimt_b200_model *> &replicas() const { return replicas_; }
  const std::vector<char> &shortlist_image() const { return shortlist_; }

 private:
  size_t id_;
  Config config_;
  std::vector<int> devices_;
  Mmap mmap_;  // only used by the path constructor
  std::vector<slimt_b200_model *> replicas_;
  size_t vocab_ = 0;
  std::vector<char> shortlist_;
  std::unique_ptr<Vocabulary> vocabulary_;
  std::unique_ptr<TextProcessor> processor_;
};

// Model.hh:85-89, Model.cc:206-245
namespace preset {
inline Model::Config tiny() { return Model::Config{6, 2, 2, 8, "sentence"}; }
inline Model::Config base() { return Model::Config{6, 2, 2, 8, "sentence"}; }
inline Model::Config nano() { return Model::Config{4, 2, 2, 8, "sentence"}; }
}  // namespace preset

// ---------------------------------------------------------------- translation cache (slimt/Cache.hh, Request.cc:20-26)
// AtomicCache (Cache.hh:11-58): a direct-mapped table -- no probing, a newer key simply replaces the record in its
// slot -- with one mutex per bucket of slots.  The key of a translation is cache_key(model id, segment words), the
// value its History; two segments whose keys collide are indistinguishable, as in the reference.
template <class Key, class Value, class Hash = std::hash<Key>, class Equals = std::equal_to<Key>>
class AtomicCache {
 public:
  explicit AtomicCache(size_t size, size_t buckets) : records_(size), locks_(buckets) {}
  std::pair<bool, Value> find(const Key &key) const {
    const size_t index = hash_(key) % records_.size();
    std::lock_guard<std::mutex> guard(locks_[index % locks_.size()]);
    const Record &candidate = records_[index];
    if (equals_(key, candidate.first)) return {true, candidate.second};
    return {false, Value()};
  }
  void store(const Key &key, Value value) {
    const size_t index = hash_(key) % records_.size();
    std::lock_guard<std::mutex> guard(locks_[index % locks_.size()]);
    records_[index] = Record(key, std::move(value));
  }

 private:
  using Record = std::pair<Key, Value>;
  std::vector<Record> records_;
  mutable std::vector<std::mutex> locks_;
  Hash hash_;
  Equals equals_;
};
using TranslationCache = AtomicCache<size_t, History>;  // Types.hh:62

// Utils.hh:47-57 (boost-style combinator over std::hash) and Request.cc:20-26
template <class T, class HashType = std::size_t>
inline void hash_combine(HashType &seed, const T &v) {
  seed ^= (static_cast<HashType>(std::hash<T>()(v)) + 0x9e3779b9 + (seed << 6) + (seed >> 2));
}
inline size_t cache_key(size_t model_id, const Words &words) {
  size_t seed = model_id;
  for (size_t word : words) hash_combine<size_t>(seed, word);
  return seed;
}
inline Ptr<TranslationCache> make_cache(size_t cache_size) {  // Frontend.cc:78-85
  constexpr size_t kCacheBucketSize = 16;
  return cache_size > 0 ? std::make_shared<TranslationCache>(cache_size, kCacheBucketSize) : nullptr;
}

// TextProcessor::wrap (TextProcessor.cc:123-157) on word ids: a sentence of more than wrap_length tokens is cut into
// segments of wrap_length - 1 words, each closed with its own EOS (the decoder needs the marker); shorter sentences
// pass through untouched.  The sentence's own closing EOS, when present, is not counted as a word.
inline void wrap(const Words &sentence, size_t wrap_length, Word eos_id, Sentences &segments) {
  if (sentence.empty()) return;  // TextProcessor.cc:113-117: nothing to translate, no segment
  if (wrap_length < 2 || sentence.size() <= wrap_length) {
    segments.push_back(sentence);
    return;
  }
  const size_t words = sentence.back() == eos_id ? sentence.size() - 1 : sentence.size();
  const size_t step = wrap_length - 1;
  for (size_t offset = 0; offset < words; offset += step) {
    const size_t diff = std::min(step, words - offset);
    segments.emplace_back(sentence.begin() + offset, sentence.begin() + offset + diff);
    segments.back().push_back(eos_id);
  }
}

// ---------------------------------------------------------------- services (slimt/Frontend.hh, slimt/Response.hh)
struct Config {
  size_t max_words = 1024;
  size_t cache_size = 1024;
  size_t workers = 1;
  float tgt_length_limit_factor = 1.5;
  size_t wrap_length = 128;
};

// Response (Response.hh:20-43) at the WORD-ID level of this path: the reference's AnnotatedText source / target are the
// sentences' word ids here; alignments[i][t][s] = p(source token s | target token t) of sentence i (head 0 of the last
// decoder layer's cross-attention, Model.cc:84-108), empty unless Options::alignment.  The text-level slimt::Response
// (AnnotatedText source / target) and Options are in slimt_b200_text.hh.
struct WordsResponse {
  Sentences source;  // one entry per SEGMENT (a sentence longer than Config::wrap_length is several, TextProcessor.cc:123)
  Sentences target;
  std::vector<Alignment> alignments;
  // segments [sentence_begin[i], sentence_begin[i + 1]) came from input sentence i (the reference keeps this relation
  // in the byte ranges of its AnnotatedText); the identity while nothing was wrapped
  std::vector<size_t> sentence_begin;
  size_t size() const { return source.size(); }
};

// remap_alignments + combine (Response.cc:126-175) for pivoting on word ids: the pivot sentence is handed to the second
// model as produced, so the character-overlap transfer between two tokenisations of the pivot text is the identity and
// what remains is the marginalisation p(s | t) = sum_q p(s | q) p(q | t).
inline WordsResponse combine(WordsResponse &&first, WordsResponse &&second) {
  WordsResponse out;
  // (a pivot sentence the second service had to wrap again has no one-to-one segment any more: no combined alignment)
  if (!first.alignments.empty() && second.alignments.size() == first.alignments.size()) {
    for (size_t i = 0; i < first.source.size(); i++) {
      const Alignment &s_given_q = first.alignments[i];
      const Alignment &q_given_t = second.alignments[i];
      const size_t S = first.source[i].size(), Q = s_given_q.size();
      Alignment a(q_given_t.size(), Distribution(S, 0.0F));
      for (size_t t = 0; t < q_given_t.size(); t++)
        for (size_t q = 0; q < Q && q < q_given_t[t].size(); q++)
          for (size_t src = 0; src < S; src++) a[t][src] += s_given_q[q][src] * q_given_t[t][q];
      out.alignments.push_back(std::move(a));
    }
  }
  out.source = std::move(first.source);
  out.target = std::move(second.target);
  out.sentence_begin = std::move(first.sentence_begin);
  return out;
}

// Blocking (Frontend.hh:41-57, Frontend.cc:88-205).  Both levels end in serve(): the segments of the whole call go
// through the cache and then through ONE C-ABI call -- one Batcher, per-batch shortlist, Model::forward per batch,
// batches dealt to every replica of the model (exhaust(), Frontend.cc:42-60).
class Blocking {
 public:
  explicit Blocking(const Config &config) : config_(config), cache_(make_cache(config.cache_size)) {}
  // a service that shares another one's cache (Async's workers, Frontend.cc:207-210)
  Blocking(const Config &config, Ptr<TranslationCache> cache) : config_(config), cache_(std::move(cache)) {}

  // ---- text level: the reference's own signatures (Frontend.cc:91-145)
  std::vector<Response> translate(const Ptr<Model> &model, std::vector<std::string> sources, const Options &options = Options()) {
    if (options.html) throw std::runtime_error("Options::html: markup handling (HTML.cc) is not part of this path");
    const TextProcessor &processor = model->processor();
    // TextProcessor::process per source; independent, so spread over Config::workers host threads
    std::vector<AnnotatedText> annotated(sources.size());
    std::vector<Segments> segments(sources.size());
    parallel_for(sources.size(), [&](size_t i) {
      std::tie(annotated[i], segments[i]) = processor.process(std::move(sources[i]), config_.wrap_length);
    });
    return respond(model, std::move(annotated), std::move(segments), options);
  }

  // Frontend.cc:147-205: source -> pivot with `first`; the pivot TEXT is re-tokenised sentence by sentence with the
  // second model's processor (no re-splitting, no wrapping) -> target; alignments are carried across the two
  // tokenisations of the pivot text (remap_alignments)
  std::vector<Response> pivot(const Ptr<Model> &first, const Ptr<Model> &second, std::vector<std::string> sources,
                              const Options &options = Options()) {
    std::vector<Response> source_to_pivots = translate(first, std::move(sources), options);
    const TextProcessor &processor = second->processor();
    std::vector<AnnotatedText> annotated(source_to_pivots.size());
    std::vector<Segments> segments(source_to_pivots.size());
    parallel_for(source_to_pivots.size(), [&](size_t i) {
      std::tie(annotated[i], segments[i]) = processor.process(source_to_pivots[i].target);
    });
    std::vector<Response> pivot_to_targets = respond(second, std::move(annotated), std::move(segments), options);
    std::vector<Response> responses;
    for (size_t i = 0; i < source_to_pivots.size(); i++)
      responses.push_back(combine(std::move(source_to_pivots[i]), std::move(pivot_to_targets[i])));
    return responses;
  }

  // ---- word-id level
  WordsResponse translate(const Ptr<Model> &model, const Sentences &sources, const Options &options = Options()) {
    WordsResponse response;
    // segments (TextProcessor::process + wrap, on word ids)
    response.sentence_begin.push_back(0);
    for (const Words &s : sources) {
      wrap(s, config_.wrap_length, model->config().eos_id, response.source);
      response.sentence_begin.push_back(response.source.size());
    }
    const Histories histories = serve(model, response.source, options);
    response.target.reserve(histories.size());
    for (const History &h : histories) response.target.push_back(h->target);
    if (options.alignment)
      for (const History &h : histories) response.alignments.push_back(h->alignment);
    return response;
  }
  // Blocking::pivot on word ids: the two models must share the pivot-language vocabulary; the pivot sentences are
  // passed on as produced, EOS included, like the reference's segments (TextProcessor.cc:132-143).
  WordsResponse pivot(const Ptr<Model> &first, const Ptr<Model> &second, const Sentences &sources, const Options &options = Options()) {
    WordsResponse source_to_pivot = translate(first, sources, options);
    WordsResponse pivot_to_target = translate(second, source_to_pivot.target, options);
    return combine(std::move(source_to_pivot), std::move(pivot_to_target));
  }
  size_t cache_hits() const { return cache_hits_; }

 private:
  template <class F>
  void parallel_for(size_t n, F &&body) const {
    const size_t threads = std::min(n, std::max<size_t>(1, config_.workers));
    if (threads <= 1) {
      for (size_t i = 0; i < n; i++) body(i);
      return;
    }
    std::atomic<size_t> next{0};
    std::exception_ptr error;
    std::mutex error_mu;
    std::vector<std::thread> pool;
    for (size_t t = 0; t < threads; t++)
      pool.emplace_back([&]() {
        try {
          for (size_t i = next++; i < n; i = next++) body(i);
        } catch (...) {
          std::lock_guard<std::mutex> lock(error_mu);
          if (!error) error = std::current_exception();
        }
      });
    for (std::thread &t : pool) t.join();
    if (error) std::rethrow_exception(error);
  }

  // all segments of all requests of a call in one pool -> serve() -> one Response per request (Request::complete)
  std::vector<Response> respond(const Ptr<Model> &model, std::vector<AnnotatedText> &&annotated, std::vector<Segments> &&segments,
                                const Options &options) {
    Sentences pool;
    for (const Segments &s : segments) pool.insert(pool.end(), s.begin(), s.end());
    // the decoded text needs every history's alignment only when asked for; the words always
    const Histories histories = serve(model, pool, options);
    std::vector<Response> responses(annotated.size());
    std::vector<size_t> first(annotated.size() + 1, 0);
    for (size_t i = 0; i < annotated.size(); i++) first[i + 1] = first[i] + segments[i].size();
    // detokenisation and Response building per request: independent, on the same host threads as the tokenisation
    parallel_for(annotated.size(), [&](size_t i) {
      Histories mine(histories.begin() + first[i], histories.begin() + first[i + 1]);
      responses[i] = make_response(std::move(annotated[i]), mine, model->vocabulary());
      if (!options.alignment) responses[i].alignments.clear();
    });
    return responses;
  }

  // cache prefill (Request.cc:58-78): a segment this model has translated before is not batched again.  A record
  // stored by a request that did not ask for alignments cannot answer one that does.  The rest: run().
  Histories serve(const Ptr<Model> &model, const Sentences &segments, const Options &options) {
    Histories histories(segments.size());
    std::vector<size_t> todo;
    for (size_t i = 0; i < segments.size(); i++) {
      if (cache_) {
        auto [found, history] = cache_->find(cache_key(model->id(), segments[i]));
        if (found && history && (!options.alignment || history->alignment.size() == history->target.size())) {
          histories[i] = history;
          cache_hits_++;
          continue;
        }
      }
      todo.push_back(i);
    }
    if (!todo.empty()) run(model, segments, todo, options, histories);
    for (size_t i : todo)
      if (cache_) cache_->store(cache_key(model->id(), segments[i]), histories[i]);  // Request.cc:120-125
    return histories;
  }

  // Frontend.cc:91-145 + exhaust() :42-60 for the segments listed in `todo`: one Batcher, per-batch shortlist,
  // Model::forward per batch -- dealt to every replica of the model -- all inside one C-ABI call.
  void run(const Ptr<Model> &model, const Sentences &segments, const std::vector<size_t> &todo, const Options &options,
           Histories &histories) {
    std::vector<uint32_t> tokens;
    std::vector<uint64_t> offsets(1, 0);
    size_t longest = 0;
    for (size_t i : todo) {
      const Words &s = segments[i];
      tokens.insert(tokens.end(), s.begin(), s.end());
      offsets.push_back(tokens.size());
      longest = std::max(longest, s.size());
    }
    const size_t per = std::max<size_t>(1, static_cast<size_t>(config_.tgt_length_limit_factor * static_cast<float>(longest)));
    std::vector<uint32_t> out(std::max<size_t>(1, per * todo.size()));
    std::vector<uint64_t> out_offsets(todo.size() + 1, 0);
    std::vector<float> align;
    std::vector<uint64_t> align_offsets(todo.size() + 1, 0);
    slimt_b200_translate_io io;
    std::memset(&io, 0, sizeof(io));
    io.tokens = tokens.data(), io.offsets = offsets.data(), io.n_sentences = todo.size();
    io.max_words = config_.max_words, io.limit_factor = config_.tgt_length_limit_factor;
    const std::vector<char> &sl = model->shortlist_image();
    io.shortlist_bin = sl.empty() ? nullptr : sl.data(), io.shortlist_bytes = sl.size();
    io.out_tokens = out.data(), io.out_capacity = out.size(), io.out_offsets = out_offsets.data();
    if (options.alignment) {
      align.resize(std::max<size_t>(1, per * tokens.size()));
      io.out_alignments = align.data(), io.align_capacity = align.size(), io.out_align_offsets = align_offsets.data();
    }
    const std::vector<slimt_b200_model *> &replicas = model->replicas();
    detail::check(slimt_b200_translate_multi(replicas.data(), replicas.size(), &io), "slimt_b200_translate_multi");
    for (size_t k = 0; k < todo.size(); k++) {
      auto h = std::make_shared<Hypothesis>();
      h->target.assign(out.begin() + out_offsets[k], out.begin() + out_offsets[k + 1]);
      if (options.alignment) {
        const size_t S = segments[todo[k]].size();
        const float *p = align.data() + align_offsets[k];
        for (size_t t = 0; t < h->target.size(); t++) h->alignment.emplace_back(p + t * S, p + (t + 1) * S);
      }
      histories[todo[k]] = std::move(h);
    }
  }

  Config config_;
  Ptr<TranslationCache> cache_;
  size_t cache_hits_ = 0;
};

// Types.hh:24-27
struct Fraction {
  size_t p = 0;
  size_t q = 0;
};

// Handle (Response.hh:60-91): what Async returns for a text request -- the future of its Response.  info() has the
// reference's shape; a request is served by one C-ABI call here, so only `parts` moves (0 / n until the answer is there,
// then n / n; a pivot has two parts) and the word / segment counters stay 0 / 0: they are in the Response.
class Handle {
 public:
  Handle(std::future<Response> &&future, size_t parts, size_t words, size_t segments)
      : future_(std::move(future)), parts_(parts), words_(words), segments_(segments), start_(std::chrono::steady_clock::now()) {}
  explicit Handle(std::future<Response> &&future) : Handle(std::move(future), 1, 0, 0) {}
  struct Info {
    double wps;
    Fraction parts;
    Fraction words;
    Fraction segments;
  };
  Info info() {
    const bool done = future_.valid() && future_.wait_for(std::chrono::seconds(0)) == std::future_status::ready;
    const double elapsed = std::chrono::duration<double>(std::chrono::steady_clock::now() - start_).count();
    return Info{done && elapsed > 0 ? static_cast<double>(words_) / elapsed : 0.0, Fraction{done ? parts_ : 0, parts_},
                Fraction{done ? words_ : 0, words_}, Fraction{done ? segments_ : 0, segments_}};
  }
  std::future<Response> &future() { return future_; }

 private:
  std::future<Response> future_;
  size_t parts_, words_, segments_;
  std::chrono::steady_clock::time_point start_;
};

// Async (Frontend.hh:59-78, Frontend.cc:207-323): `workers` threads take requests from one queue and answer through
// futures.  A request is served by Blocking's path, i.e. its batches are dealt to every GPU replica of its model;
// requests in flight at the same time share the replicas (each device context serialises the batches it is given).
class Async {
 public:
  explicit Async(const Config &config) : config_(config), cache_(make_cache(config.cache_size)) {
    for (size_t i = 0; i < std::max<size_t>(1, config_.workers); i++) workers_.emplace_back([this]() { work(); });
  }
  ~Async() {
    {
      std::lock_guard<std::mutex> lock(mu_);
      shutdown_ = true;
    }
    cv_.notify_all();
    for (std::thread &t : workers_) t.join();
  }
  // ---- text level (Frontend.cc:229-314)
  Handle translate(const Ptr<Model> &model, std::string source, const Options &options = Options()) {
    Job job{model, nullptr, {}, options, {}, true, std::move(source), {}};
    Handle handle(job.text_promise.get_future(), /*parts=*/1, 0, 0);
    enqueue(std::move(job));
    return handle;
  }
  Handle pivot(const Ptr<Model> &first, const Ptr<Model> &second, std::string source, const Options &options = Options()) {
    Job job{first, second, {}, options, {}, true, std::move(source), {}};
    Handle handle(job.text_promise.get_future(), /*parts=*/2, 0, 0);
    enqueue(std::move(job));
    return handle;
  }
  // ---- word-id level
  std::future<WordsResponse> translate(const Ptr<Model> &model, Sentences sources, const Options &options = Options()) {
    Job job{model, nullptr, std::move(sources), options, {}, false, {}, {}};
    std::future<WordsResponse> f = job.promise.get_future();
    enqueue(std::move(job));
    return f;
  }
  // Async::pivot (Frontend.cc:259-314): the second translation is chained behind the first inside the worker
  std::future<WordsResponse> pivot(const Ptr<Model> &first, const Ptr<Model> &second, Sentences sources,
                                   const Options &options = Options()) {
    Job job{first, second, std::move(sources), options, {}, false, {}, {}};
    std::future<WordsResponse> f = job.promise.get_future();
    enqueue(std::move(job));
    return f;
  }

 private:
  struct Job {
    Ptr<Model> first, second;
    Sentences sources;
    Options options;
    std::promise<WordsResponse> promise;
    bool is_text = false;
    std::string text;
    std::promise<Response> text_promise;
  };
  void enqueue(Job job) {
    {
      std::lock_guard<std::mutex> lock(mu_);
      queue_.push_back(std::move(job));
    }
    cv_.notify_one();
  }
  // AggregateBatcher (Batcher.hh:128-200): requests that wait at the same time are batched TOGETHER.  A worker that
  // wakes up takes the oldest request and every queued request of the same kind (same model, same level, same
  // options, not a pivot) and serves them in one service call, so a burst of single-sentence requests fills GPU-sized
  // batches instead of running one tiny batch each.  As in the reference, what a shortlisted model answers may then
  // depend on who shared the batch (the candidate set is the union over the batch, Model.cc:116-120).
  static bool poolable(const Job &a, const Job &b) {
    return !a.second && !b.second && a.first == b.first && a.is_text == b.is_text && a.options.alignment == b.options.alignment &&
           a.options.html == b.options.html;
  }
  void work() {
    Config one = config_;
    one.workers = 1;  // (a request's own tokenisation stays on the worker that serves it)
    Blocking service(one, cache_);  // one cache for the whole service (Frontend.cc:207-210)
    for (;;) {
      std::vector<Job> jobs;
      {
        std::unique_lock<std::mutex> lock(mu_);
        cv_.wait(lock, [this]() { return shutdown_ || !queue_.empty(); });
        if (queue_.empty()) return;
        jobs.push_back(std::move(queue_.front()));
        queue_.pop_front();
        for (auto it = queue_.begin(); it != queue_.end();) {
          if (poolable(jobs.front(), *it)) {
            jobs.push_back(std::move(*it));
            it = queue_.erase(it);
          } else {
            ++it;
          }
        }
      }
      service_calls_++;
      requests_served_ += jobs.size();
      try {
        Job &head = jobs.front();
        if (head.is_text) {
          if (head.second) {
            std::vector<Response> r = service.pivot(head.first, head.second, std::vector<std::string>(1, std::move(head.text)), head.options);
            head.text_promise.set_value(std::move(r[0]));
          } else {
            std::vector<std::string> sources;
            for (Job &j : jobs) sources.push_back(std::move(j.text));
            std::vector<Response> r = service.translate(head.first, std::move(sources), head.options);
            for (size_t k = 0; k < jobs.size(); k++) jobs[k].text_promise.set_value(std::move(r[k]));
          }
        } else if (head.second) {
          head.promise.set_value(service.pivot(head.first, head.second, head.sources, head.options));
        } else if (jobs.size() == 1) {
          head.promise.set_value(service.translate(head.first, head.sources, head.options));
        } else {
          Sentences pooled;
          std::vector<size_t> first_sentence(1, 0);
          for (const Job &j : jobs) {
            pooled.insert(pooled.end(), j.sources.begin(), j.sources.end());
            first_sentence.push_back(pooled.size());
          }
          WordsResponse all = service.translate(head.first, pooled, head.options);
          for (size_t k = 0; k < jobs.size(); k++) {  // every request gets the segments of its own sentences back
            WordsResponse mine;
            const size_t s0 = first_sentence[k], s1 = first_sentence[k + 1];
            const size_t g0 = all.sentence_begin[s0], g1 = all.sentence_begin[s1];
            mine.source.assign(all.source.begin() + g0, all.source.begin() + g1);
            mine.target.assign(all.target.begin() + g0, all.target.begin() + g1);
            if (!all.alignments.empty()) mine.alignments.assign(all.alignments.begin() + g0, all.alignments.begin() + g1);
            for (size_t s = s0; s <= s1; s++) mine.sentence_begin.push_back(all.sentence_begin[s] - g0);
            jobs[k].promise.set_value(std::move(mine));
          }
        }
      } catch (...) {
        // a promise that was already answered keeps its answer; the others carry the error
        for (Job &j : jobs) {
          try {
            if (j.is_text) {
              j.text_promise.set_exception(std::current_exception());
            } else {
              j.promise.set_exception(std::current_exception());
            }
          } catch (const std::future_error &) {
          }
        }
      }
    }
  }

 public:
  // monitoring: service calls made so far and requests they answered (requests / calls > 1: requests were pooled)
  size_t service_calls() const { return service_calls_; }
  size_t requests_served() const { return requests_served_; }

 private:
  std::atomic<size_t> service_calls_{0}, requests_served_{0};
  Config config_;
  Ptr<TranslationCache> cache_;
  std::vector<std::thread> workers_;
  std::deque<Job> queue_;
  std::mutex mu_;
  std::condition_variable cv_;
  bool shutdown_ = false;
};

}  // namespace slimt
