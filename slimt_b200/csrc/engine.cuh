// Host-side engine: device context, model upload, and the orchestration of
// Model::forward (reference slimt/Model.cc:111-204) as a sequence of the
// kernels in gemm_i8.cu / kernels.cu on one CUDA stream.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "fused_rows.cuh"
#include "gemm_i8.cuh"
#include "kernels.cuh"
#include "out_argmax.cuh"

namespace sb {

void set_error(const std::string& msg);
const char* last_error();

#define SB_CUDA(expr)                                                                      \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess) {                                                               \
      sb::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
      (void)cudaGetLastError(); /* reported: do not leave it for an unrelated later check */ \
      return 1;                                                                            \
    }                                                                                      \
  } while (0)

struct Context {
  // One stream, one workspace arena, one staging block and one set of polling slots per context: every entry point
  // that touches them (qmm::*, Model::forward, the translate service) holds this lock for the duration of the call,
  // so replicas or services that share a device context serialise instead of corrupting each other's workspace.
  // Recursive because the service path calls model_forward with the lock held.
  std::recursive_mutex mu;
  // Arithmetic mode of every kernel launched through this context.  false (default): bit-exact restatement of the
  // reference's float arithmetic (the verifier).  true (SLIMT_B200_MATH=fast or slimt_b200_ctx_set_math): tolerance
  // mode -- FMA-contracted dequantisation, tree-reduced LayerNorm statistics, ex2/rcp-based softmax and sigmoid,
  // integer argmax proxy -- held to north_star's bars (logits rtol 1e-3, >= 99 % greedy tokens) instead of bit equality.
  bool fast = false;
  int device = 0;
  int num_sms = 148;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // cuTensorMapEncodeTiled, fetched through the runtime so libcuda is not a link-time dependency
  CUresult (*encode_tiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                           const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                           CUtensorMapL2promotion, CUtensorMapFloatOOBfill) = nullptr;
  // workspace arena (grown on demand, reused across calls; Workspace cuts it into buffers)
  char* arena = nullptr;
  size_t arena_bytes = 0;
  char* flush_buf = nullptr;
  size_t flush_bytes = 0;
  // pinned host staging of the service path (padded batch in, step tokens out): grown on demand, reused across calls;
  // Workspace cuts it into buffers too
  char* staging = nullptr;
  size_t staging_bytes = 0;
  char* staging_reserve(size_t bytes);
  uint64_t launches = 0;
  uint64_t h2d_bytes = 0, d2h_bytes = 0;
  // early-exit polling of the decode loop: pinned slots + events, so the host never drains the stream
  int* done_slots = nullptr;  // pinned host [kPollSlots]
  cudaEvent_t done_events[8] = {};
  // optional per-kernel device timing (CUDA events around every launch on `stream`)
  struct ProfRec {
    const char* tag;
    cudaEvent_t e0, e1;
    double ops, bytes;
  };
  bool profiling = false;
  std::vector<ProfRec> prof;
  std::vector<cudaEvent_t> event_pool;
  cudaEvent_t pooled_event();

  int init(int dev);
  void destroy();
  int reserve(size_t bytes);
  // int8 row-major [rows][cols] -> 2D tensor map, box = {128 bytes, box_rows}, 128B swizzle
  int make_map(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
  // f32 row-major [rows][cols] -> 2D tensor map, box = {32 floats (128 bytes), box_rows}, 128B swizzle
  int make_map_f32(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows);
};

// Margin behind the last buffer of the arena: not every kernel has been shown to keep its loads inside its buffer (the
// output GEMMs index per-column arrays by 256-column tile), so the arena keeps ending with 16 KB that no buffer owns.
constexpr size_t kTailPad = 64 * 256;

// The buffers of one call, each listed once: add() records where a buffer's pointer goes and how many elements it
// holds; carve() reserves the sum in the context's device arena, or with `staging` in its pinned host staging block, and
// hands out the pointers in list order, each buffer starting on a 256-byte boundary.
struct Workspace {
  size_t bytes = 0;
  std::vector<std::pair<void**, size_t>> bufs;
  template <class T>
  void add(T*& slot, size_t count) {
    bufs.emplace_back(reinterpret_cast<void**>(&slot), (count * sizeof(T) + 255) & ~size_t(255));
    bytes += bufs.back().second;
  }
  int carve(Context& c, bool staging = false) const {
    char* p = staging ? c.staging_reserve(bytes) : c.reserve(bytes + kTailPad) ? nullptr : c.arena;
    if (p == nullptr) return 1;
    for (const auto& b : bufs) *b.first = p, p += b.second;
    return 0;
  }
};

// Counts a kernel launch and, in profiling mode, brackets it with events.  `ops` = algorithmic int8
// operations (2*MAC), `bytes` = algorithmic HBM bytes of the launch (DESIGN.md lists both per kernel).
struct LaunchScope {
  Context& c;
  bool on;
  LaunchScope(Context& ctx, const char* tag, double ops, double bytes) : c(ctx), on(ctx.profiling) {
    c.launches++;
    if (on) {
      Context::ProfRec r{tag, c.pooled_event(), c.pooled_event(), ops, bytes};
      cudaEventRecord(r.e0, c.stream);
      c.prof.push_back(r);
    }
  }
  ~LaunchScope() {
    if (on) cudaEventRecord(c.prof.back().e1, c.stream);
  }
};

// One int8 weight matrix on the device, with everything the epilogue needs precomputed at load
// (the reference recomputes PrepareBias on every call: qmm/Intgemm.inl.cc:112-128).
struct DevWeight {
  int K = 0, N = 0;
  float aq = 0, bq = 0, um = 0;
  int8_t* w = nullptr;      // [N][K]
  CUtensorMap map128;       // TMA view of w with box {128 B, 128 rows}: the A operand of the row-tile kernels
  CUtensorMap map32;        // box {128 B, 32 rows}: one head's features, the B operand of the fused encoder attention
  float* pb = nullptr;      // [N]
};

struct DevLN {
  float* scale = nullptr;
  float* bias = nullptr;
};

struct AttnW {
  DevWeight q, k, v, o;
  DevLN ln;
};
struct FfnW {
  DevWeight w1, w2;
  DevLN ln;
};
struct EncLayerW {
  AttnW self;
  FfnW ffn;
};
struct DecLayerW {
  DevWeight rnn_w, rnn_wf;
  DevLN rnn_ln;
  AttnW ctx;
  FfnW ffn;
};

struct Model {
  Context* ctx = nullptr;
  int E = 0, F = 0, V = 0, H = 8, dh = 32;
  std::vector<EncLayerW> enc;
  std::vector<DecLayerW> dec;
  int8_t* emb_q = nullptr;  // [V][E] stored embedding (lookup: float(q) * (1/qm), Io.cc:275-283)
  float emb_qm = 0, inv_qm = 0, sqrt_e = 0;
  DevWeight out;            // Wemb_intgemm8 (re-quantised embedding) + decoder_ff_logit_out_b + none_QuantMultA
  OutColumns vocab;         // out's columns as the fused argmax reads them, with the encoding chosen at load
  float* pos = nullptr;     // sinusoidal table [max_pos][E]
  int max_pos = 0;
  uint32_t eos_id = 0, pad_id = 0;  // Vocabulary::eos_id() / pad_id() (Vocabulary.hh:22-23); both 0 for browsermt vocabularies
  std::vector<void*> owned;
  // extra lanes (stream + workspace + staging) on this model's device, created on demand by the service path
  std::vector<std::unique_ptr<Context>> lanes;
  std::mutex lanes_mu;
  Context* lane(size_t i);  // lane 0 is the model's own context
  // Longest sentence a batch may hold: starts at 256 and may be raised up to max_pos (slimt_b200_model_set_max_length).
  int len_bound = 256;
  int max_len() const { return len_bound < max_pos ? len_bound : max_pos; }

  int load(Context* c, const void* bin, size_t bytes, int enc_layers, int dec_layers, int heads);
  void destroy();
};

struct ForwardArgs {
  const uint32_t* tokens = nullptr;
  const uint32_t* lengths = nullptr;
  size_t B = 0, T = 0;
  float limit_factor = 1.5f;
  const uint32_t* shortlist = nullptr;
  size_t n_shortlist = 0;
  // Alternative to `shortlist` (host-buffer mode only): called once, after the encoder has been enqueued,
  // so that ShortlistGenerator::generate runs on the host while the GPU works.  Returns nonzero on failure.
  int (*shortlist_cb)(void* user, const uint32_t** words, size_t* n) = nullptr;
  void* shortlist_user = nullptr;
  const uint32_t* forced = nullptr;
  bool device_io = false;
  uint32_t* step_tokens = nullptr;
  // Host-buffer mode, alternative to step_tokens: the step matrix transposed on the device to one row per sentence,
  // [B][row_stride] (row_stride >= limit_factor * T), plus each sentence's recorded length (Model.cc:127-137) -- what
  // the service path's record() needs, contiguous per sentence.
  uint32_t* sentence_tokens = nullptr;
  size_t row_stride = 0;
  uint32_t* target_lengths = nullptr;
  size_t steps = 0;
  uint64_t target_tokens = 0;
  float* encoder_out = nullptr;
  float* logits = nullptr;
  float* alignment = nullptr;
  // [max_steps][B] log-probability of each step's chosen (or forced) word over the step's output columns; a device
  // pointer with device_io (score_partial.cuh)
  float* scores = nullptr;
  // Sampling (include/slimt_b200.h, DESIGN §4.4b): each step's word drawn from softmax(fl32(y * inv_t)) with the
  // uniform number of (seed, keys[b], step) instead of the greedy choice.  keys: [B], a device pointer with device_io;
  // null = the row index.  The caller has checked the temperature and that forced is null.
  bool sample = false;
  float inv_t = 1.0f;
  uint64_t seed = 0;
  const uint64_t* keys = nullptr;
  // Top-k sampling (DESIGN §4.4e), with sample set: each step's word drawn from the first top_k (1 .. 256) columns by
  // (logit descending, column ascending) of the logits GEMM's output; 0 = from every column, as above.
  int top_k = 0;
  // Scoring pass (model_score_on, DESIGN §4.4c): the given targets [B][target_T] (host, padded), scored at every
  // position into scores [B][target_T]; alignment, when set, receives [B][target_T][T].
  const uint32_t* targets = nullptr;
  size_t target_T = 0;
  // Beam search (model_beam_on, DESIGN §4.4d): `beam` hypotheses per sentence in decoder rows b * beam + k.  Host
  // buffers: beam_steps [max_steps][B * beam] receives each step's surviving hypotheses, beam_finished [B][beam] every
  // sentence's finished ones; alignment, when set, receives [max_steps][B * beam][T].  steps = the steps executed.
  int beam = 0;
  BeamRec* beam_steps = nullptr;
  BeamFin* beam_finished = nullptr;
};

int model_forward(Model& m, ForwardArgs& a);
// The same pass with stream, workspace and staging taken from `lane` instead of the model's own context: weights are
// read-only, so several lanes on the model's device can run batches of one model concurrently (translate.cu).
int model_forward_on(Model& m, Context& lane, ForwardArgs& a);
// Teacher-forced scoring of a.targets in one time-parallel pass (bit-exact arithmetic whatever lane.fast says): the
// scores and alignments model_forward would give with forced = the targets, at every target position.
int model_score_on(Model& m, Context& lane, ForwardArgs& a);
// Beam search over a.beam slots per sentence (bit-exact arithmetic whatever lane.fast says): the records from which the
// host rebuilds and ranks each sentence's hypotheses.
int model_beam_on(Model& m, Context& lane, ForwardArgs& a);

// Decoder steps Model::decode may run for a batch of width T: the first step is unconditional (Model.cc:145-157), the
// loop that follows runs while i < size_t(limit_factor * T) (Model.cc:160-161).
inline int forward_max_steps(float limit_factor, size_t T) {
  const size_t n = static_cast<size_t>(limit_factor * static_cast<float>(T));
  return static_cast<int>(n < 1 ? 1 : n);
}

// qmm::affine family on host buffers (operator-level drop-in + parity taps)
int qmm_affine_host(Context& c, const float* x, size_t M, size_t K, const int8_t* W, size_t N, const float* bias,
                    float aq, float bq, const uint32_t* indices, size_t n_idx, float* y, int8_t* qa_out,
                    int32_t* acc_out);

// Host-side exact helpers shared by loader and operator API
void host_prepare_bias(const int8_t* Bt, const float* bias, float aq, float bq, size_t K, size_t N, float* pb);
void host_quantize(const float* x, int8_t* q, float mult, size_t n);

}  // namespace sb
