// See engine.cuh.
#include "engine.cuh"

#include "score_partial.cuh"

#include <math.h>
#include <string.h>

#include <algorithm>

namespace sb {

namespace {
thread_local std::string g_error;
}
void set_error(const std::string& msg) { g_error = msg; }
const char* last_error() { return g_error.c_str(); }

// ------------------------------------------------------------------ host exact helpers
// clamp(rne(x*mult), -127, 127) with x86 cvtps2dq overflow semantics (see exact_math.cuh quantize1).
void host_quantize(const float* x, int8_t* q, float mult, size_t n) {
  for (size_t i = 0; i < n; i++) {
    float t = x[i] * mult;
    int v;
    if (!(t == t) || t >= 2147483648.0f || t < -2147483648.0f) {
      v = -127;
    } else {
      v = static_cast<int>(lrintf(t));
      v = std::max(-127, std::min(127, v));
    }
    q[i] = static_cast<int8_t>(v);
  }
}

// Int8Shift::PrepareBias with UnquantizeAndAddBiasAndWrite (qmm/Intgemm.inl.cc:112-128):
// pb[n] = float(colsum[n]) * ((-1*((127/aq)*(127/bq)))/127) + bias[n].
void host_prepare_bias(const int8_t* Bt, const float* bias, float aq, float bq, size_t K, size_t N, float* pb) {
  const float a_alpha = 127.0f / aq;
  const float b_alpha = 127.0f / bq;
  const float m = (-1.0f * (a_alpha * b_alpha)) / 127.0f;
  for (size_t n = 0; n < N; n++) {
    int32_t cs = 0;
    const int8_t* row = Bt + n * K;
    for (size_t k = 0; k < K; k++) cs += row[k];
    volatile float prod = static_cast<float>(cs) * m;  // keep mul and add separate (no contraction)
    pb[n] = prod + (bias ? bias[n] : 0.0f);
  }
}

// ------------------------------------------------------------------ context
int Context::init(int dev) {
  device = dev;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    set_error(std::string("no CUDA device available (") + cudaGetErrorString(e) +
              "); slimt_b200 has no CPU fallback");
    return 1;
  }
  SB_CUDA(cudaSetDevice(dev));
  cudaDeviceProp prop;
  SB_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) {
    set_error("slimt_b200 requires an sm_100a (B200) device, found sm_" + std::to_string(prop.major) +
              std::to_string(prop.minor));
    return 1;
  }
  num_sms = prop.multiProcessorCount;
  SB_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  SB_CUDA(cudaEventCreate(&ev0));
  SB_CUDA(cudaEventCreate(&ev1));
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  SB_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (fn == nullptr || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return 1;
  }
  encode_tiled = reinterpret_cast<decltype(encode_tiled)>(fn);
  if (const char* e = getenv("SLIMT_B200_MATH")) fast = strcmp(e, "fast") == 0;
  SB_CUDA(cudaMallocHost(&done_slots, 8 * sizeof(int)));
  for (auto& e : done_events) SB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
  return 0;
}

void Context::destroy() {
  cudaSetDevice(device);
  if (arena) cudaFree(arena);
  if (flush_buf) cudaFree(flush_buf);
  if (done_slots) cudaFreeHost(done_slots);
  if (staging) cudaFreeHost(staging);
  for (auto& e : done_events)
    if (e) cudaEventDestroy(e);
  if (ev0) cudaEventDestroy(ev0);
  if (ev1) cudaEventDestroy(ev1);
  if (stream) cudaStreamDestroy(stream);
}

char* Context::staging_reserve(size_t bytes) {
  if (bytes > staging_bytes) {
    if (staging) cudaFreeHost(staging);
    staging = nullptr, staging_bytes = 0;
    const size_t want = bytes + bytes / 4;
    if (cudaHostAlloc(reinterpret_cast<void**>(&staging), want, cudaHostAllocDefault) != cudaSuccess) {
      set_error("pinned staging allocation failed");
      return nullptr;
    }
    staging_bytes = want;
  }
  return staging;
}

cudaEvent_t Context::pooled_event() {
  cudaEvent_t e;
  if (!event_pool.empty()) {
    e = event_pool.back();
    event_pool.pop_back();
  } else {
    cudaEventCreate(&e);
  }
  return e;
}

int Context::reserve(size_t bytes) {
  if (bytes <= arena_bytes) return 0;
  SB_CUDA(cudaStreamSynchronize(stream));
  if (arena) SB_CUDA(cudaFree(arena));
  arena = nullptr;
  arena_bytes = 0;
  size_t want = bytes + (bytes >> 3);
  if (cudaMalloc(&arena, want) != cudaSuccess) {
    (void)cudaGetLastError();
    arena = nullptr;
    set_error("workspace of " + std::to_string(want) + " bytes could not be allocated on the device (a smaller batch, or "
              "no alignment output, needs less)");
    return 1;
  }
  arena_bytes = want;
  return 0;
}

int Context::make_map(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(kBK), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult " + std::to_string(static_cast<int>(r)) + " (rows=" +
              std::to_string(rows) + ", cols=" + std::to_string(cols) + ")");
    return 1;
  }
  return 0;
}

int Context::make_map_f32(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 4};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = encode_tiled(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (f32) failed with CUresult " + std::to_string(static_cast<int>(r)));
    return 1;
  }
  return 0;
}

// ------------------------------------------------------------------ model loading
namespace {

struct Item {
  std::string name;
  uint64_t type = 0;
  std::vector<int> shape;
  const char* data = nullptr;
  uint64_t bytes = 0;
  size_t elements() const {
    size_t n = 1;
    for (int d : shape) n *= static_cast<size_t>(d);
    return n;
  }
};

constexpr uint64_t kTypeF32 = 0x0404, kTypeIG8 = 0x4101;

// marian binary v1 (slimt/Io.cc:114-153, Io.hh:19-29)
int parse_items(const void* bin, size_t bytes, std::map<std::string, Item>& out) {
  const char* p = static_cast<const char*>(bin);
  const char* end = p + bytes;
  auto rd64 = [&p]() {
    uint64_t v;
    memcpy(&v, p, 8);
    p += 8;
    return v;
  };
  if (bytes < 16) {
    set_error("model image too small");
    return 1;
  }
  uint64_t version = rd64();
  if (version != 1) {
    set_error("Binary file versions do not match: " + std::to_string(version) + " (file) != 1 (expected)");
    return 1;
  }
  uint64_t n = rd64();
  struct Hdr {
    uint64_t name_len, type, shape_len, data_len;
  };
  // every count below comes from the file: check it against what is left of the image before using it
  auto left = [&p, end]() { return static_cast<uint64_t>(end - p); };
  if (n > left() / sizeof(Hdr)) {
    set_error("model image truncated: header table of " + std::to_string(n) + " items does not fit");
    return 1;
  }
  std::vector<Hdr> hdrs(n);
  for (auto& h : hdrs) {
    h.name_len = rd64(), h.type = rd64(), h.shape_len = rd64(), h.data_len = rd64();
  }
  std::vector<Item> items(n);
  for (uint64_t i = 0; i < n; i++) {
    if (hdrs[i].name_len == 0 || hdrs[i].name_len > left()) {
      set_error("model image truncated in the name table (item " + std::to_string(i) + ")");
      return 1;
    }
    items[i].name = std::string(p, hdrs[i].name_len - 1);
    items[i].type = hdrs[i].type;
    p += hdrs[i].name_len;
  }
  for (uint64_t i = 0; i < n; i++) {
    if (hdrs[i].shape_len > 8 || 4 * hdrs[i].shape_len > left()) {
      set_error("model image truncated or malformed in the shape table (item " + items[i].name + ")");
      return 1;
    }
    items[i].shape.resize(hdrs[i].shape_len);
    memcpy(items[i].shape.data(), p, 4 * hdrs[i].shape_len);
    for (int d : items[i].shape)
      if (d < 0) {
        set_error("negative dimension in model item " + items[i].name);
        return 1;
      }
    p += 4 * hdrs[i].shape_len;
  }
  if (left() < 8) {
    set_error("model image truncated before the data section");
    return 1;
  }
  uint64_t pad = rd64();
  if (pad > left()) {
    set_error("model image truncated in the alignment padding");
    return 1;
  }
  p += pad;
  for (uint64_t i = 0; i < n; i++) {
    if (hdrs[i].data_len > left()) {
      set_error("model image truncated at item " + items[i].name);
      return 1;
    }
    items[i].data = p;
    items[i].bytes = hdrs[i].data_len;
    p += hdrs[i].data_len;
    if (items[i].type != kTypeF32 && items[i].type != kTypeIG8 && items[i].type != 0x0101) {
      set_error("Incompatible type in model item " + items[i].name);
      return 1;
    }
    out[items[i].name] = items[i];
  }
  return 0;
}

// The tensor maps of o's weights and, on the digits, of its digit rows.
int out_maps(Context& c, OutColumns& o, int K) {
  if (o.digits && c.make_map(&o.map_ext, o.ext, OutColumns::pad(o.N), 128, kOutBN)) return 1;
  return c.make_map(&o.map_w, o.w, o.N, K, kOutBN);
}

}  // namespace

int Model::load(Context* c, const void* bin, size_t bytes, int enc_layers, int dec_layers, int heads) {
  ctx = c;
  H = heads;
  SB_CUDA(cudaSetDevice(c->device));
  std::map<std::string, Item> items;
  if (parse_items(bin, bytes, items)) return 1;

  auto need = [&items](const std::string& name) -> const Item* {
    auto it = items.find(name);
    if (it == items.end()) {
      set_error("model is missing parameter " + name);
      return nullptr;
    }
    return &it->second;
  };
  auto alloc = [this](void** dst, size_t nbytes) -> int {
    SB_CUDA(cudaMalloc(dst, nbytes));
    owned.push_back(*dst);
    return 0;
  };
  auto upload = [&](const void* src, size_t nbytes, void** dst) -> int {
    if (alloc(dst, nbytes)) return 1;
    SB_CUDA(cudaMemcpy(*dst, src, nbytes, cudaMemcpyHostToDevice));
    ctx->h2d_bytes += nbytes;
    return 0;
  };
  auto f32_vec = [&](const std::string& name, size_t n, float** dst) -> int {
    const Item* it = need(name);
    if (!it) return 1;
    if (it->elements() != n || it->bytes < n * 4) {
      set_error("parameter " + name + " has unexpected size");
      return 1;
    }
    return upload(it->data, n * 4, reinterpret_cast<void**>(dst));
  };
  auto scalar = [&](const std::string& name, float* v) -> int {
    const Item* it = need(name);
    if (!it) return 1;
    if (it->bytes < 4) {
      set_error("parameter " + name + " holds no value");
      return 1;
    }
    memcpy(v, it->data, 4);
    return 0;
  };
  // ig8 item [K,N]: blob = N rows of K int8 (B^T) then the f32 b_quant (Io.cc:227-242).
  auto weight = [&](const std::string& wname, const std::string& bname, DevWeight& w, const int8_t* override_q = nullptr,
                    const std::string& aq_name = "") -> int {
    const Item* it = need(wname);
    if (!it) return 1;
    if (it->shape.size() != 2 || it->bytes < static_cast<uint64_t>(it->shape[0]) * it->shape[1] + 4) {
      set_error("weight " + wname + " is not a 2-D intgemm8 item followed by its quantization multiplier");
      return 1;
    }
    int K = it->shape[0], N = it->shape[1];
    const int8_t* q = reinterpret_cast<const int8_t*>(it->data);
    if (wname == "Wemb") std::swap(K, N);  // stored [V][E]: as an output weight K = E, N = V
    memcpy(&w.bq, it->data + static_cast<size_t>(K) * N, 4);
    if (override_q) q = override_q;
    if (scalar(aq_name.empty() ? wname + "_QuantMultA" : aq_name, &w.aq)) return 1;
    w.K = K, w.N = N;
    w.um = 1.0f / (w.aq * w.bq);
    const float* bias = nullptr;
    if (!bname.empty()) {
      const Item* b = need(bname);
      if (!b) return 1;
      if (b->elements() != static_cast<size_t>(N) || b->bytes < 4ull * N) {
        set_error("bias " + bname + " has unexpected size");
        return 1;
      }
      bias = reinterpret_cast<const float*>(b->data);
    }
    if (K % 64 != 0 || N % 8 != 0) {
      set_error("weight " + wname + ": intgemm shape preconditions violated (K % 64, N % 8)");
      return 1;
    }
    std::vector<float> pb(N);
    host_prepare_bias(q, bias, w.aq, w.bq, K, N, pb.data());
    if (upload(q, static_cast<size_t>(K) * N, reinterpret_cast<void**>(&w.w))) return 1;
    if (upload(pb.data(), 4ul * N, reinterpret_cast<void**>(&w.pb))) return 1;
    if (ctx->make_map(&w.map128, w.w, N, K, 128)) return 1;
    if (N >= 32 && ctx->make_map(&w.map32, w.w, N, K, 32)) return 1;
    return 0;
  };
  auto ln = [&](const std::string& prefix, DevLN& l) -> int {
    return f32_vec(prefix + "_ln_scale", E, &l.scale) || f32_vec(prefix + "_ln_bias", E, &l.bias);
  };
  auto attention = [&](const std::string& prefix, AttnW& a) -> int {
    return weight(prefix + "_Wq", prefix + "_bq", a.q) || weight(prefix + "_Wk", prefix + "_bk", a.k) ||
           weight(prefix + "_Wv", prefix + "_bv", a.v) || weight(prefix + "_Wo", prefix + "_bo", a.o) ||
           ln(prefix + "_Wo", a.ln);
  };
  auto ffn = [&](const std::string& prefix, FfnW& f) -> int {
    return weight(prefix + "_ffn_W1", prefix + "_ffn_b1", f.w1) || weight(prefix + "_ffn_W2", prefix + "_ffn_b2", f.w2) ||
           ln(prefix + "_ffn_ffn", f.ln);
  };

  const Item* wemb = need("Wemb");
  if (!wemb) return 1;
  if (wemb->shape.size() != 2 || wemb->bytes < static_cast<uint64_t>(wemb->shape[0]) * wemb->shape[1] + 4) {
    set_error("Wemb is not a 2-D item followed by its quantization multiplier");
    return 1;
  }
  V = wemb->shape[0];
  E = wemb->shape[1];
  if (E % H != 0 || (E / H != 32 && E / H != 64)) {
    set_error("unsupported head size " + std::to_string(E / std::max(1, H)));
    return 1;
  }
  if (E != 256 && E != 512) {
    set_error("unsupported embedding size " + std::to_string(E) + " (256 and 512 are built)");
    return 1;
  }
  dh = E / H;
  memcpy(&emb_qm, wemb->data + static_cast<size_t>(V) * E, 4);
  inv_qm = 1 / emb_qm;  // Io.cc:281: `(1 / quantization_multiplier)` in float
  sqrt_e = sqrtf(static_cast<float>(E));
  if (upload(wemb->data, static_cast<size_t>(V) * E, reinterpret_cast<void**>(&emb_q))) return 1;

  // Output layer: dequantise the embedding and quantise it again (Io.cc:183-224): identical to the
  // stored bytes except that -128 becomes -127.
  {
    std::vector<float> deq(static_cast<size_t>(V) * E);
    const int8_t* q = reinterpret_cast<const int8_t*>(wemb->data);
    for (size_t i = 0; i < deq.size(); i++) deq[i] = static_cast<float>(q[i]) * inv_qm;
    std::vector<int8_t> req(deq.size());
    host_quantize(deq.data(), req.data(), emb_qm, deq.size());
    if (weight("Wemb", "decoder_ff_logit_out_b", out, req.data(), "none_QuantMultA")) return 1;
    std::vector<int32_t> c127(V);  // 127 * colsum per column
    for (int n = 0; n < V; n++) {
      int32_t cs = 0;
      for (int k = 0; k < E; k++) cs += req[static_cast<size_t>(n) * E + k];
      c127[n] = 127 * cs;
    }
    vocab.N = V, vocab.um = out.um, vocab.w = out.w, vocab.pb = out.pb;
    if (upload(c127.data(), 4ul * V, reinterpret_cast<void**>(&vocab.c127))) return 1;
  }
  // The fused argmax takes the digits when every column's offset fits them (their build reports one that does not),
  // otherwise the bound filter, whose slack eta covers the float roundings of the exact formula.
  {
    int bad = 0;
    auto alloc_tables = [&] {
      vocab.tables([&](auto*& p, size_t n) { bad = bad || alloc(reinterpret_cast<void**>(&p), n * sizeof(*p)); });
      return bad;
    };
    vocab.digits = true;
    int* d_flag = nullptr;
    int flag = 0;
    if (alloc_tables()) return 1;
    SB_CUDA(cudaMalloc(&d_flag, 4));
    SB_CUDA(cudaMemsetAsync(d_flag, 0, 4, c->stream));
    launch_out_tables(vocab, d_flag, c->stream);
    SB_CUDA(cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, c->stream));
    SB_CUDA(cudaStreamSynchronize(c->stream));
    SB_CUDA(cudaFree(d_flag));
    if (flag) {
      vocab.digits = false;
      if (alloc_tables()) return 1;
      launch_out_tables(vocab, nullptr, c->stream);
      std::vector<float> pbh(V);
      SB_CUDA(cudaMemcpy(pbh.data(), vocab.pb, 4ul * V, cudaMemcpyDeviceToHost));
      double pbabs = 0;
      for (float v : pbh) pbabs = std::max(pbabs, static_cast<double>(fabsf(v)));
      const double vmax = static_cast<double>(E) * 254.0 * 128.0;
      vocab.eta = static_cast<float>((2.0 * vmax * vocab.um + pbabs) * ldexp(1.0, -22));
    }
    if (out_maps(*ctx, vocab, E)) return 1;
  }

  enc.resize(enc_layers);
  for (int i = 0; i < enc_layers; i++) {
    const std::string p = "encoder_l" + std::to_string(i + 1);
    if (attention(p + "_self", enc[i].self) || ffn(p, enc[i].ffn)) return 1;
  }
  dec.resize(dec_layers);
  for (int j = 0; j < dec_layers; j++) {
    const std::string p = "decoder_l" + std::to_string(j + 1);
    if (weight(p + "_rnn_W", "", dec[j].rnn_w) || weight(p + "_rnn_Wf", p + "_rnn_bf", dec[j].rnn_wf) ||
        ln(p + "_rnn_ffn", dec[j].rnn_ln) || attention(p + "_context", dec[j].ctx) || ffn(p, dec[j].ffn))
      return 1;
  }
  F = enc_layers ? enc[0].ffn.w1.N : (dec_layers ? dec[0].ffn.w1.N : 0);

  // sinusoidal_signal (TensorOps.cc:245-265), evaluated with the host libm like the reference
  max_pos = 1024;
  std::vector<float> table(static_cast<size_t>(max_pos) * E);
  {
    float num_timescales = static_cast<float>(E) / 2;
    float inc = std::log(10000.0F) / (num_timescales - 1.0F);
    for (size_t pp = 0; pp < static_cast<size_t>(max_pos); ++pp) {
      for (int i = 0; i < num_timescales; ++i) {
        float v = pp * std::exp(i * -inc);
        table[pp * E + i] = std::sin(v);
        table[pp * E + i + static_cast<int>(num_timescales)] = std::cos(v);
      }
    }
  }
  if (upload(table.data(), table.size() * 4, reinterpret_cast<void**>(&pos))) return 1;
  return 0;
}

void Model::destroy() {
  for (auto& l : lanes) l->destroy();
  lanes.clear();
  if (ctx) cudaSetDevice(ctx->device);
  for (void* p : owned) cudaFree(p);
  owned.clear();
}

// ------------------------------------------------------------------ workspace
namespace {

// Rows of the scoring pass's output layer per launch: bounds its strip partials to ceil(N / 64) * 16 k * 8 bytes.
constexpr int kScoreChunk = 16384;

}  // namespace

// ------------------------------------------------------------------ GEMM helpers
namespace {

int pick_bn(int M, int N, int n_prob, bool full_row) {
  if (full_row) return N;  // RES_LN: one CTA owns whole rows
  const int m_tiles = (M + kBM - 1) / kBM;
  int bn = 256;
  while (bn > 64 && static_cast<long>(m_tiles) * ((N + bn - 1) / bn) * n_prob < 148) bn >>= 1;
  if (N < bn) bn = std::max(64, 1 << static_cast<int>(ceil(log2(static_cast<double>(N)))));
  return std::min(bn, 256);
}

struct GemmCall {
  Context* c;
  GemmBatch b{};
  int n = 0;
  int epi = EPI_F32;
  int bn = 256;
  const char* tag = "gemm";
  GemmCall(Context* ctx, const char* tag_, int M, int N, int K, int epilogue, int n_prob_hint = 1)
      : c(ctx), epi(epilogue), tag(tag_) {
    b.M = M, b.N = N, b.K = K;
    bn = pick_bn(M, N, n_prob_hint, epilogue == EPI_RES_LN);
  }
  // adds one problem; returns its slot (or nullptr on failure)
  GemmProblem* add(const int8_t* A, const int8_t* Wt, const float* pb, float um) {
    GemmProblem& p = b.prob[n];
    memset(&p, 0, sizeof(p));
    const uint32_t box_b = static_cast<uint32_t>(std::min(bn, 256));
    if (c->make_map(&p.tma_a, A, b.M, b.K, kBM)) return nullptr;
    if (c->make_map(&p.tma_b, Wt, b.N, b.K, box_b)) return nullptr;
    p.pb = pb, p.um = um;
    p.ln_eps = 1e-6f;  // TensorOps.hh:67-68
    n++;
    return &p;
  }
  GemmProblem* add(const int8_t* A, const DevWeight& w) { return add(A, w.w, w.pb, w.um); }
  int launch() {
    const double M = b.M, N = b.N, K = b.K;
    double out_bytes = 0;
    for (int i = 0; i < n; i++) {
      const GemmProblem& p = b.prob[i];
      if (epi == EPI_F32 || epi == EPI_ACC) out_bytes += 4 * M * N;
      if (epi == EPI_QUANT) out_bytes += M * N;
      if (epi == EPI_RES_LN) out_bytes += 4 * M * N + (p.out ? 4 * M * N : 0) + p.n_qout * M * N;
    }
    LaunchScope ls(*c, tag, 2.0 * M * N * K * n, n * (M * K + N * K) + out_bytes);
    launch_gemm_i8(b, n, epi, bn, c->stream);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
      set_error(std::string("GEMM launch failed: ") + cudaGetErrorString(e));
      return 1;
    }
    return 0;
  }
};

QuantOuts qouts() {
  QuantOuts q;
  memset(&q, 0, sizeof(q));
  return q;
}
void qadd(QuantOuts& q, int8_t* p, float aq) {
  q.ptr[q.n] = p;
  q.aq[q.n] = aq;
  q.n++;
}
void padd(GemmProblem* p, int8_t* ptr, float aq) {
  p->qout[p->n_qout] = ptr;
  p->aq_out[p->n_qout] = aq;
  p->n_qout++;
}

// The row-tile kernel's arguments for one layer's Wo + residual + LN and FFN + residual + LN over M rows: the weights,
// biases, multipliers and LayerNorms of `att` and `ffn`.  The caller adds the A operand's map, y_park and the outputs.
RowsFfnArgs rows_ffn_args(const AttnW& att, const FfnW& ffn, const float* res, int M) {
  RowsFfnArgs k{};
  k.map_wo = att.o.map128, k.map_w1 = ffn.w1.map128, k.map_w2 = ffn.w2.map128;
  k.pb_o = att.o.pb, k.pb_1 = ffn.w1.pb, k.pb_2 = ffn.w2.pb;
  k.um_o = att.o.um, k.um_1 = ffn.w1.um, k.um_2 = ffn.w2.um;
  k.aq_1 = ffn.w1.aq, k.aq_2 = ffn.w2.aq;
  k.res = res;
  k.ln1_scale = att.ln.scale, k.ln1_bias = att.ln.bias;
  k.ln2_scale = ffn.ln.scale, k.ln2_bias = ffn.ln.bias, k.eps = 1e-6f;
  k.M = M;
  return k;
}

}  // namespace

// ------------------------------------------------------------------ operator API
int qmm_affine_host(Context& c, const float* x, size_t M, size_t K, const int8_t* W, size_t N, const float* bias,
                    float aq, float bq, const uint32_t* indices, size_t n_idx, float* y, int8_t* qa_out,
                    int32_t* acc_out) {
  std::lock_guard<std::recursive_mutex> ctx_lock(c.mu);
  SB_CUDA(cudaSetDevice(c.device));
  if (K % 64 != 0 || N % 8 != 0 || (indices && n_idx % 8 != 0)) {
    set_error("qmm::affine shape preconditions violated: K % 64 == 0, N % 8 == 0, indices % 8 == 0");
    return 1;
  }
  if (M == 0) return 0;
  // PrepareBias on the FULL B, then gather (qmm/Intgemm.inl.cc:33-66)
  std::vector<float> pb(N);
  host_prepare_bias(W, bias, aq, bq, K, N, pb.data());
  const size_t Nout = indices ? n_idx : N;
  float *dx = nullptr, *dpb = nullptr, *dy = nullptr, *dpbs = nullptr;
  int8_t *dqa = nullptr, *dW = nullptr, *dWs = nullptr;
  int32_t* dacc = nullptr;
  uint32_t* didx = nullptr;
  Workspace ws;
  ws.add(dx, M * K), ws.add(dqa, M * K), ws.add(dW, N * K), ws.add(dpb, N), ws.add(dy, M * Nout);
  if (acc_out) ws.add(dacc, M * Nout);
  if (indices) ws.add(didx, n_idx), ws.add(dWs, n_idx * K), ws.add(dpbs, n_idx);
  if (ws.carve(c)) return 1;
  cudaStream_t s = c.stream;
  SB_CUDA(cudaMemcpyAsync(dx, x, M * K * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(dW, W, N * K, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(dpb, pb.data(), N * 4, cudaMemcpyHostToDevice, s));
  c.h2d_bytes += M * K * 4 + N * K + N * 8;
  const int8_t* Wuse = dW;
  const float* pbuse = dpb;
  if (indices) {
    SB_CUDA(cudaMemcpyAsync(didx, indices, n_idx * 4, cudaMemcpyHostToDevice, s));
    {
      LaunchScope ls(c, "gather_rows", 0, 2.0 * n_idx * K);
      launch_gather_rows(dW, dpb, nullptr, didx, static_cast<int>(n_idx), static_cast<int>(K), dWs, dpbs, nullptr, s);
    }
    Wuse = dWs, pbuse = dpbs;
  }
  QuantOuts q = qouts();
  qadd(q, dqa, aq);
  {
    LaunchScope ls(c, "quantize", 0, 5.0 * M * K);
    launch_quantize(dx, M * K, q, s);
  }
  const float um = 1.0f / (aq * bq);
  {
    GemmCall g(&c, "qmm_affine_gemm", static_cast<int>(M), static_cast<int>(Nout), static_cast<int>(K), EPI_F32);
    GemmProblem* p = g.add(dqa, Wuse, pbuse, um);
    if (!p) return 1;
    p->out = dy, p->ldo = static_cast<int>(Nout);
    if (g.launch()) return 1;
  }
  if (acc_out) {
    GemmCall g(&c, "qmm_acc_gemm", static_cast<int>(M), static_cast<int>(Nout), static_cast<int>(K), EPI_ACC);
    GemmProblem* p = g.add(dqa, Wuse, pbuse, um);
    if (!p) return 1;
    p->out = dacc, p->ldo = static_cast<int>(Nout);
    if (g.launch()) return 1;
    SB_CUDA(cudaMemcpyAsync(acc_out, dacc, M * Nout * 4, cudaMemcpyDeviceToHost, s));
  }
  if (qa_out) SB_CUDA(cudaMemcpyAsync(qa_out, dqa, M * K, cudaMemcpyDeviceToHost, s));
  SB_CUDA(cudaMemcpyAsync(y, dy, M * Nout * 4, cudaMemcpyDeviceToHost, s));
  c.d2h_bytes += M * Nout * 4;
  SB_CUDA(cudaStreamSynchronize(s));
  if (qa_out) {
    for (size_t i = 0; i < M * K; i++) qa_out[i] = static_cast<int8_t>(static_cast<int>(static_cast<uint8_t>(qa_out[i])) - 127);
  }
  return 0;
}

// ------------------------------------------------------------------ kernel routes
namespace {

enum class SelfAttn { Fused, Rowwise, Tiled, Long };
enum class Cross { Cached, Rc, Rcl };

const char* const kSelfAttnName[] = {"Fused", "Rowwise", "Tiled", "Long"};  // indexed by SelfAttn

enum class EncFfn { Rows, Gemm };
// output: the fused argmax GEMM (out_argmax.cu, in the encoding Model::load chose), logits tap + argmax_rows, the
// scores GEMM (the fused GEMM with every logit evaluated exactly) + score_step or sample_step, or the logits GEMM alone +
// topk_sample (top-k sampling, which needs every logit of a row)
enum class Out { Argmax, Logits, Scores, TopK };

struct Routes {
  SelfAttn self;
  Cross cross;
  EncFfn ffn;
  Out out;
};

// Which kernel runs each stage of one forward call that has more than one.  The two environment variables are read on
// every call, so that tests can switch kernels between calls; a value not listed below means the default.
Routes choose_routes(const Model& m, int T, int B, bool fast, bool logits, bool scores, bool topk) {
  const int E = m.E, H = m.H, dh = m.dh;
  auto env_is = [](const char* env, const char* v) { return env != nullptr && strcmp(env, v) == 0; };
  Routes r{};
  // SLIMT_B200_SELFATTN = split keeps the projections and the attention as separate kernels; rowwise | tiled | long
  // also force that attention kernel (parity cross-checks)
  const char* sa = getenv("SLIMT_B200_SELFATTN");
  if (env_is(sa, "rowwise")) r.self = SelfAttn::Rowwise;
  else if (env_is(sa, "tiled")) r.self = SelfAttn::Tiled;
  else if (env_is(sa, "long")) r.self = SelfAttn::Long;
  else if (!env_is(sa, "split") && enc_attention_supported(E, H, dh, T)) r.self = SelfAttn::Fused;
  // the tiled kernel's 64-query x 128-key tiles pay off from T > 64 (mixed lengths: 15.9 -> 8.5 ms per layer of a
  // 1M-word batch); at T <= 64 with head size 64 (base) half of every tile is idle and the row-wise kernel is faster
  // (666 vs 1149 us per layer at 4096 x 32)
  else if (T <= 64) r.self = SelfAttn::Rowwise;
  // The long kernel (self_attention_long.cu) takes what the tiled kernel cannot hold (T > 556 at head size 32, T > 400
  // at 64) and 257 .. 384 tokens, where its 32-row score block lets two or three blocks share an SM against the tiled
  // kernel's one: 16.5 vs 19.9 ms for the six layers of 455 x 288, 20.1 vs 22.3 ms at 341 x 384; at 256 x 512 the
  // tiled kernel's 64-row reuse wins, 29.3 vs 30.4 ms (B200, 1000 W; profiles/r4_long_bench.jsonl).
  else if ((T > 256 && T <= 384) || !self_attention_tiled_supported(T, dh)) r.self = SelfAttn::Long;
  else r.self = SelfAttn::Tiled;

  // Cross-attention K/V: the reference re-projects them every step (Modules.cc:244-249); so do the recompute kernels
  // (tensor cores, from the u8 encoder output); the cached kernel reads them projected once.  Small batches take the
  // cached kernel: below ~4 k source tokens the recompute kernel has fewer sentence groups than SMs and its launch is
  // all latency (64 x 32: 8.6 us cached against 12.8 us recomputed per launch, 5.40 -> 5.13 ms per batch; the two are
  // bit-identical).  SLIMT_B200_CROSS = cached | rc overrides the choice (tests, A/B runs).
  const char* ca = getenv("SLIMT_B200_CROSS");
  if (env_is(ca, "cached") || (!env_is(ca, "rc") && static_cast<long>(B) * T <= 4096)) r.cross = Cross::Cached;
  else if (cross_attention_rc_supported(E, H, dh, T)) r.cross = Cross::Rc;
  // long sentences (65 .. 256 tokens) take the sentence-at-a-time recompute kernel (cross_attention_rc.cu; bit-exact mode)
  else if (!fast && cross_attention_rcl_supported(E, H, dh, T)) r.cross = Cross::Rcl;
  else r.cross = Cross::Cached;

  // Wo + residual + LN, FFN1 + ReLU, FFN2 + residual + LN in one row-tile kernel, 128 rows per CTA
  r.ffn = E == 256 && m.F == 1536 ? EncFfn::Rows : EncFfn::Gemm;

  // a caller that wants the logits gets them from the tap (and scores or samples, when asked for, from them); scores
  // or samples alone come from the scores epilogue of the fused GEMM.  Top-k sampling reads the tap's logits, whether
  // or not the caller wants a copy.
  r.out = topk ? Out::TopK : logits ? Out::Logits : scores ? Out::Scores : Out::Argmax;
  return r;
}

// ------------------------------------------------------------------ Model::forward
// What the stages of one forward call share: its shape, its routes, its workspace buffers and their tensor maps.
// Built as Pass{m, c, a, c.stream}, which value-initialises the rest: a buffer no chosen route reads stays null.
struct Pass {
  Model& m;
  Context& c;
  ForwardArgs& a;
  cudaStream_t s;
  int B, T, R, E, F, H, dh, Le, Ld, max_steps, Nout;  // Nout: with a lazy shortlist the vocabulary until its callback
  double src_tokens;
  bool lazy_sl, use_sl;
  // scoring pass (a.targets set): Tt target positions per sentence, M = B * Tt decoder rows, always bit-exact arithmetic.
  // Decode loop: M = B * K decoder rows, K = a.beam for beam search (bit-exact arithmetic too), else 1.
  bool scoring, fast;
  int Tt, M, K;
  Routes route;
  // batch inputs and outputs: workspace copies with host buffers, the caller's buffers with device_io
  uint32_t *d_tokens, *d_lengths, *d_steps, *d_forced, *d_sl, *d_rows, *tgt_len;
  uint64_t* d_keys;  // [B] sampling keys (null: the row index)
  // encoder; Kc/Vc: the cross K/V projected once per decoder layer (Cross::Cached)
  float *x0, *x1, *Qb, *Kb, *Vb, *Kc[2], *Vc[2];
  int8_t *qa[4], *attn_q, *ffn_q;
  // decoder state (Model.cc:111-185); counters: [0] n_done, [1] step counter, [2] ticket
  float *xd, *hb, *qd, *zb, *state[2], *d_logits, *d_align_all;  // zb: the first of two decoder layers' output
  // beam search: the other half of each layer's state ping-pong, the step's candidates, the slots' cumulative scores,
  // each sentence's width, the step records and the finished hypotheses (kernels.cuh)
  float* state_nx[2];
  BeamCand* cand;
  float* cum;
  uint8_t* width;
  BeamRec* d_rec;
  BeamFin* d_fin;
  // scoring pass: the targets, the SSRU's two projections of all rows, h's u8 copy (Wq's operand)
  uint32_t* d_tgt;
  float *Fb, *Wx;
  int8_t* hq;
  float* d_scores;    // [max_steps][B]
  float2* partials;   // [ceil(Nout / 64)][B] strip partials of the step's scores
  int8_t *xq[2], *zq[2], *caq, *oq;
  unsigned long long* best;
  uint8_t* done;
  int* counters;
  OutColumns out;  // the output layer's columns: the model's, or the shortlist's gathered copy
  CUtensorMap map_attn_q;  // u8 [R][E], box {128 B, 128 rows}: operand of the encoder's row-tile kernel
  CUtensorMap map_qa[3], map_qa32[3], mapK[2], mapV[2];
  CUtensorMap map_xq[2], map_zq[2], map_caq;  // u8 activation operands of the row-tile kernels, box {128 B, 32 rows}
  CUtensorMap map_oq;
  int plan(), plan_step(Workspace& ws), plan_score(Workspace& ws), carve(const Workspace& ws);
  int encode(), prepare_cross(), prepare_output(), decode_step(int step), decode(), score();
  int poll_done(int step, bool* all_done);
  QuantOuts enc_inputs(int i);
  int cross_attention_mq(int l, int queries, float* al, const char* tag, const char* what);
  int wo_ffn(int l, float* z, int8_t* xf, int8_t* xw, const char* tag);
  int scores_gemm(const CUtensorMap& map, int rows, const char* tag);
  ScoreStepArgs score_step_args(int rows, const int8_t* oq_rows, const uint32_t* forced, int step, float* scores) const;
};

// Checks the request, chooses the routes and plans the workspace: each buffer is listed once, under the condition in
// which the chosen routes read it.  The buffers both paths share are listed here, the rest by plan_step / plan_score.
int Pass::plan() {
  B = static_cast<int>(a.B), T = static_cast<int>(a.T), E = m.E, F = m.F, H = m.H, dh = m.dh;
  R = B * T;
  Le = static_cast<int>(m.enc.size()), Ld = static_cast<int>(m.dec.size());
  if (T > m.max_len()) {
    set_error("sequence length " + std::to_string(T) + " exceeds the supported maximum of " + std::to_string(m.max_len()));
    return 1;
  }
  if (Ld < 1 || 2 * Ld > kMaxQuantOut) {
    set_error("decoder_layers must be 1 or 2");
    return 1;
  }
  // Model.cc:160: size_t max_seq_length = limit_factor * source_sequence_length (float product, truncated).  The first
  // decoder step runs before that loop (Model.cc:145-157), so at least one step is always executed and recorded.
  max_steps = forward_max_steps(a.limit_factor, a.T);
  src_tokens = static_cast<double>(R);  // cross-attention reads only valid keys; exact count when lengths are on the host
  if (!a.device_io || c.profiling) {
    // per-kernel accounting only (profiling passes are never timed): with device-resident input the lengths are fetched
    std::vector<uint32_t> lens_h(B);
    const uint32_t* lp = a.lengths;
    if (a.device_io) {
      SB_CUDA(cudaMemcpyAsync(lens_h.data(), a.lengths, 4ul * B, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaStreamSynchronize(s));
      lp = lens_h.data();
    }
    src_tokens = 0;
    for (int b = 0; b < B; b++) src_tokens += std::min<uint32_t>(lp[b], T);
  }
  lazy_sl = a.shortlist == nullptr && a.shortlist_cb != nullptr && !a.device_io;
  use_sl = lazy_sl || (a.shortlist != nullptr && a.n_shortlist > 0);
  Nout = use_sl && !lazy_sl ? static_cast<int>(a.n_shortlist) : m.V;  // lazy: upper bound until the callback ran
  if (use_sl && !lazy_sl && a.n_shortlist % 8 != 0) {
    set_error("shortlist size must be a multiple of 8");
    return 1;
  }
  scoring = a.targets != nullptr;
  K = a.beam > 0 ? a.beam : 1;
  fast = c.fast && !scoring && a.beam == 0;
  route = choose_routes(m, T, B, fast, a.logits != nullptr, a.scores != nullptr || a.sample, a.top_k > 0);
  if (scoring || a.beam > 0) {
    // T_target (or K) queries read each layer's cross K/V: projected once (Cached); every logit evaluated exactly (Scores)
    route.cross = Cross::Cached;
    route.out = Out::Scores;
  }

  const size_t RE = static_cast<size_t>(R) * E, N = static_cast<size_t>(Nout);
  // the output layer's columns are the model's unless the shortlist's are listed below; a subset of the columns fits
  // the model's encoding and its eta
  out = m.vocab;
  Workspace ws;
  if (!a.device_io) ws.add(d_tokens, R), ws.add(d_lengths, B);
  ws.add(x0, RE), ws.add(x1, RE);
  for (int i = 0; i < std::max(3, 2 * Ld); i++) ws.add(qa[i], RE);  // encoder q/k/v inputs, decoder layers' K/V inputs
  if (route.self != SelfAttn::Fused) ws.add(Qb, RE), ws.add(Kb, RE), ws.add(Vb, RE);
  ws.add(attn_q, RE);
  if (route.ffn == EncFfn::Gemm) ws.add(ffn_q, static_cast<size_t>(R) * F);
  for (int l = 0; l < Ld && route.cross == Cross::Cached; l++) ws.add(Kc[l], RE), ws.add(Vc[l], RE);
  if (use_sl) {
    if (!a.device_io) ws.add(d_sl, N);
    out.N = Nout;
    ws.add(out.w, N * E), ws.add(out.pb, N), ws.add(out.c127, N);
    if (route.out == Out::Argmax) out.tables([&ws](auto*& p, size_t n) { ws.add(p, n); });
  }
  return scoring ? plan_score(ws) : plan_step(ws);
}

// Reserves the workspace once a path has listed its buffers, and makes the encoder's tensor maps.
int Pass::carve(const Workspace& ws) {
  if (ws.carve(c)) return 1;
  // cross-attention K/V operands: projected once (Cross::Cached), or the u8 encoder output the recompute kernels read
  const uint32_t box_rows = static_cast<uint32_t>(cross_attention_box_rows(T));
  for (int l = 0; l < Ld; l++)
    if (route.cross == Cross::Cached
            ? c.make_map_f32(&mapK[l], Kc[l], R, E, box_rows) || c.make_map_f32(&mapV[l], Vc[l], R, E, box_rows)
            : c.make_map(&mapK[l], qa[2 * l], R, E, 32) || c.make_map(&mapV[l], qa[2 * l + 1], R, E, 32))
      return 1;
  if (route.ffn == EncFfn::Rows && c.make_map(&map_attn_q, attn_q, R, E, 128)) return 1;
  if (route.self == SelfAttn::Fused)
    for (int i = 0; i < 3; i++)
      if (c.make_map(&map_qa[i], qa[i], R, E, 128) || c.make_map(&map_qa32[i], qa[i], R, E, 32)) return 1;
  return 0;
}

// The decode loop's buffers and the row-tile kernels' operand maps: one row per sentence, or K with beam search.
int Pass::plan_step(Workspace& ws) {
  M = B * K;
  const size_t BE = static_cast<size_t>(M) * E, SB = static_cast<size_t>(max_steps) * B;
  ws.add(xd, BE), ws.add(hb, BE), ws.add(qd, BE), ws.add(zb, BE);
  for (int l = 0; l < Ld; l++) ws.add(state[l], BE);
  ws.add(xq[0], BE), ws.add(xq[1], BE), ws.add(zq[0], BE), ws.add(zq[1], BE), ws.add(caq, BE), ws.add(oq, BE);
  ws.add(best, M), ws.add(done, B), ws.add(tgt_len, B), ws.add(counters, 64);
  if (a.beam > 0) {
    for (int l = 0; l < Ld; l++) ws.add(state_nx[l], BE);
    ws.add(cand, static_cast<size_t>(M) * K), ws.add(cum, M), ws.add(width, B);
    ws.add(d_rec, static_cast<size_t>(max_steps) * M), ws.add(d_fin, M);
    ws.add(partials, (Nout + kScoreStrip - 1) / kScoreStrip * static_cast<size_t>(M));
  }
  if (!a.device_io && a.beam == 0) {
    ws.add(d_steps, SB);
    if (a.forced) ws.add(d_forced, SB);
  }
  if (route.out == Out::Logits || route.out == Out::TopK) ws.add(d_logits, static_cast<size_t>(B) * Nout);
  if (a.scores && !a.device_io) ws.add(d_scores, SB);
  if ((a.scores || a.sample) && route.out != Out::TopK)
    ws.add(partials, (Nout + kScoreStrip - 1) / kScoreStrip * static_cast<size_t>(B));
  if (a.sample && a.keys && !a.device_io) ws.add(d_keys, B);
  // head-0 probabilities of every step stay on the device and come back in one copy after the loop
  if (a.alignment) ws.add(d_align_all, SB * K * T);
  if (!a.device_io && a.sentence_tokens) ws.add(d_rows, SB);
  if (carve(ws)) return 1;
  if (a.device_io) {
    d_tokens = const_cast<uint32_t*>(a.tokens), d_lengths = const_cast<uint32_t*>(a.lengths), d_steps = a.step_tokens;
    d_forced = const_cast<uint32_t*>(a.forced), d_sl = use_sl ? const_cast<uint32_t*>(a.shortlist) : nullptr;
    d_scores = a.scores;
    d_keys = const_cast<uint64_t*>(a.keys);
  }
  for (int i = 0; i < 2; i++)
    if (c.make_map(&map_xq[i], xq[i], M, E, kRowTile) || c.make_map(&map_zq[i], zq[i], M, E, kRowTile)) return 1;
  return c.make_map(&map_caq, caq, M, E, kRowTile) || c.make_map(&map_oq, oq, M, E, kBM);
}

// The scoring pass's buffers: one row per (sentence, target position); the layer input xd is rewritten in place by each
// layer's FFN.  The output operand's maps are made per row chunk.
int Pass::plan_score(Workspace& ws) {
  Tt = static_cast<int>(a.target_T), M = B * Tt;
  if (Tt > m.max_len()) {
    set_error("target length " + std::to_string(Tt) + " exceeds the supported maximum of " + std::to_string(m.max_len()));
    return 1;
  }
  const size_t ME = static_cast<size_t>(M) * E, rows = std::min(M, kScoreChunk);
  ws.add(d_tgt, M);
  ws.add(xd, ME), ws.add(Fb, ME), ws.add(Wx, ME), ws.add(hb, ME), ws.add(qd, ME);
  ws.add(xq[0], ME), ws.add(xq[1], ME), ws.add(hq, ME), ws.add(caq, ME), ws.add(oq, ME);
  ws.add(d_scores, M), ws.add(best, rows), ws.add(partials, (Nout + kScoreStrip - 1) / kScoreStrip * rows);
  if (a.alignment) ws.add(d_align_all, ME / E * T);
  return carve(ws) || c.make_map(&map_caq, caq, M, E, kRowTile);
}

// The u8 operands quantised from the input of encoder layer i: its q/k/v projections', or for i == Le every decoder
// layer's cross K/V projections'.
QuantOuts Pass::enc_inputs(int i) {
  QuantOuts q = qouts();
  if (i < Le) {
    const AttnW& A = m.enc[i].self;
    qadd(q, qa[0], A.q.aq), qadd(q, qa[1], A.k.aq), qadd(q, qa[2], A.v.aq);
  } else {
    for (int l = 0; l < Ld; l++) qadd(q, qa[2 * l], m.dec[l].ctx.k.aq), qadd(q, qa[2 * l + 1], m.dec[l].ctx.v.aq);
  }
  return q;
}

// Multi-query cross-attention of decoder layer l against its cached K/V, `queries` consecutive rows per sentence (beam
// search's K slots, the scoring pass's Tt target positions); head 0's probabilities go to al when it is set.  `what`
// names the path in the error.
int Pass::cross_attention_mq(int l, int queries, float* al, const char* tag, const char* what) {
  QuantOuts q = qouts();
  qadd(q, caq, m.dec[l].ctx.o.aq);
  const double Md = M, Ed = E;
  LaunchScope ls(c, tag, 4.0 * Md * (src_tokens / B) * Ed,
                 Md * Ed * 5.0 + 2.0 * src_tokens * Ed * 4.0 + (al ? 4.0 * Md * T : 0.0));
  const int rc = self_attention_tiled_supported(T, dh)
                     ? launch_self_attention_tiled(qd, Kc[l], Vc[l], d_lengths, B, T, H, dh, q, s, queries, al)
                     : launch_self_attention_long(qd, Kc[l], Vc[l], d_lengths, B, T, H, dh, q, s, queries, al);
  if (rc) {
    set_error(std::string(what) + " cross-attention: no kernel for head size " + std::to_string(dh) + " over " +
              std::to_string(T) + " source tokens");
    return 1;
  }
  return 0;
}

// Wo + residual + LN, FFN1 + ReLU, FFN2 + residual + LN of decoder layer l over the M rows in one row-tile kernel
// (Modules.cc:308-316, 251-257).  After the last layer the output goes only into the output operand (signed for the
// fused GEMMs, u8 for the generic logits GEMM of the tap and of top-k); after an earlier layer into z and the next
// layer's SSRU operands xf and xw.
int Pass::wo_ffn(int l, float* z, int8_t* xf, int8_t* xw, const char* tag) {
  const DecLayerW& L = m.dec[l];
  const bool last = l + 1 == Ld;
  RowsFfnArgs k = rows_ffn_args(L.ctx, L.ffn, hb, M);
  k.map_a = map_caq;
  if (last) {
    k.zq[0] = reinterpret_cast<uint8_t*>(oq), k.zaq[0] = m.out.aq, k.n_zq = 1;
    k.zq_signed = route.out == Out::Logits || route.out == Out::TopK ? 0 : 1;
  } else {
    k.z_out = z;
    k.zq[0] = reinterpret_cast<uint8_t*>(xf), k.zaq[0] = m.dec[l + 1].rnn_wf.aq;
    k.zq[1] = reinterpret_cast<uint8_t*>(xw), k.zaq[1] = m.dec[l + 1].rnn_w.aq;
    k.n_zq = 2;
  }
  const double Md = M, Ed = E, Fd = F;
  LaunchScope ls(c, tag, 2.0 * Md * (Ed * Ed + 2.0 * Ed * Fd),
                 Ed * Ed + 2.0 * Ed * Fd + Md * Ed * (1.0 + 4.0 + (last ? 1.0 : 6.0)));
  if (launch_rows_ffn(k, E, F, kRowTile, fast, s)) {
    set_error("fused FFN kernel: unsupported sizes E=" + std::to_string(E) + " F=" + std::to_string(F));
    return 1;
  }
  return 0;
}

// The output GEMM with the scores epilogue over `rows` rows of the operand `map`: every logit evaluated exactly, each
// row's best column into best and its strip partials (of the logits tempered by inv_t when sampling) into partials.
int Pass::scores_gemm(const CUtensorMap& map, int rows, const char* tag) {
  const double Rd = rows, Nd = Nout, Kd = E, strips = (Nout + kScoreStrip - 1) / kScoreStrip;
  LaunchScope ls(c, tag, 2.0 * Rd * Nd * Kd, Rd * Kd + Nd * Kd + 8.0 * Nd + 8.0 * Rd + 8.0 * Rd * strips);
  if (launch_out_scores(out, map, rows, E, best, partials, a.sample ? a.inv_t : 1.0f, c.num_sms, s)) {
    set_error("output GEMM (scores): unsupported K " + std::to_string(E));
    return 1;
  }
  return 0;
}

// score_step's arguments for `rows` output rows whose operands start at oq_rows; forced and scores are [step][rows].
// The sampling fields, which only sample_step reads, are the decode step's to set.
ScoreStepArgs Pass::score_step_args(int rows, const int8_t* oq_rows, const uint32_t* forced, int step,
                                    float* scores) const {
  ScoreStepArgs k{};
  k.partials = partials, k.best = best, k.forced = forced, k.shortlist = use_sl ? d_sl : nullptr;
  k.oq = oq_rows, k.w = out.w, k.c127 = out.c127, k.pb = out.pb, k.um = out.um;
  k.logits = route.out == Out::Logits || route.out == Out::TopK ? d_logits : nullptr;
  k.B = rows, k.N = Nout, k.K = E, k.step = step, k.scores = scores;
  return k;
}

int Pass::encode() {
  if (!a.device_io) {
    SB_CUDA(cudaMemcpyAsync(d_tokens, a.tokens, 4ul * R, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_lengths, a.lengths, 4ul * B, cudaMemcpyHostToDevice, s));
    c.h2d_bytes += 4ul * R + 4ul * B;
  }
  // ---- embedding (Model.cc:195-197)
  {
    const QuantOuts q = Le > 0 ? enc_inputs(0) : qouts();
    LaunchScope ls(c, "enc_embed", 0, (1.0 + 4.0 + q.n) * R * E);
    launch_embed(d_tokens, m.emb_q, m.inv_qm, m.sqrt_e, m.pos, R, T, E, 1, 0, x0, q, s);
  }

  // ---- encoder (Transformer.cc:57-69; EncoderLayer::forward Modules.cc:321-334)
  for (int i = 0; i < Le; i++) {
    const EncLayerW& L = m.enc[i];
    if (route.self == SelfAttn::Fused) {
      // q/k/v projections + scaled dot-product attention in one kernel: Q, K, V stay on the SM (enc_attention.cu)
      EncAttnArgs k{};
      k.map_aq = map_qa[0], k.map_ak = map_qa[1], k.map_av = map_qa[2];
      k.map_aq32 = map_qa32[0], k.map_ak32 = map_qa32[1], k.map_av32 = map_qa32[2];
      k.map_wq = L.self.q.map32, k.map_wk = L.self.k.map32, k.map_wv = L.self.v.map32;
      k.pb_q = L.self.q.pb, k.pb_k = L.self.k.pb, k.pb_v = L.self.v.pb;
      k.um_q = L.self.q.um, k.um_k = L.self.k.um, k.um_v = L.self.v.um;
      k.lengths = d_lengths, k.B = B, k.T = T;
      // 1/sqrt(dim_head) evaluated in double then narrowed, as `1.0F / std::sqrt(size_t)` does (Modules.cc:43)
      k.dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
      k.out_q = reinterpret_cast<uint8_t*>(attn_q), k.aq_out = L.self.o.aq;
      const double Rd = R, Ed = E;
      LaunchScope ls(c, "enc_qkv_attention_fused", 2.0 * Rd * Ed * Ed * 3.0, 4.0 * Rd * Ed + 3.0 * Ed * Ed);
      if (launch_enc_attention(k, c.num_sms, s)) {
        set_error("fused encoder attention kernel launch failed");
        return 1;
      }
    } else {
      {
        GemmCall g(&c, "enc_gemm_qkv_f32", R, E, E, EPI_F32, 3);
        GemmProblem* pq = g.add(qa[0], L.self.q);
        GemmProblem* pk = g.add(qa[1], L.self.k);
        GemmProblem* pv = g.add(qa[2], L.self.v);
        if (!pq || !pk || !pv) return 1;
        pq->out = Qb, pk->out = Kb, pv->out = Vb;
        pq->ldo = pk->ldo = pv->ldo = E;
        if (g.launch()) return 1;
      }
      QuantOuts q = qouts();
      qadd(q, attn_q, L.self.o.aq);
      LaunchScope ls(c, "enc_self_attention", 0, 13.0 * R * E);
      int rc = 1;
      switch (route.self) {
        case SelfAttn::Rowwise: rc = launch_self_attention(Qb, Kb, Vb, d_lengths, B, T, H, dh, q, s); break;
        case SelfAttn::Tiled: rc = launch_self_attention_tiled(Qb, Kb, Vb, d_lengths, B, T, H, dh, q, s); break;
        case SelfAttn::Long: rc = launch_self_attention_long(Qb, Kb, Vb, d_lengths, B, T, H, dh, q, s); break;
        case SelfAttn::Fused: break;
      }
      if (rc) {
        set_error(std::string("self-attention: the ") + kSelfAttnName[static_cast<int>(route.self)] +
                  " kernel does not take head size " + std::to_string(dh) + " at sequence length " + std::to_string(T));
        return 1;
      }
    }
    const QuantOuts next = enc_inputs(i + 1);
    if (route.ffn == EncFfn::Rows) {
      RowsFfnArgs k = rows_ffn_args(L.self, L.ffn, x0, R);
      k.map_a = map_attn_q, k.y_park = x1, k.z_out = x0;
      for (int j = 0; j < next.n; j++) k.zq[j] = reinterpret_cast<uint8_t*>(next.ptr[j]), k.zaq[j] = next.aq[j];
      k.n_zq = next.n;
      const double Rd = R, Ed = E, Fd = F;
      LaunchScope ls(c, "enc_wo_ffn_fused", 2.0 * Rd * (Ed * Ed + 2.0 * Ed * Fd),
                     Ed * Ed + 2.0 * Ed * Fd + Rd * Ed * (1.0 + 4.0 + 4.0 + k.n_zq));  // u8 in, residual, f32 out, u8 copies
      // (the y rows this variant parks in global memory and reads back are overhead, not algorithmic bytes)
      if (launch_rows_ffn(k, E, F, 128, fast, s)) {
        set_error("fused encoder FFN kernel launch failed");
        return 1;
      }
      continue;
    }
    {
      GemmCall g(&c, "enc_gemm_wo_res_ln", R, E, E, EPI_RES_LN);
      GemmProblem* p = g.add(attn_q, L.self.o);
      if (!p) return 1;
      p->residual = x0, p->ln_scale = L.self.ln.scale, p->ln_bias = L.self.ln.bias;
      p->out = x1;
      padd(p, qa[0], L.ffn.w1.aq);
      if (g.launch()) return 1;
    }
    {
      GemmCall g(&c, "enc_gemm_ffn1_relu_quant", R, F, E, EPI_QUANT);
      GemmProblem* p = g.add(qa[0], L.ffn.w1);
      if (!p) return 1;
      p->relu = 1;
      padd(p, ffn_q, L.ffn.w2.aq);
      if (g.launch()) return 1;
    }
    {
      GemmCall g(&c, "enc_gemm_ffn2_res_ln", R, E, F, EPI_RES_LN);
      GemmProblem* p = g.add(ffn_q, L.ffn.w2);
      if (!p) return 1;
      p->residual = x1, p->ln_scale = L.ffn.ln.scale, p->ln_bias = L.ffn.ln.bias;
      p->out = x0;
      for (int j = 0; j < next.n; j++) padd(p, next.ptr[j], next.aq[j]);
      if (g.launch()) return 1;
    }
  }
  if (Le == 0) {  // degenerate: quantize the embedding for the decoder's K/V projections
    const QuantOuts q = enc_inputs(0);
    LaunchScope ls(c, "quantize", 0, (4.0 + q.n) * R * E);
    launch_quantize(x0, static_cast<size_t>(R) * E, q, s);
  }
  if (a.encoder_out) {
    SB_CUDA(cudaMemcpyAsync(a.encoder_out, x0, 4ul * R * E, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * R * E;
  }
  return 0;
}

// Cross-attention K/V for the cached kernel, projected once here (the recompute kernels read the u8 encoder output).
int Pass::prepare_cross() {
  for (int l = 0; l < Ld && route.cross == Cross::Cached; l++) {
    GemmCall g(&c, "dec_gemm_cross_kv_f32", R, E, E, EPI_F32, 2);
    GemmProblem* pk = g.add(qa[2 * l], m.dec[l].ctx.k);
    GemmProblem* pv = g.add(qa[2 * l + 1], m.dec[l].ctx.v);
    if (!pk || !pv) return 1;
    pk->out = Kc[l], pv->out = Vc[l];
    pk->ldo = pv->ldo = E;
    if (g.launch()) return 1;
  }
  return 0;
}

// The output layer's columns: the model's, or the shortlist's gathered once per batch with what the route reads.
int Pass::prepare_output() {
  if (a.forced && !a.device_io) {
    SB_CUDA(cudaMemcpyAsync(d_forced, a.forced, 4ul * max_steps * B, cudaMemcpyHostToDevice, s));
    c.h2d_bytes += 4ul * max_steps * B;
  }
  if (d_keys && !a.device_io) {
    SB_CUDA(cudaMemcpyAsync(d_keys, a.keys, 8ul * B, cudaMemcpyHostToDevice, s));
    c.h2d_bytes += 8ul * B;
  }
  if (lazy_sl) {
    // the encoder and the cross K/V projections are already queued: build the candidate set meanwhile
    const uint32_t* words = nullptr;
    size_t n = 0;
    if (a.shortlist_cb(a.shortlist_user, &words, &n)) return 1;
    if (n == 0 || n % 8 != 0 || n > static_cast<size_t>(m.V)) {
      set_error("shortlist size must be a positive multiple of 8 no larger than the vocabulary");
      return 1;
    }
    a.shortlist = words, a.n_shortlist = n;
    Nout = static_cast<int>(n);
  }
  if (use_sl) {
    if (!a.device_io) {
      SB_CUDA(cudaMemcpyAsync(d_sl, a.shortlist, 4ul * Nout, cudaMemcpyHostToDevice, s));
      c.h2d_bytes += 4ul * Nout;
    }
    // SelectColumnsB + bias gather, once per batch (qmm/Intgemm.inl.cc:49-66)
    out.N = Nout;
    {
      LaunchScope ls(c, "gather_rows", 0, 2.0 * Nout * E);
      launch_gather_rows(m.vocab.w, m.vocab.pb, m.vocab.c127, d_sl, Nout, E, out.w, out.pb, out.c127, s);
    }
    if (route.out == Out::Argmax) {
      LaunchScope ls(c, "out_bounds", 0, (out.digits ? 140.0 : 8.0) * Nout);
      launch_out_tables(out, nullptr, s);
      if (out_maps(c, out, E)) return 1;
    }
    // the scores GEMM reads the weights alone: no table
    if (route.out == Out::Scores && c.make_map(&out.map_w, out.w, out.N, E, kOutBN)) return 1;
  }
  return 0;
}

// One decoder step over the M decoder rows: the decoder layers and the output projection with the greedy choice, or
// with beam search the candidates of every live slot and each sentence's merge.
int Pass::decode_step(int step) {
  const bool beam = a.beam > 0;
  float* d_align = d_align_all ? d_align_all + static_cast<size_t>(step) * M * T : nullptr;
  for (int l = 0; l < Ld; l++) {
    const DecLayerW& L = m.dec[l];
    const bool last = (l + 1 == Ld);
    {  // SSRU cell + query projection in one row-tile kernel (Modules.cc:190-235, 291)
      DecSsruArgs k{};
      k.map_xf = l == 0 ? map_xq[0] : map_zq[0];
      k.map_xw = l == 0 ? map_xq[1] : map_zq[1];
      k.map_wf = L.rnn_wf.map128, k.map_w = L.rnn_w.map128, k.map_wq = L.ctx.q.map128;
      k.pb_f = L.rnn_wf.pb, k.pb_w = L.rnn_w.pb, k.pb_q = L.ctx.q.pb;
      k.um_f = L.rnn_wf.um, k.um_w = L.rnn_w.um, k.um_q = L.ctx.q.um;
      k.aq_q = L.ctx.q.aq;
      k.x = l == 0 ? xd : zb, k.state = state[l];
      if (l == 0 && step > 0 && !beam) {  // close the previous step and embed its words in this kernel's front
        k.embed = 1, k.prev_step = step - 1;
        k.best = best, k.shortlist = d_sl, k.forced = d_forced, k.step_tokens = d_steps;
        k.done = done, k.tgt_len = tgt_len, k.n_done = counters, k.eos_id = m.eos_id;
        k.emb_q = m.emb_q, k.inv_qm = m.inv_qm, k.sqrt_e = m.sqrt_e, k.pos0 = m.pos;
        k.aq_xf = L.rnn_wf.aq, k.aq_xw = L.rnn_w.aq;
      }
      k.ln_scale = L.rnn_ln.scale, k.ln_bias = L.rnn_ln.bias, k.eps = 1e-6f;
      k.h_out = hb, k.q_out = qd, k.M = M;
      const double Bd = M, Ed = E;
      LaunchScope ls(c, "dec_ssru_q_fused", 2.0 * Bd * 3.0 * Ed * Ed, 3.0 * Ed * Ed + Bd * Ed * (2.0 + 4.0 * 5.0));
      if (launch_dec_ssru(k, E, fast, s)) {
        set_error("fused SSRU kernel: unsupported embedding size " + std::to_string(E));
        return 1;
      }
    }
    if (beam) {  // K queries per sentence against its cached K/V, as the scoring pass runs them
      if (cross_attention_mq(l, K, last ? d_align : nullptr, "beam_cross_attention", "beam")) return 1;
    } else if (route.cross != Cross::Cached) {
      CrossRcArgs k{};
      k.map_ak = mapK[l], k.map_av = mapV[l];
      k.map_wk = L.ctx.k.map128, k.map_wv = L.ctx.v.map128;
      k.pb_k = L.ctx.k.pb, k.pb_v = L.ctx.v.pb;
      k.um_k = L.ctx.k.um, k.um_v = L.ctx.v.um;
      k.q = qd, k.lengths = d_lengths, k.B = B, k.T = T;
      k.dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
      k.qo = qouts();
      qadd(k.qo, caq, L.ctx.o.aq);
      k.attn_head0 = last ? d_align : nullptr;
      const double Bd = B, Ed = E;
      const bool rcl = route.cross == Cross::Rcl;
      LaunchScope ls(c, "dec_cross_attention_rc", 2.0 * (rcl ? src_tokens : Bd * (T > 32 ? 64.0 : 32.0)) * Ed * 2.0 * Ed,
                     2.0 * src_tokens * Ed + 2.0 * Ed * Ed + 5.0 * Bd * Ed);  // valid keys only
      if (rcl ? launch_cross_attention_rcl(k, c.num_sms, s) : launch_cross_attention_rc(k, c.num_sms, fast, s)) {
        set_error("recompute cross-attention launch failed");
        return 1;
      }
    } else {
      QuantOuts q = qouts();
      qadd(q, caq, L.ctx.o.aq);
      LaunchScope ls(c, "dec_cross_attention", 0, 8.0 * src_tokens * E + 5.0 * B * E);
      if (launch_cross_attention(mapK[l], mapV[l], qd, d_lengths, B, T, H, dh, c.num_sms, q,
                                 last ? d_align : nullptr, s)) {
        set_error("cross-attention: no kernel for " + std::to_string(H) + " heads of " + std::to_string(dh) +
                  " over " + std::to_string(T) + " source tokens");
        return 1;
      }
    }
    if (wo_ffn(l, zb, zq[0], zq[1], "dec_wo_ffn_fused")) return 1;
  }
  // output projection (+ shortlist) and greedy choice (Transformer.cc:176-182, 279-339)
  if (route.out == Out::Logits || route.out == Out::TopK) {
    GemmCall g(&c, "dec_gemm_out_logits", B, Nout, E, EPI_F32);
    GemmProblem* p = g.add(oq, out.w, out.pb, out.um);
    if (!p) return 1;
    p->out = d_logits, p->ldo = Nout;
    if (g.launch()) return 1;
    if (route.out == Out::Logits) {
      LaunchScope ls(c, "argmax_rows", 0, 4.0 * B * Nout);
      launch_argmax_rows(d_logits, B, Nout, best, s);
    }
    if (a.logits) {
      SB_CUDA(cudaMemcpyAsync(a.logits + static_cast<size_t>(step) * B * Nout, d_logits, 4ul * B * Nout,
                              cudaMemcpyDeviceToHost, s));
      c.d2h_bytes += 4ul * B * Nout;
    }
    if ((a.scores || a.sample) && route.out == Out::Logits) {
      LaunchScope ls(c, "score_rows", 0, 4.0 * B * Nout + 8.0 * B * ((Nout + kScoreStrip - 1) / kScoreStrip));
      launch_score_rows(d_logits, B, Nout, partials, a.sample ? a.inv_t : 1.0f, s);
    }
  } else if (route.out == Out::Scores) {
    if (scores_gemm(map_oq, M, "dec_gemm_out_scores")) return 1;
  } else {
    const double Md = B, Nd = Nout, Kd = E;
    LaunchScope ls(c, "dec_gemm_out_argmax", 2.0 * Md * Nd * Kd, Md * Kd + Nd * Kd + 4.0 * Nd + 8.0 * Md);
    if (launch_out_argmax(out, map_oq, fast, B, E, best, c.num_sms, s)) {
      set_error("output GEMM: unsupported K " + std::to_string(E));
      return 1;
    }
  }
  if (beam) {
    BeamStepArgs k{};
    k.s = score_step_args(M, oq, nullptr, step, nullptr);
    k.beam = K, k.n_sent = B, k.step = step, k.last_step = max_steps - 1;
    k.cand = cand, k.cum = cum, k.width = width, k.rec = d_rec, k.fin = d_fin, k.n_done = counters;
    for (int l = 0; l < Ld; l++) k.state_cur[l] = state[l], k.state_nxt[l] = state_nx[l];
    k.Ld = Ld, k.E = E, k.eos_id = m.eos_id;
    k.emb_q = m.emb_q, k.inv_qm = m.inv_qm, k.sqrt_e = m.sqrt_e, k.pos0 = m.pos, k.x = xd;
    k.q = qouts();
    qadd(k.q, xq[0], m.dec[0].rnn_wf.aq), qadd(k.q, xq[1], m.dec[0].rnn_w.aq);
    const double Md = M, strips = (Nout + kScoreStrip - 1) / kScoreStrip;
    {  // the K strips of largest maximum are re-evaluated: 64 K weight rows and the row's operand
      LaunchScope ls(c, "beam_topk", 0, 8.0 * Md * strips * 2.0 + 8.0 * Md * K + 65.0 * K * E * Md);
      if (launch_beam_topk(k, s)) {
        set_error("beam search: candidate kernel launch failed");
        return 1;
      }
    }
    {
      LaunchScope ls(c, "beam_merge", 0, 8.0 * Md * K + 16.0 * Md + Md * E * (8.0 * Ld + 4.0 + 2.0 + 1.0));
      if (launch_beam_merge(k, s)) {
        set_error("beam search: merge kernel launch failed");
        return 1;
      }
    }
    for (int l = 0; l < Ld; l++) std::swap(state[l], state_nx[l]);
    return 0;
  }
  if (a.scores || a.sample) {
    ScoreStepArgs k = score_step_args(B, oq, d_forced, step, d_scores);
    k.inv_t = a.inv_t, k.seed = a.seed, k.keys = d_keys;
    const double strips = (Nout + kScoreStrip - 1) / kScoreStrip;
    if (route.out == Out::TopK) {
      // the row's logits, read twice (the first digit's histogram, then the columns it stages)
      LaunchScope ls(c, "topk_sample", 0, 8.0 * B * Nout + 24.0 * B);
      if (launch_topk_sample(k, a.top_k, s)) {
        set_error("top-k sampling: step kernel launch failed");
        return 1;
      }
    } else if (a.sample) {
      // the chosen strip's 64 columns are re-evaluated: 64 weight rows and the row's operand (or 64 tap logits)
      LaunchScope ls(c, "sample_step", 0, 8.0 * B * strips + 24.0 * B + (k.logits ? 256.0 : 65.0 * E) * B);
      if (launch_sample_step(k, s)) {
        set_error("sampling: step kernel launch failed");
        return 1;
      }
    } else {
      LaunchScope ls(c, "score_step", 0, 8.0 * B * strips + 16.0 * B + (a.forced ? 2.0 * B * E : 0.0));
      if (launch_score_step(k, s)) {
        set_error("token scores: step kernel launch failed");
        return 1;
      }
    }
  }
  return 0;
}

// Model.cc:161: the loop stops once every sentence has produced EOS.  Every second step the done-counter is copied to a
// pinned slot behind an event and the host looks at the previous copy, so the stream always holds a few queued steps
// and is never drained (extra steps only produce discarded tokens); the steps in between stay chained by programmatic
// dependent launch.
int Pass::poll_done(int step, bool* all_done) {
  if ((step & 1) == 1) {
    constexpr int kSlots = 8;
    const int poll = step >> 1;
    SB_CUDA(cudaMemcpyAsync(&c.done_slots[poll % kSlots], counters, 4, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaEventRecord(c.done_events[poll % kSlots], s));
    c.d2h_bytes += 4;
    if (poll >= 1) {
      const int old = (poll - 1) % kSlots;
      SB_CUDA(cudaEventSynchronize(c.done_events[old]));
      *all_done = c.done_slots[old] >= B;
    }
  }
  return 0;
}

// The decode loop (Model.cc:111-185) over the M decoder rows with its early exit, then the result copies: greedy
// decoding closes its last step with one more kernel and returns the step matrix, lengths and scores; beam search
// (DESIGN §4.4d) returns the step records and finished hypotheses from which the host rebuilds and ranks each
// sentence's hypotheses.
int Pass::decode() {
  const bool beam = a.beam > 0;
  for (int l = 0; l < Ld; l++) SB_CUDA(cudaMemsetAsync(state[l], 0, 4ul * M * E, s));  // Decoder::start_states
  SB_CUDA(cudaMemsetAsync(best, 0, 8ul * M, s));
  if (beam) {
    SB_CUDA(cudaMemsetAsync(cum, 0, 4ul * M, s));
    SB_CUDA(cudaMemsetAsync(width, K, B, s));
  } else {
    SB_CUDA(cudaMemsetAsync(done, 0, B, s));
    SB_CUDA(cudaMemsetAsync(tgt_len, 0, 4ul * B, s));
  }
  SB_CUDA(cudaMemsetAsync(counters, 0, 256, s));

  // step 0 input of every row: zero embedding + position-0 signal (Transformer.cc:133-160)
  QuantOuts q = qouts();
  qadd(q, xq[0], m.dec[0].rnn_wf.aq), qadd(q, xq[1], m.dec[0].rnn_w.aq);
  {
    LaunchScope ls(c, "dec_embed0", 0, 6.0 * M * E);
    launch_embed(nullptr, m.emb_q, m.inv_qm, m.sqrt_e, m.pos, M, 1, E, 0, 1, xd, q, s);
  }

  int executed = 0;
  for (int step = 0; step < max_steps; step++) {
    if (decode_step(step)) return 1;
    // Greedy: the step's bookkeeping (argmax -> word, record(), EOS flags) and the next step's input embedding are done
    // by the FRONT of the next step's first kernel (dec_ssru_kernel with embed set); the last executed step is closed by
    // the stand-alone kernel after the loop.
    executed = step + 1;
    bool all_done = false;
    if (poll_done(step, &all_done)) return 1;
    if (all_done) break;
  }

  // ---- results
  if (beam) {
    SB_CUDA(cudaMemcpyAsync(a.beam_steps, d_rec, sizeof(BeamRec) * executed * M, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaMemcpyAsync(a.beam_finished, d_fin, sizeof(BeamFin) * M, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += sizeof(BeamRec) * executed * M + sizeof(BeamFin) * M;
    a.steps = static_cast<size_t>(executed);
  } else {
    {
      LaunchScope ls(c, "dec_finalize_embed", 0, 7.0 * B * E + 20.0 * B);
      launch_finalize_step(best, d_sl, d_forced, executed - 1, d_steps, done, tgt_len, counters, m.eos_id, m.emb_q, m.inv_qm,
                           m.sqrt_e, m.pos, B, E, xd, q, s);
    }
    std::vector<uint32_t> lens(B);
    SB_CUDA(cudaMemcpyAsync(&c.done_slots[0], counters, 4, cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaMemcpyAsync(lens.data(), tgt_len, 4ul * B, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4 + 4ul * B;
    SB_CUDA(cudaStreamSynchronize(s));
    if (a.target_lengths) memcpy(a.target_lengths, lens.data(), 4ul * B);
    uint64_t total = 0;
    uint32_t longest = 0;
    for (uint32_t n : lens) total += n, longest = std::max(longest, n);
    a.target_tokens = total;
    // steps the reference would have run: up to the step where the last sentence finished
    a.steps = c.done_slots[0] >= B ? longest : static_cast<size_t>(executed);
    if (!a.device_io && a.scores) {
      SB_CUDA(cudaMemcpyAsync(a.scores, d_scores, 4ul * executed * B, cudaMemcpyDeviceToHost, s));
      c.d2h_bytes += 4ul * executed * B;
    }
    if (!a.device_io && a.step_tokens) {
      SB_CUDA(cudaMemcpyAsync(a.step_tokens, d_steps, 4ul * executed * B, cudaMemcpyDeviceToHost, s));
      c.d2h_bytes += 4ul * executed * B;
    }
    if (!a.device_io && a.sentence_tokens) {
      if (a.row_stride < static_cast<size_t>(executed)) {
        set_error("sentence_tokens: row_stride smaller than the number of decode steps");
        return 1;
      }
      // one row per sentence: the host then copies each sentence's recorded prefix without striding through the matrix
      {
        LaunchScope ls(c, "transpose_steps", 0, 8.0 * executed * B);
        launch_transpose_u32(d_steps, executed, B, d_rows, executed, s);
      }
      SB_CUDA(cudaMemcpy2DAsync(a.sentence_tokens, 4ul * a.row_stride, d_rows, 4ul * executed, 4ul * executed, B,
                                cudaMemcpyDeviceToHost, s));
      c.d2h_bytes += 4ul * executed * B;
    }
  }
  if (d_align_all) {
    SB_CUDA(cudaMemcpyAsync(a.alignment, d_align_all, 4ul * executed * M * T, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * executed * M * T;
  }
  SB_CUDA(cudaStreamSynchronize(s));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(std::string(beam ? "beam search failed: " : "forward failed: ") + cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

// The scoring pass (DESIGN §4.4c): every decoder input is known, so each layer runs over all M = B * Tt rows at once --
// one GEMM for the SSRU's two projections, the scan that is left sequential, one GEMM for Wq, the multi-query
// cross-attention, the Wo/FFN row-tile kernel of the step path -- and the output layer scores the rows in chunks.
// Row (b, j) sees exactly the operands decode step j sees under teacher forcing, so its score is the same bits.
int Pass::score() {
  SB_CUDA(cudaMemcpyAsync(d_tgt, a.targets, 4ul * M, cudaMemcpyHostToDevice, s));
  c.h2d_bytes += 4ul * M;
  const double Md = M, Ed = E;
  {  // decoder inputs: zero embedding at j = 0, then the previous target word, each + the position-0 signal (quirk Q1)
    QuantOuts q = qouts();
    qadd(q, xq[0], m.dec[0].rnn_wf.aq), qadd(q, xq[1], m.dec[0].rnn_w.aq);
    LaunchScope ls(c, "score_embed", 0, Md * 4.0 + Md * Ed * (1.0 + 4.0 + 4.0 + 2.0));
    launch_embed(d_tgt, m.emb_q, m.inv_qm, m.sqrt_e, m.pos, M, Tt, E, 0, 0, xd, q, s, 1);
  }
  for (int l = 0; l < Ld; l++) {
    const DecLayerW& L = m.dec[l];
    const bool last = (l + 1 == Ld);
    {  // Wf x + bf and W x of every row (Modules.cc:190-235)
      GemmCall g(&c, "score_gemm_ssru_f32", M, E, E, EPI_F32, 2);
      GemmProblem* pf = g.add(xq[0], L.rnn_wf);
      GemmProblem* pw = g.add(xq[1], L.rnn_w);
      if (!pf || !pw) return 1;
      pf->out = Fb, pw->out = Wx;
      pf->ldo = pw->ldo = E;
      if (g.launch()) return 1;
    }
    {
      DecSsruScanArgs k{};
      k.f = Fb, k.wx = Wx, k.x = xd;
      k.ln_scale = L.rnn_ln.scale, k.ln_bias = L.rnn_ln.bias, k.eps = 1e-6f;
      k.aq_q = L.ctx.q.aq, k.h_out = hb, k.hq = reinterpret_cast<uint8_t*>(hq);
      k.B = B, k.T = Tt;
      LaunchScope ls(c, "score_ssru_scan", 0, Md * Ed * (3.0 * 4.0 + 4.0 + 1.0));
      if (launch_dec_ssru_scan(k, E, s)) {
        set_error("SSRU scan kernel: unsupported embedding size " + std::to_string(E));
        return 1;
      }
    }
    {
      GemmCall g(&c, "score_gemm_q_f32", M, E, E, EPI_F32);
      GemmProblem* p = g.add(hq, L.ctx.q);
      if (!p) return 1;
      p->out = qd, p->ldo = E;
      if (g.launch()) return 1;
    }
    // Tt queries per sentence against its cached K/V; head 0 of the last layer is the alignment
    if (cross_attention_mq(l, Tt, last ? d_align_all : nullptr, "score_cross_attention", "scoring")) return 1;
    if (wo_ffn(l, xd, xq[0], xq[1], "score_wo_ffn_fused")) return 1;  // the step path's row-tile kernel over M rows
  }
  // output layer in row chunks, so that the strip partials [ceil(N / 64)][rows] stay bounded; each chunk is one "step"
  // of score_step with the targets as the forced words
  const double strips = (Nout + kScoreStrip - 1) / kScoreStrip;
  for (int r0 = 0; r0 < M; r0 += kScoreChunk) {
    const int rows = std::min(kScoreChunk, M - r0);
    CUtensorMap map;
    if (c.make_map(&map, oq + static_cast<size_t>(r0) * E, rows, E, kBM)) return 1;
    SB_CUDA(cudaMemsetAsync(best, 0, 8ul * rows, s));
    if (scores_gemm(map, rows, "score_gemm_out_scores")) return 1;
    const ScoreStepArgs k = score_step_args(rows, oq + static_cast<size_t>(r0) * E, d_tgt + r0, 0, d_scores + r0);
    LaunchScope ls(c, "score_step", 0, 8.0 * rows * strips + 16.0 * rows + 2.0 * rows * E);
    if (launch_score_step(k, s)) {
      set_error("token scores: step kernel launch failed");
      return 1;
    }
  }
  SB_CUDA(cudaMemcpyAsync(a.scores, d_scores, 4ul * M, cudaMemcpyDeviceToHost, s));
  c.d2h_bytes += 4ul * M;
  if (d_align_all) {
    SB_CUDA(cudaMemcpyAsync(a.alignment, d_align_all, 4ul * M * T, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * M * T;
  }
  SB_CUDA(cudaStreamSynchronize(s));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(std::string("scoring pass failed: ") + cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

// One call on context c (`name` prefixes its errors): an empty request does nothing; otherwise the encoder and the
// output layer's set-up, then `decoder` (Pass::decode or Pass::score).
int run_pass(Model& m, Context& c, ForwardArgs& a, const char* name, bool empty, int (Pass::*decoder)()) {
  std::lock_guard<std::recursive_mutex> ctx_lock(c.mu);
  if (c.device != m.ctx->device) {
    set_error(std::string(name) + ": the lane context and the model live on different devices");
    return 1;
  }
  SB_CUDA(cudaSetDevice(c.device));
  if (empty) return 0;
  Pass p{m, c, a, c.stream};
  return p.plan() || p.encode() || p.prepare_cross() || p.prepare_output() || (p.*decoder)() ? 1 : 0;
}

}  // namespace

int model_forward(Model& m, ForwardArgs& a) { return model_forward_on(m, *m.ctx, a); }

int model_forward_on(Model& m, Context& c, ForwardArgs& a) {
  a.steps = 0;
  a.target_tokens = 0;
  return run_pass(m, c, a, "model_forward", a.B == 0 || a.T == 0, &Pass::decode);
}

int model_beam_on(Model& m, Context& c, ForwardArgs& a) {
  a.steps = 0;
  a.target_tokens = 0;
  if (a.beam < 1 || a.beam > kMaxBeam || a.beam_steps == nullptr || a.beam_finished == nullptr || a.targets || a.forced ||
      a.sample || a.logits || a.scores || a.device_io) {
    set_error("model_beam: a beam of 1 .. 8, host buffers for the records, and none of targets, forced, sampling, "
              "logits, scores or device_io");
    return 1;
  }
  return run_pass(m, c, a, "model_beam", a.B == 0 || a.T == 0, &Pass::decode);
}

int model_score_on(Model& m, Context& c, ForwardArgs& a) {
  if (a.targets == nullptr || a.scores == nullptr || a.forced || a.sample || a.logits || a.device_io) {
    set_error("model_score: targets and scores on host buffers, and none of forced, sampling, logits or device_io");
    return 1;
  }
  return run_pass(m, c, a, "model_score", a.B == 0 || a.T == 0 || a.target_T == 0, &Pass::score);
}

}  // namespace sb
