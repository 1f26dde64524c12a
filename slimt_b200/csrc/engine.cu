// See engine.cuh.
#include "engine.cuh"

#include <math.h>
#include <stdio.h>
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
  arena_used = 0;
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
  auto upload = [this](const void* src, size_t nbytes, void** dst) -> int {
    SB_CUDA(cudaMalloc(dst, nbytes));
    owned.push_back(*dst);
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
    // bound filter of the fused output GEMM: 127 * colsum per column, per-chunk dmax, rounding slack eta
    std::vector<int32_t> c127(V);
    for (int n = 0; n < V; n++) {
      int32_t cs = 0;
      for (int k = 0; k < E; k++) cs += req[static_cast<size_t>(n) * E + k];
      c127[n] = 127 * cs;
    }
    if (upload(c127.data(), 4ul * V, reinterpret_cast<void**>(&out.c127))) return 1;
    SB_CUDA(cudaMalloc(&out.dmax, 4ul * ((V + 31) / 32)));
    owned.push_back(out.dmax);
    launch_out_bounds(out.c127, out.pb, out.um, V, out.dmax, c->stream);
    SB_CUDA(cudaMalloc(&out.ipb6, 4ul * ((V + 255) / 256 * 256)));
    owned.push_back(out.ipb6);
    launch_out_ipb(out.c127, out.pb, out.um, V, out.ipb6, c->stream);
    {
      const size_t vpad = static_cast<size_t>((V + 255) / 256 * 256);
      int* d_flag = nullptr;
      SB_CUDA(cudaMalloc(&out.ext, vpad * 128));
      owned.push_back(out.ext);
      SB_CUDA(cudaMalloc(&out.dshift, vpad * 4));
      owned.push_back(out.dshift);
      SB_CUDA(cudaMalloc(&d_flag, 4));
      SB_CUDA(cudaMemsetAsync(d_flag, 0, 4, c->stream));
      launch_out_ext(out.c127, out.pb, out.um, V, out.ext, out.dshift, d_flag, c->stream);
      int flag = 0;
      SB_CUDA(cudaMemcpyAsync(&flag, d_flag, 4, cudaMemcpyDeviceToHost, c->stream));
      SB_CUDA(cudaStreamSynchronize(c->stream));
      SB_CUDA(cudaFree(d_flag));
      out.ext_ok = flag == 0;
      if (ctx->make_map(&out.map_ext, out.ext, vpad, 128, 256)) return 1;
    }
    SB_CUDA(cudaStreamSynchronize(c->stream));
    std::vector<float> pbh(V);
    SB_CUDA(cudaMemcpy(pbh.data(), out.pb, 4ul * V, cudaMemcpyDeviceToHost));
    double pbabs = 0;
    for (float v : pbh) pbabs = std::max(pbabs, static_cast<double>(fabsf(v)));
    const double vmax = static_cast<double>(E) * 254.0 * 128.0;
    out.eta = static_cast<float>((2.0 * vmax * out.um + pbabs) * ldexp(1.0, -22));
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
  double extra_bytes = 0;  // epilogue traffic beyond A, W and the primary output (residual reads, int8 copies)
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
      if (epi == EPI_ARGMAX) out_bytes += 8 * M;
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
  const size_t need = M * K * 5 + N * K + N * 8 + Nout * K + Nout * 8 + n_idx * 4 + M * Nout * 8 + 16 * 256;
  if (c.reserve(need)) return 1;
  float* dx = c.take<float>(M * K);
  int8_t* dqa = c.take<int8_t>(M * K);
  int8_t* dW = c.take<int8_t>(N * K);
  float* dpb = c.take<float>(N);
  float* dy = c.take<float>(M * Nout);
  int32_t* dacc = c.take<int32_t>(M * Nout);
  cudaStream_t s = c.stream;
  SB_CUDA(cudaMemcpyAsync(dx, x, M * K * 4, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(dW, W, N * K, cudaMemcpyHostToDevice, s));
  SB_CUDA(cudaMemcpyAsync(dpb, pb.data(), N * 4, cudaMemcpyHostToDevice, s));
  c.h2d_bytes += M * K * 4 + N * K + N * 8;
  const int8_t* Wuse = dW;
  const float* pbuse = dpb;
  if (indices) {
    uint32_t* didx = c.take<uint32_t>(n_idx);
    int8_t* dWs = c.take<int8_t>(n_idx * K);
    float* dpbs = c.take<float>(n_idx);
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

// ------------------------------------------------------------------ Model::forward
int model_forward(Model& m, ForwardArgs& a) { return model_forward_on(m, *m.ctx, a); }

int model_forward_on(Model& m, Context& c, ForwardArgs& a) {
  std::lock_guard<std::recursive_mutex> ctx_lock(c.mu);
  if (c.device != m.ctx->device) {
    set_error("model_forward: the lane context and the model live on different devices");
    return 1;
  }
  SB_CUDA(cudaSetDevice(c.device));
  cudaStream_t s = c.stream;
  const int B = static_cast<int>(a.B), T = static_cast<int>(a.T), E = m.E, F = m.F, H = m.H, dh = m.dh;
  const int R = B * T;
  const int Le = static_cast<int>(m.enc.size()), Ld = static_cast<int>(m.dec.size());
  a.steps = 0;
  a.target_tokens = 0;
  if (B == 0 || T == 0) return 0;
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
  const int max_steps = forward_max_steps(a.limit_factor, a.T);
  double src_tokens = static_cast<double>(R);  // cross-attention reads only valid keys; exact count when lengths are on the host
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
  const bool lazy_sl = a.shortlist == nullptr && a.shortlist_cb != nullptr && !a.device_io;
  const bool use_sl = lazy_sl || (a.shortlist != nullptr && a.n_shortlist > 0);
  int Nout = use_sl && !lazy_sl ? static_cast<int>(a.n_shortlist) : m.V;  // lazy: upper bound until the callback ran
  if (use_sl && !lazy_sl && a.n_shortlist % 8 != 0) {
    set_error("shortlist size must be a multiple of 8");
    return 1;
  }

  // ---- workspace
  size_t need = 0;
  auto acc = [&need](size_t bytes) { need += (bytes + 255) & ~size_t(255); };
  acc(4ul * R), acc(4ul * B);                                   // tokens, lengths
  acc(4ul * R * E), acc(4ul * R * E);                           // x0, x1
  for (int i = 0; i < 4; i++) acc(1ul * R * E);                 // qa[4]
  for (int i = 0; i < 3; i++) acc(4ul * R * E);                 // Q K V
  acc(1ul * R * E), acc(1ul * R * F);                           // attn_q, ffn_q
  for (int i = 0; i < 2 * Ld; i++) acc(4ul * R * E);            // cross K/V caches
  for (int i = 0; i < 9 + Ld; i++) acc(4ul * B * E);            // decode f32 rows
  for (int i = 0; i < 8; i++) acc(1ul * B * E);                 // decode int8 rows
  acc(1ul * B * F);
  acc(8ul * B), acc(B), acc(4ul * B), acc(256);                 // best, done, tgt_len, counters
  acc(4ul * max_steps * B);                        // step tokens
  if (a.forced) acc(4ul * max_steps * B);
  if (a.sentence_tokens) acc(4ul * max_steps * B);
  if (use_sl) acc(4ul * Nout), acc(1ul * Nout * E), acc(4ul * Nout), acc(4ul * Nout), acc(4ul * (Nout / 32 + 1)), acc(4ul * (Nout + 256)), acc(128ul * (Nout + 256)), acc(4ul * (Nout + 256)), acc(256);
  if (a.logits) acc(4ul * B * Nout);
  if (a.alignment) acc(4ul * max_steps * B * T);
  need += 64 * 256;
  if (c.reserve(need)) return 1;

  uint32_t* d_tokens = nullptr;
  uint32_t* d_lengths = nullptr;
  if (a.device_io) {
    d_tokens = const_cast<uint32_t*>(a.tokens);
    d_lengths = const_cast<uint32_t*>(a.lengths);
    c.take<uint32_t>(R), c.take<uint32_t>(B);
  } else {
    d_tokens = c.take<uint32_t>(R);
    d_lengths = c.take<uint32_t>(B);
    SB_CUDA(cudaMemcpyAsync(d_tokens, a.tokens, 4ul * R, cudaMemcpyHostToDevice, s));
    SB_CUDA(cudaMemcpyAsync(d_lengths, a.lengths, 4ul * B, cudaMemcpyHostToDevice, s));
    c.h2d_bytes += 4ul * R + 4ul * B;
  }
  float* x0 = c.take<float>(static_cast<size_t>(R) * E);
  float* x1 = c.take<float>(static_cast<size_t>(R) * E);
  int8_t* qa[4];
  for (auto& p : qa) p = c.take<int8_t>(static_cast<size_t>(R) * E);
  float* Qb = c.take<float>(static_cast<size_t>(R) * E);
  float* Kb = c.take<float>(static_cast<size_t>(R) * E);
  float* Vb = c.take<float>(static_cast<size_t>(R) * E);
  int8_t* attn_q = c.take<int8_t>(static_cast<size_t>(R) * E);
  int8_t* ffn_q = c.take<int8_t>(static_cast<size_t>(R) * F);
  std::vector<float*> Kc(Ld), Vc(Ld);
  std::vector<CUtensorMap> mapKc(Ld), mapVc(Ld);
  for (int l = 0; l < Ld; l++) {
    Kc[l] = c.take<float>(static_cast<size_t>(R) * E);
    Vc[l] = c.take<float>(static_cast<size_t>(R) * E);
    const uint32_t box_rows = static_cast<uint32_t>(cross_attention_box_rows(T));
    if (c.make_map_f32(&mapKc[l], Kc[l], R, E, box_rows) || c.make_map_f32(&mapVc[l], Vc[l], R, E, box_rows)) return 1;
  }

  CUtensorMap map_attn_q;  // u8 [R][E], box {128 B, 128 rows}: operand of the encoder's row-tile kernel
  if (c.make_map(&map_attn_q, attn_q, R, E, 128)) return 1;

  // SLIMT_B200_SELFATTN=split keeps the projections and the attention as separate kernels (parity cross-check);
  // =rowwise additionally takes the first-generation one-thread-per-query kernel instead of the tiled one
  const char* sa_env = getenv("SLIMT_B200_SELFATTN");
  // the tiled kernel's 64-query x 128-key tiles pay off from T > 64 (mixed lengths: 15.9 -> 8.5 ms per layer of a
  // 1M-word batch); at T <= 64 with head size 64 (base) half of every tile is idle and the row-wise kernel is faster
  // (666 vs 1149 us per layer at 4096 x 32); SLIMT_B200_SELFATTN=tiled forces the tiled kernel (parity cross-check)
  const bool sa_long = sa_env && strcmp(sa_env, "long") == 0;
  const bool attn_rowwise = (sa_env && strcmp(sa_env, "rowwise") == 0) ||
                            (T <= 64 && !(sa_env && (strcmp(sa_env, "tiled") == 0 || sa_long)));
  // The long kernel (self_attention_long.cu) takes what the tiled kernel cannot hold (T > 556 at head size 32, T > 400
  // at 64) and 257 .. 384 tokens, where its 32-row score block lets two or three blocks share an SM against the tiled
  // kernel's one: 16.5 vs 19.9 ms for the six layers of 455 x 288, 20.1 vs 22.3 ms at 341 x 384; at 256 x 512 the
  // tiled kernel's 64-row reuse wins, 29.3 vs 30.4 ms (B200, 1000 W; profiles/r4_long_bench.jsonl).  T <= 256 routes as
  // before.  SLIMT_B200_SELFATTN=long forces the long kernel (parity cross-check).
  const bool attn_long = sa_long || (!attn_rowwise && !(sa_env && strcmp(sa_env, "tiled") == 0) &&
                                     ((T > 256 && T <= 384) || !self_attention_tiled_supported(T, dh)));
  const bool attn_fused = enc_attention_supported(E, H, dh, T) &&
                          !(sa_env && (strcmp(sa_env, "split") == 0 || strcmp(sa_env, "rowwise") == 0 ||
                                       strcmp(sa_env, "tiled") == 0 || sa_long));
  CUtensorMap map_qa[3], map_qa32[3];
  if (attn_fused)
    for (int i = 0; i < 3; i++)
      if (c.make_map(&map_qa[i], qa[i], R, E, 128) || c.make_map(&map_qa32[i], qa[i], R, E, 32)) return 1;

  // debugging aid: SLIMT_B200_TRACE=<file> records the phase stamps of the row-tile kernels: the encoder's first FFN
  // launch (first tile of every CTA) and the two decoder kernels of layer 0 in decode step 3
  const char* trace_path = getenv("SLIMT_B200_TRACE");
  long long* trace_buf = nullptr;
  const size_t trace_n = static_cast<size_t>(c.num_sms) * kTraceSlots;
  if (trace_path) {
    SB_CUDA(cudaMallocManaged(&trace_buf, 5 * trace_n * sizeof(long long)));
    SB_CUDA(cudaMemsetAsync(trace_buf, 0, 5 * trace_n * sizeof(long long), s));
  }

  // ---- embedding (Model.cc:195-197)
  {
    QuantOuts q = qouts();
    if (Le > 0) {
      qadd(q, qa[0], m.enc[0].self.q.aq), qadd(q, qa[1], m.enc[0].self.k.aq), qadd(q, qa[2], m.enc[0].self.v.aq);
    }
    LaunchScope ls(c, "enc_embed", 0, (1.0 + 4.0 + q.n) * R * E);
    launch_embed(d_tokens, m.emb_q, m.inv_qm, m.sqrt_e, m.pos, R, T, E, 1, 0, x0, q, s);
  }

  // ---- encoder (Transformer.cc:57-69; EncoderLayer::forward Modules.cc:321-334)
  for (int i = 0; i < Le; i++) {
    const EncLayerW& L = m.enc[i];
    if (attn_fused) {
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
    {
      QuantOuts q = qouts();
      qadd(q, attn_q, L.self.o.aq);
      LaunchScope ls(c, "enc_self_attention", 0, 13.0 * R * E);
      const int rc = attn_long      ? launch_self_attention_long(Qb, Kb, Vb, d_lengths, B, T, H, dh, nullptr, q, s)
                     : attn_rowwise ? launch_self_attention(Qb, Kb, Vb, d_lengths, B, T, H, dh, nullptr, q, s)
                                    : launch_self_attention_tiled(Qb, Kb, Vb, d_lengths, B, T, H, dh, nullptr, q, s);
      if (rc) {
        set_error(std::string("self-attention: the ") + (attn_long ? "long" : attn_rowwise ? "row-wise" : "tiled") +
                  " kernel does not take head size " + std::to_string(dh) + " at sequence length " + std::to_string(T));
        return 1;
      }
    }
    }
    if (E == 256 && F == 1536) {
      // Wo + residual + LN, FFN1 + ReLU, FFN2 + residual + LN in one row-tile kernel, 128 rows per CTA
      RowsFfnArgs k{};
      k.map_a = map_attn_q;
      k.map_wo = L.self.o.map128, k.map_w1 = L.ffn.w1.map128, k.map_w2 = L.ffn.w2.map128;
      k.pb_o = L.self.o.pb, k.pb_1 = L.ffn.w1.pb, k.pb_2 = L.ffn.w2.pb;
      k.um_o = L.self.o.um, k.um_1 = L.ffn.w1.um, k.um_2 = L.ffn.w2.um;
      k.aq_1 = L.ffn.w1.aq, k.aq_2 = L.ffn.w2.aq;
      k.res = x0, k.y_park = x1, k.z_out = x0;
      k.ln1_scale = L.self.ln.scale, k.ln1_bias = L.self.ln.bias;
      k.ln2_scale = L.ffn.ln.scale, k.ln2_bias = L.ffn.ln.bias, k.eps = 1e-6f;
      if (i + 1 < Le) {
        const EncLayerW& Nx = m.enc[i + 1];
        k.zq[0] = reinterpret_cast<uint8_t*>(qa[0]), k.zaq[0] = Nx.self.q.aq;
        k.zq[1] = reinterpret_cast<uint8_t*>(qa[1]), k.zaq[1] = Nx.self.k.aq;
        k.zq[2] = reinterpret_cast<uint8_t*>(qa[2]), k.zaq[2] = Nx.self.v.aq;
        k.n_zq = 3;
      } else {
        for (int l = 0; l < Ld; l++) {
          k.zq[2 * l] = reinterpret_cast<uint8_t*>(qa[2 * l]), k.zaq[2 * l] = m.dec[l].ctx.k.aq;
          k.zq[2 * l + 1] = reinterpret_cast<uint8_t*>(qa[2 * l + 1]), k.zaq[2 * l + 1] = m.dec[l].ctx.v.aq;
        }
        k.n_zq = 2 * Ld;
      }
      k.M = R;
      if (trace_buf && i == 0) k.trace = trace_buf + 2 * trace_n;
      const double Rd = R, Ed = E, Fd = F;
      LaunchScope ls(c, "enc_wo_ffn_fused", 2.0 * Rd * (Ed * Ed + 2.0 * Ed * Fd),
                     Ed * Ed + 2.0 * Ed * Fd + Rd * Ed * (1.0 + 4.0 + 4.0 + k.n_zq));  // u8 in, residual, f32 out, u8 copies
      // (the y rows this variant parks in global memory and reads back are overhead, not algorithmic bytes)
      if (launch_rows_ffn(k, E, F, 128, c.fast, s)) {
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
      if (i + 1 < Le) {
        const EncLayerW& Nx = m.enc[i + 1];
        padd(p, qa[0], Nx.self.q.aq), padd(p, qa[1], Nx.self.k.aq), padd(p, qa[2], Nx.self.v.aq);
      } else {
        for (int l = 0; l < Ld; l++) padd(p, qa[2 * l], m.dec[l].ctx.k.aq), padd(p, qa[2 * l + 1], m.dec[l].ctx.v.aq);
      }
      if (g.launch()) return 1;
    }
  }
  if (Le == 0) {  // degenerate: quantize the embedding for the decoder's K/V projections
    QuantOuts q = qouts();
    for (int l = 0; l < Ld; l++) qadd(q, qa[2 * l], m.dec[l].ctx.k.aq), qadd(q, qa[2 * l + 1], m.dec[l].ctx.v.aq);
    LaunchScope ls(c, "quantize", 0, (4.0 + q.n) * R * E);
    launch_quantize(x0, static_cast<size_t>(R) * E, q, s);
  }
  if (a.encoder_out) {
    SB_CUDA(cudaMemcpyAsync(a.encoder_out, x0, 4ul * R * E, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * R * E;
  }

  // ---- cross-attention K/V.  The reference re-projects them every step (Modules.cc:244-249); so does the
  // recompute kernel (tensor cores, from the u8 encoder output); otherwise they are projected once and cached.
  // Small batches take the cached kernel: below ~4 k source tokens the recompute kernel has fewer sentence groups than
  // SMs and its launch is all latency (64 x 32: 8.6 us cached against 12.8 us recomputed per launch, 5.40 -> 5.13 ms per
  // batch; the two are bit-identical).  SLIMT_B200_CROSS = cached | rc overrides the choice (tests, A/B runs).
  const char* ca_env = getenv("SLIMT_B200_CROSS");
  const bool ca_force_rc = ca_env && strcmp(ca_env, "rc") == 0;
  const bool ca_cached = (ca_env && strcmp(ca_env, "cached") == 0) || (!ca_force_rc && static_cast<long>(B) * T <= 4096);
  // long sentences (65 .. 256 tokens) take the sentence-at-a-time recompute kernel (cross_attention_rcl.cu; bit-exact mode)
  const bool cross_rcl = !ca_cached && !c.fast && !cross_attention_rc_supported(E, H, dh, T) && cross_attention_rcl_supported(E, H, dh, T);
  const bool cross_rc = cross_rcl || (cross_attention_rc_supported(E, H, dh, T) && !ca_cached);
  std::vector<CUtensorMap> mapAk(Ld), mapAv(Ld);
  if (cross_rc) {
    for (int l = 0; l < Ld; l++)
      if (c.make_map(&mapAk[l], qa[2 * l], R, E, 32) || c.make_map(&mapAv[l], qa[2 * l + 1], R, E, 32)) return 1;
  }
  for (int l = 0; l < Ld && !cross_rc; l++) {
    GemmCall g(&c, "dec_gemm_cross_kv_f32", R, E, E, EPI_F32, 2);
    GemmProblem* pk = g.add(qa[2 * l], m.dec[l].ctx.k);
    GemmProblem* pv = g.add(qa[2 * l + 1], m.dec[l].ctx.v);
    if (!pk || !pv) return 1;
    pk->out = Kc[l], pv->out = Vc[l];
    pk->ldo = pv->ldo = E;
    if (g.launch()) return 1;
  }

  // ---- decoder state (Model.cc:111-185)
  float* xd = c.take<float>(static_cast<size_t>(B) * E);
  float* fb = c.take<float>(static_cast<size_t>(B) * E);
  float* wxb = c.take<float>(static_cast<size_t>(B) * E);
  float* hb = c.take<float>(static_cast<size_t>(B) * E);
  float* qd = c.take<float>(static_cast<size_t>(B) * E);
  float* yb = c.take<float>(static_cast<size_t>(B) * E);
  float* zb[2] = {c.take<float>(static_cast<size_t>(B) * E), c.take<float>(static_cast<size_t>(B) * E)};
  c.take<float>(static_cast<size_t>(B) * E);
  std::vector<float*> state(Ld);
  for (int l = 0; l < Ld; l++) state[l] = c.take<float>(static_cast<size_t>(B) * E);
  int8_t* xq[2] = {c.take<int8_t>(static_cast<size_t>(B) * E), c.take<int8_t>(static_cast<size_t>(B) * E)};
  int8_t* zq[2] = {c.take<int8_t>(static_cast<size_t>(B) * E), c.take<int8_t>(static_cast<size_t>(B) * E)};
  int8_t* hq = c.take<int8_t>(static_cast<size_t>(B) * E);
  int8_t* caq = c.take<int8_t>(static_cast<size_t>(B) * E);
  int8_t* yq = c.take<int8_t>(static_cast<size_t>(B) * E);
  int8_t* oq = c.take<int8_t>(static_cast<size_t>(B) * E);
  int8_t* fq = c.take<int8_t>(static_cast<size_t>(B) * F);
  unsigned long long* best = c.take<unsigned long long>(B);
  uint8_t* done = c.take<uint8_t>(B);
  uint32_t* tgt_len = c.take<uint32_t>(B);
  int* counters = c.take<int>(64);  // [0] n_done, [1] step counter, [2] ticket
  uint32_t* d_steps = nullptr;
  if (a.device_io) {
    d_steps = a.step_tokens;
    c.take<uint32_t>(static_cast<size_t>(max_steps) * B);
  } else {
    d_steps = c.take<uint32_t>(static_cast<size_t>(max_steps) * B);
  }
  const uint32_t* d_forced = nullptr;
  if (a.forced) {
    if (a.device_io) {
      d_forced = a.forced;
    } else {
      uint32_t* t = c.take<uint32_t>(static_cast<size_t>(max_steps) * B);
      SB_CUDA(cudaMemcpyAsync(t, a.forced, 4ul * max_steps * B, cudaMemcpyHostToDevice, s));
      c.h2d_bytes += 4ul * max_steps * B;
      d_forced = t;
    }
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
  const uint32_t* d_sl = nullptr;
  const int8_t* Wout = m.out.w;
  const float* pb_out = m.out.pb;
  const int32_t* c127_out = m.out.c127;
  const float* dmax_out = m.out.dmax;
  const int32_t* ipb6_out = m.out.ipb6;
  const int32_t* dshift_out = m.out.dshift;
  CUtensorMap map_ext = m.out.map_ext;
  static const bool out_legacy = [] {
    const char* e = getenv("SLIMT_B200_OUT");  // SLIMT_B200_OUT=legacy keeps gemm_out.cu (A/B measurements, cross-checks)
    return e && strcmp(e, "legacy") == 0;
  }();
  const bool out_ext = m.out.ext_ok && !out_legacy;
  if (use_sl) {
    if (a.device_io) {
      d_sl = a.shortlist;
      c.take<uint32_t>(Nout);
    } else {
      uint32_t* t = c.take<uint32_t>(Nout);
      SB_CUDA(cudaMemcpyAsync(t, a.shortlist, 4ul * Nout, cudaMemcpyHostToDevice, s));
      c.h2d_bytes += 4ul * Nout;
      d_sl = t;
    }
    // SelectColumnsB + bias gather, once per batch (qmm/Intgemm.inl.cc:49-66)
    int8_t* Ws = c.take<int8_t>(static_cast<size_t>(Nout) * E);
    float* pbs = c.take<float>(Nout);
    int32_t* cs = c.take<int32_t>(Nout);
    float* dms = c.take<float>(Nout / 32 + 1);
    {
      LaunchScope ls(c, "gather_rows", 0, 2.0 * Nout * E);
      launch_gather_rows(m.out.w, m.out.pb, m.out.c127, d_sl, Nout, E, Ws, pbs, cs, s);
    }
    {
      LaunchScope ls(c, "out_bounds", 0, 8.0 * Nout);
      launch_out_bounds(cs, pbs, m.out.um, Nout, dms, s);
    }
    int32_t* ips = c.take<int32_t>(static_cast<size_t>(Nout) + 256);
    uint8_t* exts = c.take<uint8_t>(128ul * (static_cast<size_t>(Nout) + 256));
    int32_t* dss = c.take<int32_t>(static_cast<size_t>(Nout) + 256);
    int* flag = c.take<int>(64);
    if (out_ext) {
      // a subset of columns whose offsets all fit the digits fits them too: the flag is not read back
      LaunchScope ls(c, "out_bounds", 0, 140.0 * Nout);
      launch_out_ext(cs, pbs, m.out.um, Nout, exts, dss, flag, s);
      if (c.make_map(&map_ext, exts, static_cast<uint64_t>((Nout + 255) / 256 * 256), 128, 256)) return 1;
    } else if (c.fast) {
      LaunchScope ls(c, "out_bounds", 0, 12.0 * Nout);
      launch_out_ipb(cs, pbs, m.out.um, Nout, ips, s);
    }
    Wout = Ws, pb_out = pbs, c127_out = cs, dmax_out = dms, ipb6_out = ips, dshift_out = dss;
  }
  CUtensorMap map_xq[2], map_zq[2], map_caq;  // u8 activation operands of the row-tile kernels, box {128 B, 32 rows}
  for (int i = 0; i < 2; i++) {
    if (c.make_map(&map_xq[i], xq[i], B, E, kRowTile) || c.make_map(&map_zq[i], zq[i], B, E, kRowTile)) return 1;
  }
  if (c.make_map(&map_caq, caq, B, E, kRowTile)) return 1;
  CUtensorMap map_oq, map_wout;
  if (c.make_map(&map_oq, oq, B, E, kBM) || c.make_map(&map_wout, Wout, Nout, E, 256)) return 1;
  float* d_logits = a.logits ? c.take<float>(static_cast<size_t>(B) * Nout) : nullptr;
  // head-0 probabilities of every step stay on the device and come back in one copy after the loop
  float* d_align_all = a.alignment ? c.take<float>(static_cast<size_t>(max_steps) * B * T) : nullptr;

  for (int l = 0; l < Ld; l++) SB_CUDA(cudaMemsetAsync(state[l], 0, 4ul * B * E, s));  // Decoder::start_states
  SB_CUDA(cudaMemsetAsync(best, 0, 8ul * B, s));
  SB_CUDA(cudaMemsetAsync(done, 0, B, s));
  SB_CUDA(cudaMemsetAsync(tgt_len, 0, 4ul * B, s));
  SB_CUDA(cudaMemsetAsync(counters, 0, 256, s));

  // step 0 input: zero embedding + position-0 signal (Transformer.cc:133-160)
  {
    QuantOuts q = qouts();
    qadd(q, xq[0], m.dec[0].rnn_wf.aq), qadd(q, xq[1], m.dec[0].rnn_w.aq);
    LaunchScope ls(c, "dec_embed0", 0, 6.0 * B * E);
    launch_embed(nullptr, m.emb_q, m.inv_qm, m.sqrt_e, m.pos, B, 1, E, 0, 1, xd, q, s);
  }

  int executed = 0;
  int host_done = 0;
  for (int step = 0; step < max_steps; step++) {
    float* d_align = d_align_all ? d_align_all + static_cast<size_t>(step) * B * T : nullptr;
    const float* in_f = xd;
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
        k.x = in_f, k.state = state[l];
        if (l == 0 && step > 0) {  // close the previous step and embed its words in this kernel's front
          k.embed = 1, k.prev_step = step - 1;
          k.best = best, k.shortlist = d_sl, k.forced = d_forced, k.step_tokens = d_steps;
          k.done = done, k.tgt_len = tgt_len, k.n_done = counters, k.eos_id = m.eos_id;
          k.emb_q = m.emb_q, k.inv_qm = m.inv_qm, k.sqrt_e = m.sqrt_e, k.pos0 = m.pos;
          k.aq_xf = L.rnn_wf.aq, k.aq_xw = L.rnn_w.aq;
        }
        k.ln_scale = L.rnn_ln.scale, k.ln_bias = L.rnn_ln.bias, k.eps = 1e-6f;
        k.h_out = hb, k.q_out = qd, k.M = B;
        if (trace_buf && step == 3 && l == 0) k.trace = trace_buf;
        const double Bd = B, Ed = E;
        LaunchScope ls(c, "dec_ssru_q_fused", 2.0 * Bd * 3.0 * Ed * Ed, 3.0 * Ed * Ed + Bd * Ed * (2.0 + 4.0 * 5.0));
        if (launch_dec_ssru(k, E, c.fast, s)) {
          set_error("fused SSRU kernel: unsupported embedding size " + std::to_string(E));
          return 1;
        }
      }
      if (cross_rc) {
        CrossRcArgs k{};
        k.map_ak = mapAk[l], k.map_av = mapAv[l];
        k.map_wk = L.ctx.k.map128, k.map_wv = L.ctx.v.map128;
        k.pb_k = L.ctx.k.pb, k.pb_v = L.ctx.v.pb;
        k.um_k = L.ctx.k.um, k.um_v = L.ctx.v.um;
        k.q = qd, k.lengths = d_lengths, k.B = B, k.T = T;
        k.dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
        k.out_f32 = nullptr;
        k.qo = qouts();
        qadd(k.qo, caq, L.ctx.o.aq);
        k.attn_head0 = last ? d_align : nullptr;
        if (trace_buf && step == 3 && l == 0) k.trace = trace_buf + 3 * trace_n;
        const double Bd = B, Ed = E;
        LaunchScope ls(c, "dec_cross_attention_rc", 2.0 * (cross_rcl ? src_tokens : Bd * (T > 32 ? 64.0 : 32.0)) * Ed * 2.0 * Ed,
                       2.0 * src_tokens * Ed + 2.0 * Ed * Ed + 5.0 * Bd * Ed);  // valid keys only
        if (cross_rcl ? launch_cross_attention_rcl(k, c.num_sms, s) : launch_cross_attention_rc(k, c.num_sms, c.fast, s)) {
          set_error("recompute cross-attention launch failed");
          return 1;
        }
      } else {
        QuantOuts q = qouts();
        qadd(q, caq, L.ctx.o.aq);
        LaunchScope ls(c, "dec_cross_attention", 0, 8.0 * src_tokens * E + 5.0 * B * E);
        if (launch_cross_attention(mapKc[l], mapVc[l], qd, d_lengths, B, T, H, dh, c.num_sms, nullptr, q,
                                   last ? d_align : nullptr, s)) {
          set_error("cross-attention: no kernel for " + std::to_string(H) + " heads of " + std::to_string(dh) +
                    " over " + std::to_string(T) + " source tokens");
          return 1;
        }
      }
      {  // Wo + residual + LN, FFN1 + ReLU, FFN2 + residual + LN in one row-tile kernel (Modules.cc:308-316, 251-257)
        RowsFfnArgs k{};
        k.map_a = map_caq;
        k.map_wo = L.ctx.o.map128, k.map_w1 = L.ffn.w1.map128, k.map_w2 = L.ffn.w2.map128;
        k.pb_o = L.ctx.o.pb, k.pb_1 = L.ffn.w1.pb, k.pb_2 = L.ffn.w2.pb;
        k.um_o = L.ctx.o.um, k.um_1 = L.ffn.w1.um, k.um_2 = L.ffn.w2.um;
        k.aq_1 = L.ffn.w1.aq, k.aq_2 = L.ffn.w2.aq;
        k.res = hb;
        k.ln1_scale = L.ctx.ln.scale, k.ln1_bias = L.ctx.ln.bias;
        k.ln2_scale = L.ffn.ln.scale, k.ln2_bias = L.ffn.ln.bias, k.eps = 1e-6f;
        if (last) {
          k.z_out = nullptr;
          k.zq[0] = reinterpret_cast<uint8_t*>(oq), k.zaq[0] = m.out.aq, k.n_zq = 1;
          k.zq_signed = a.logits ? 0 : 1;  // the fused argmax GEMM takes the signed qa (gemm_out.cu)
        } else {
          k.z_out = zb[l & 1];
          k.zq[0] = reinterpret_cast<uint8_t*>(zq[0]), k.zaq[0] = m.dec[l + 1].rnn_wf.aq;
          k.zq[1] = reinterpret_cast<uint8_t*>(zq[1]), k.zaq[1] = m.dec[l + 1].rnn_w.aq;
          k.n_zq = 2;
        }
        k.M = B;
        if (trace_buf && step == 3 && l == 0) k.trace = trace_buf + trace_n;
        const double Bd = B, Ed = E, Fd = F;
        LaunchScope ls(c, "dec_wo_ffn_fused", 2.0 * Bd * (Ed * Ed + 2.0 * Ed * Fd),
                       Ed * Ed + 2.0 * Ed * Fd + Bd * Ed * (1.0 + 4.0 + (last ? 1.0 : 6.0)));
        if (launch_rows_ffn(k, E, F, kRowTile, c.fast, s)) {
          set_error("fused FFN kernel: unsupported sizes E=" + std::to_string(E) + " F=" + std::to_string(F));
          return 1;
        }
      }
      in_f = zb[l & 1];
    }
    // output projection (+ shortlist) and greedy choice (Transformer.cc:176-182, 279-339)
    if (d_logits) {
      GemmCall g(&c, "dec_gemm_out_logits", B, Nout, E, EPI_F32);
      GemmProblem* p = g.add(oq, Wout, pb_out, m.out.um);
      if (!p) return 1;
      p->out = d_logits, p->ldo = Nout;
      if (g.launch()) return 1;
      {
        LaunchScope ls(c, "argmax_rows", 0, 4.0 * B * Nout);
        launch_argmax_rows(d_logits, B, Nout, best, s);
      }
      SB_CUDA(cudaMemcpyAsync(a.logits + static_cast<size_t>(step) * B * Nout, d_logits, 4ul * B * Nout,
                              cudaMemcpyDeviceToHost, s));
      c.d2h_bytes += 4ul * B * Nout;
    } else {
      const double Md = B, Nd = Nout, Kd = E;
      LaunchScope ls(c, "dec_gemm_out_argmax", 2.0 * Md * Nd * Kd, Md * Kd + Nd * Kd + 4.0 * Nd + 8.0 * Md);
      const int rc = out_ext ? launch_gemm_out_argmax_ext(map_oq, map_wout, map_ext, pb_out, dshift_out, m.out.um, c.fast, B,
                                                          Nout, E, best, c.num_sms, s,
                                                          (trace_buf && step == 3) ? trace_buf + 4 * trace_n : nullptr)
                             : launch_gemm_out_argmax(map_oq, map_wout, pb_out, c127_out, dmax_out,
                                                      c.fast ? ipb6_out : nullptr, m.out.um, m.out.eta, B, Nout, E, best,
                                                      c.num_sms, s);
      if (rc) {
        set_error("output GEMM: unsupported K " + std::to_string(E));
        return 1;
      }
    }
    // The step's bookkeeping (argmax -> word, record(), EOS flags) and the next step's input embedding are done by the
    // FRONT of the next step's first kernel (dec_ssru_kernel with embed set); the last executed step is closed by the
    // stand-alone kernel after the loop.
    executed = step + 1;
    // Model.cc:161: the loop stops once every sentence has produced EOS.  Every second step the done-counter is copied
    // to a pinned slot behind an event and the host looks at the previous copy, so the stream always holds a few
    // queued steps and is never drained (extra steps only produce discarded tokens); the steps in between stay
    // chained by programmatic dependent launch.
    if ((step & 1) == 1) {
      constexpr int kSlots = 8;
      const int poll = step >> 1;
      SB_CUDA(cudaMemcpyAsync(&c.done_slots[poll % kSlots], counters, 4, cudaMemcpyDeviceToHost, s));
      SB_CUDA(cudaEventRecord(c.done_events[poll % kSlots], s));
      c.d2h_bytes += 4;
      if (poll >= 1) {
        const int old = (poll - 1) % kSlots;
        SB_CUDA(cudaEventSynchronize(c.done_events[old]));
        if (c.done_slots[old] >= B) break;
      }
    }
  }
  if (executed > 0) {
    QuantOuts q = qouts();
    qadd(q, xq[0], m.dec[0].rnn_wf.aq), qadd(q, xq[1], m.dec[0].rnn_w.aq);
    {
      LaunchScope ls(c, "dec_finalize_embed", 0, 7.0 * B * E + 20.0 * B);
      launch_finalize_step(best, d_sl, d_forced, executed - 1, d_steps, done, tgt_len, counters, m.eos_id, m.emb_q, m.inv_qm,
                           m.sqrt_e, m.pos, B, E, xd, q, s);
    }
    SB_CUDA(cudaMemcpyAsync(&c.done_slots[0], counters, 4, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4;
    SB_CUDA(cudaStreamSynchronize(s));
    host_done = c.done_slots[0];
  }

  if (trace_buf) {
    SB_CUDA(cudaStreamSynchronize(s));
    if (FILE* f = fopen(trace_path, "w")) {
      for (int k = 0; k < 5; k++)
        for (int cta = 0; cta < c.num_sms; cta++) {
          const long long* t = trace_buf + k * trace_n + static_cast<size_t>(cta) * kTraceSlots;
          if (t[0] == 0) continue;
          fprintf(f, "%s %d", k == 0 ? "ssru" : k == 1 ? "ffn" : k == 2 ? "encffn" : k == 3 ? "cross" : "out", cta);
          // (the output GEMM's slots 4.. are counts and accumulated waits, not stamps)
          for (int i = 0; i < kTraceSlots; i++) fprintf(f, " %lld", (k == 4 && i >= 4) ? t[i] : (t[i] ? t[i] - t[0] : -1));
          fprintf(f, "\n");
        }
      fclose(f);
    }
    cudaFree(trace_buf);
  }

  // ---- results
  std::vector<uint32_t> lens(B);
  SB_CUDA(cudaMemcpyAsync(lens.data(), tgt_len, 4ul * B, cudaMemcpyDeviceToHost, s));
  if (d_align_all && executed > 0) {
    SB_CUDA(cudaMemcpyAsync(a.alignment, d_align_all, 4ul * executed * B * T, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * executed * B * T;
  }
  if (!a.device_io && a.step_tokens && executed > 0) {
    SB_CUDA(cudaMemcpyAsync(a.step_tokens, d_steps, 4ul * executed * B, cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * executed * B;
  }
  if (!a.device_io && a.sentence_tokens && executed > 0) {
    if (a.row_stride < static_cast<size_t>(executed)) {
      set_error("sentence_tokens: row_stride smaller than the number of decode steps");
      return 1;
    }
    // one row per sentence: the host then copies each sentence's recorded prefix without striding through the matrix
    uint32_t* d_rows = c.take<uint32_t>(static_cast<size_t>(max_steps) * B);
    {
      LaunchScope ls(c, "transpose_steps", 0, 8.0 * executed * B);
      launch_transpose_u32(d_steps, executed, B, d_rows, executed, s);
    }
    SB_CUDA(cudaMemcpy2DAsync(a.sentence_tokens, 4ul * a.row_stride, d_rows, 4ul * executed, 4ul * executed, B,
                              cudaMemcpyDeviceToHost, s));
    c.d2h_bytes += 4ul * executed * B;
  }
  SB_CUDA(cudaStreamSynchronize(s));
  if (a.target_lengths) memcpy(a.target_lengths, lens.data(), 4ul * B);
  c.d2h_bytes += 4ul * B;
  uint64_t total = 0;
  uint32_t longest = 0;
  bool all_done = host_done >= B;
  for (int b = 0; b < B; b++) {
    total += lens[b];
    longest = std::max(longest, lens[b]);
  }
  a.target_tokens = total;
  // steps the reference would have run: up to the step where the last sentence finished
  a.steps = all_done ? longest : static_cast<size_t>(executed);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error(std::string("forward failed: ") + cudaGetErrorString(e));
    return 1;
  }
  return 0;
}

}  // namespace sb
