// See kernels.cuh.  sm_100a; compiled with -fmad=false, all f32 arithmetic spelled with explicit
// round-to-nearest intrinsics in the reference's evaluation order.
#include "kernels.cuh"

#include <limits.h>
#include <stdio.h>

#include "exact_math.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

__device__ __forceinline__ void store_quant4(const QuantOuts& q, size_t off, const float (&y)[4]) {
  for (int k = 0; k < q.n; k++) {
    const float aq = q.aq[k];
    *reinterpret_cast<uint32_t*>(q.ptr[k] + off) =
        pack4(quantize1(y[0], aq), quantize1(y[1], aq), quantize1(y[2], aq), quantize1(y[3], aq));
  }
}

// ------------------------------------------------------------------ embedding
__global__ void embed_kernel(const uint32_t* __restrict__ tokens, const int8_t* __restrict__ emb_q, float inv_qm,
                             float sqrt_e, const float* __restrict__ pos, int rows, int T, int E, int pos_from_row,
                             int zero_embed, float* __restrict__ x, QuantOuts q) {
  const int per_row = E >> 2;
  const size_t gid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<size_t>(rows) * per_row) return;
  const int r = static_cast<int>(gid / per_row);
  const int e = static_cast<int>(gid % per_row) * 4;
  float w[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  if (!zero_embed) {
    const uint32_t tok = tokens[r];
    const char4 c = *reinterpret_cast<const char4*>(emb_q + static_cast<size_t>(tok) * E + e);
    w[0] = __fmul_rn(static_cast<float>(c.x), inv_qm);
    w[1] = __fmul_rn(static_cast<float>(c.y), inv_qm);
    w[2] = __fmul_rn(static_cast<float>(c.z), inv_qm);
    w[3] = __fmul_rn(static_cast<float>(c.w), inv_qm);
  }
  const int p = pos_from_row ? (r % T) : 0;
  const float4 ps = *reinterpret_cast<const float4*>(pos + static_cast<size_t>(p) * E + e);
  float y[4];
  y[0] = __fadd_rn(__fmul_rn(w[0], sqrt_e), ps.x);
  y[1] = __fadd_rn(__fmul_rn(w[1], sqrt_e), ps.y);
  y[2] = __fadd_rn(__fmul_rn(w[2], sqrt_e), ps.z);
  y[3] = __fadd_rn(__fmul_rn(w[3], sqrt_e), ps.w);
  const size_t off = static_cast<size_t>(r) * E + e;
  if (x) *reinterpret_cast<float4*>(x + off) = make_float4(y[0], y[1], y[2], y[3]);
  store_quant4(q, off, y);
}

__global__ void quantize_kernel(const float* __restrict__ x, size_t n4, QuantOuts q) {
  const size_t gid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= n4) return;
  const float4 v = reinterpret_cast<const float4*>(x)[gid];
  const float y[4] = {v.x, v.y, v.z, v.w};
  store_quant4(q, gid * 4, y);
}

// ------------------------------------------------------------------ self attention
// Block = one (sentence, head); thread = one query row.  K and V of the head sit in shared memory and are
// read as warp broadcasts; every dot product is a sequential fmaf chain (ruy's sgemm order), the
// softmax max/sum/divide follow slimt/TensorOps.cc:282-315.
template <int DH>
__global__ void self_attention_kernel(const float* __restrict__ Q, const float* __restrict__ K,
                                      const float* __restrict__ V, const uint32_t* __restrict__ lengths, int T,
                                      int H, float dk, float* __restrict__ out_f32, QuantOuts q) {
  extern __shared__ float smem_f[];
  const int b = blockIdx.x / H;
  const int h = blockIdx.x % H;
  const int E = H * DH;
  const int len = min(static_cast<int>(lengths[b]), T);
  const int Tp = T | 1;
  __shared__ uint64_t exp_tab[32];
  if (threadIdx.x < 32) exp_tab[threadIdx.x] = kExp2fTab[threadIdx.x];
  float* Ks = smem_f;
  float* Vs = Ks + static_cast<size_t>(T) * DH;
  float* Ss = Vs + static_cast<size_t>(T) * DH;

  const size_t base = static_cast<size_t>(b) * T * E + static_cast<size_t>(h) * DH;
  for (int i = threadIdx.x; i < len * (DH / 4); i += blockDim.x) {
    const int j = i / (DH / 4);
    const int c = (i % (DH / 4)) * 4;
    *reinterpret_cast<float4*>(Ks + j * DH + c) = *reinterpret_cast<const float4*>(K + base + static_cast<size_t>(j) * E + c);
    *reinterpret_cast<float4*>(Vs + j * DH + c) = *reinterpret_cast<const float4*>(V + base + static_cast<size_t>(j) * E + c);
  }
  __syncthreads();

  float* S = Ss + static_cast<size_t>(threadIdx.x) * Tp;
  for (int i = threadIdx.x; i < T; i += blockDim.x) {
    float acc[DH];
    const size_t off = base + static_cast<size_t>(i) * E;
    if (i < len) {
      float qv[DH];
#pragma unroll
      for (int d = 0; d < DH; d += 4) {
        const float4 t = *reinterpret_cast<const float4*>(Q + off + d);
        qv[d] = t.x, qv[d + 1] = t.y, qv[d + 2] = t.z, qv[d + 3] = t.w;
      }
      // Four keys at a time: each dot product stays the reference's sequential fma chain, but four independent
      // chains (and four expf evaluations) are in flight per thread -- with one block per SM at long T there are
      // few warps to hide a single chain's latency behind.
      float mx = -3.402823466e+38f;
      int j = 0;
      for (; j + 4 <= len; j += 4) {
        const float* kp = Ks + j * DH;
        float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
#pragma unroll
        for (int d = 0; d < DH; d++) {
          s0 = fmaf(qv[d], kp[d], s0);
          s1 = fmaf(qv[d], kp[DH + d], s1);
          s2 = fmaf(qv[d], kp[2 * DH + d], s2);
          s3 = fmaf(qv[d], kp[3 * DH + d], s3);
        }
        s0 = __fmul_rn(dk, s0), s1 = __fmul_rn(dk, s1), s2 = __fmul_rn(dk, s2), s3 = __fmul_rn(dk, s3);
        S[j] = s0, S[j + 1] = s1, S[j + 2] = s2, S[j + 3] = s3;
        mx = fmaxf(fmaxf(fmaxf(mx, s0), fmaxf(s1, s2)), s3);
      }
      for (; j < len; j++) {
        float s = 0.0f;
#pragma unroll
        for (int d = 0; d < DH; d++) s = fmaf(qv[d], Ks[j * DH + d], s);
        s = __fmul_rn(dk, s);
        S[j] = s;
        mx = fmaxf(mx, s);
      }
      float sum = 0.0f;
      j = 0;
      for (; j + 4 <= len; j += 4) {
        const float e0 = expf_glibc_nonpos_tab(__fsub_rn(S[j], mx), exp_tab);
        const float e1 = expf_glibc_nonpos_tab(__fsub_rn(S[j + 1], mx), exp_tab);
        const float e2 = expf_glibc_nonpos_tab(__fsub_rn(S[j + 2], mx), exp_tab);
        const float e3 = expf_glibc_nonpos_tab(__fsub_rn(S[j + 3], mx), exp_tab);
        S[j] = e0, S[j + 1] = e1, S[j + 2] = e2, S[j + 3] = e3;
        sum = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(sum, e0), e1), e2), e3);
      }
      for (; j < len; j++) {
        const float e = expf_glibc_nonpos_tab(__fsub_rn(S[j], mx), exp_tab);
        S[j] = e;
        sum = __fadd_rn(sum, e);
      }
#pragma unroll
      for (int d = 0; d < DH; d++) acc[d] = 0.0f;
      // every probability of the row divides by `sum`: reciprocal once, three FFMAs per key (exact_math.cuh)
      const float sum_rcp = rcp_refined(sum);
      const float sum_lo = div_guard_lo(sum);
      for (j = 0; j < len; j++) {
        const float p = div_by_rcp(S[j], sum, sum_rcp, sum_lo);
#pragma unroll
        for (int d = 0; d < DH; d++) acc[d] = fmaf(p, Vs[j * DH + d], acc[d]);
      }
    } else {
#pragma unroll
      for (int d = 0; d < DH; d++) acc[d] = 0.0f;  // padded query rows never reach a valid output
    }
    if (out_f32) {
#pragma unroll
      for (int d = 0; d < DH; d += 4) *reinterpret_cast<float4*>(out_f32 + off + d) = make_float4(acc[d], acc[d + 1], acc[d + 2], acc[d + 3]);
    }
#pragma unroll
    for (int d = 0; d < DH; d += 4) {
      const float y[4] = {acc[d], acc[d + 1], acc[d + 2], acc[d + 3]};
      store_quant4(q, off + d, y);
    }
  }
}

// ------------------------------------------------------------------ SSRU tail
// Warp = one sentence row.  Elementwise part is lane-parallel and coalesced; the two LayerNorm sums
// run in element order over the row parked in shared memory (every lane walks the same chain).
__global__ void ssru_ln_kernel(const float* __restrict__ f, const float* __restrict__ wx, float* __restrict__ state,
                               const float* __restrict__ x, const float* __restrict__ ln_scale,
                               const float* __restrict__ ln_bias, float eps, int B, int E, float* __restrict__ h,
                               QuantOuts q) {
  extern __shared__ float smem_f[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + warp;
  if (row >= B) return;
  float* t = smem_f + static_cast<size_t>(warp) * E;
  const size_t base = static_cast<size_t>(row) * E;
  for (int e = lane; e < E; e += 32) {
    const float sg = sigmoid_ref(f[base + e]);
    const float a = __fmul_rn(sg, state[base + e]);
    const float bb = __fmul_rn(__fsub_rn(1.0f, sg), wx[base + e]);
    const float c = __fadd_rn(a, bb);  // highway(c_prev, Wx, f), slimt/TensorOps.cc:662-682
    state[base + e] = c;
    const float y = c > 0.0f ? c : 0.0f;
    t[e] = __fadd_rn(x[base + e], y);
  }
  __syncwarp();
  float sum = 0.0f;
  for (int e = 0; e < E; e++) sum = __fadd_rn(sum, t[e]);
  const float cols = static_cast<float>(E);
  const float mean = __fdiv_rn(sum, cols);
  float sq = 0.0f;
  for (int e = 0; e < E; e++) {
    const float d = __fsub_rn(t[e], mean);
    sq = __fadd_rn(sq, __fmul_rn(d, d));
  }
  const float sigma = __fsqrt_rn(__fadd_rn(__fdiv_rn(sq, cols), eps));
  for (int e = lane; e < E; e += 32) {
    const float n = __fdiv_rn(__fsub_rn(t[e], mean), sigma);
    const float y = __fadd_rn(__fmul_rn(ln_scale[e], n), ln_bias[e]);
    if (h) h[base + e] = y;
    for (int k = 0; k < q.n; k++) q.ptr[k][base + e] = static_cast<int8_t>(quantize1(y, q.aq[k]));
  }
}

// ------------------------------------------------------------------ step bookkeeping
// Warp = one sentence row, eight rows per block: lane 0 does the row's bookkeeping and broadcasts the next input word,
// the warp then builds that word's decoder input.  (One 64-thread block per row -- the first version -- spent most of
// its 10.9 us at B = 4096 launching 4096 tiny blocks.)
__global__ void __launch_bounds__(256) finalize_step_kernel(
    unsigned long long* __restrict__ best, const uint32_t* __restrict__ shortlist, const uint32_t* __restrict__ forced,
    int step, uint32_t* __restrict__ step_tokens, uint8_t* __restrict__ done, uint32_t* __restrict__ tgt_len,
    int* __restrict__ n_done, uint32_t eos_id, const int8_t* __restrict__ emb_q, float inv_qm, float sqrt_e,
    const float* __restrict__ pos0, int B, int E, float* __restrict__ x, QuantOuts q) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  pdl_launch_dependents();
  pdl_wait();
  if (b >= B) return;
  uint32_t tok = 0;
  if (lane == 0) {
    const unsigned long long packed = best[b];
    const uint32_t idx = 0xFFFFFFFFu - static_cast<uint32_t>(packed & 0xFFFFFFFFull);
    const uint32_t word = shortlist ? shortlist[idx] : idx;
    step_tokens[static_cast<size_t>(step) * B + b] = word;
    if (!done[b]) {  // record(), slimt/Model.cc:127-137: append unless already finished
      tgt_len[b] += 1;
      if (word == eos_id) {
        done[b] = 1;
        atomicAdd(n_done, 1);
      }
    }
    best[b] = 0ull;
    tok = forced ? forced[static_cast<size_t>(step) * B + b] : word;
  }
  tok = __shfl_sync(0xffffffffu, tok, 0);
  for (int e = lane * 4; e < E; e += 128) {
    const char4 c = *reinterpret_cast<const char4*>(emb_q + static_cast<size_t>(tok) * E + e);
    const float4 ps = *reinterpret_cast<const float4*>(pos0 + e);
    float y[4];
    y[0] = __fadd_rn(__fmul_rn(__fmul_rn(static_cast<float>(c.x), inv_qm), sqrt_e), ps.x);
    y[1] = __fadd_rn(__fmul_rn(__fmul_rn(static_cast<float>(c.y), inv_qm), sqrt_e), ps.y);
    y[2] = __fadd_rn(__fmul_rn(__fmul_rn(static_cast<float>(c.z), inv_qm), sqrt_e), ps.z);
    y[3] = __fadd_rn(__fmul_rn(__fmul_rn(static_cast<float>(c.w), inv_qm), sqrt_e), ps.w);
    const size_t off = static_cast<size_t>(b) * E + e;
    *reinterpret_cast<float4*>(x + off) = make_float4(y[0], y[1], y[2], y[3]);
    store_quant4(q, off, y);
  }
}

__global__ void gather_rows_kernel(const int8_t* __restrict__ W, const float* __restrict__ pb,
                                   const int32_t* __restrict__ c127, const uint32_t* __restrict__ idx, int K,
                                   int8_t* __restrict__ W_sel, float* __restrict__ pb_sel,
                                   int32_t* __restrict__ c127_sel) {
  const int i = blockIdx.x;
  const uint32_t src = idx[i];
  const uint4* s = reinterpret_cast<const uint4*>(W + static_cast<size_t>(src) * K);
  uint4* d = reinterpret_cast<uint4*>(W_sel + static_cast<size_t>(i) * K);
  for (int t = threadIdx.x; t < K / 16; t += blockDim.x) d[t] = s[t];
  if (threadIdx.x == 0) {
    pb_sel[i] = pb[src];
    if (c127_sel) c127_sel[i] = c127[src];
  }
}

// dmax[chunk] = max over the chunk's 32 columns of (c127[n] * um + pb[n]), rounded up to float: the
// column-dependent part of the logit upper bound used by the fused output GEMM (gemm_out.cu).
__global__ void out_bounds_kernel(const int32_t* __restrict__ c127, const float* __restrict__ pb, float um, int N,
                                  float* __restrict__ dmax) {
  const int chunk = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (chunk * 32 >= N) return;
  const int n = chunk * 32 + lane;
  double d = -1.0e300;
  if (n < N) d = static_cast<double>(c127[n]) * static_cast<double>(um) + static_cast<double>(pb[n]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d = fmax(d, __shfl_xor_sync(0xffffffffu, d, o));
  if (lane == 0) dmax[chunk] = __double2float_ru(d);
}

// ipb6[n] = (round(c127[n] + pb[n] / um) << 6) + (63 - n % 64): the per-column offset of the tolerance-mode output
// GEMM's integer logit proxy (gemm_out.cu), evaluated in double.  Entries from N up to the end of the last 256-column
// tile get the most negative value that cannot overflow when a zero accumulator is added.
__global__ void out_ipb_kernel(const int32_t* __restrict__ c127, const float* __restrict__ pb, float um, int N, int n_pad,
                               int32_t* __restrict__ ipb6) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_pad) return;
  if (n >= N) {
    ipb6[n] = INT_MIN + 64;
    return;
  }
  double t = rint(static_cast<double>(c127[n]) + static_cast<double>(pb[n]) / static_cast<double>(um));
  t = fmin(fmax(t, -16777216.0), 16777216.0);  // |accumulator| < 2^22, so (v' + ipb) << 6 stays inside int32
  ipb6[n] = (static_cast<int32_t>(t) << 6) + (63 - (n & 63));
}

// Per output column n (gemm_out_ext.cu): ipb[n] = round(c127[n] + pb[n] / um) in double, written as 32 int8 digits
// e[n][0..31] with sum_k a_k * e[n][k] = ipb[n] for a = (127 x 31, 1), one 128-byte row per column (the layout the
// weight tile's TMA box uses; bytes 32..127 stay zero); dshift[n] = c127[n] - ipb[n] turns a proxy back into the
// shifted accumulator of the exact formula.  Columns N .. n_pad - 1 are zero.  *overflow is set when some |ipb|
// exceeds what the digits can hold (31 * 127 * 127 + 63).
__global__ void out_ext_kernel(const int32_t* __restrict__ c127, const float* __restrict__ pb, float um, int N, int n_pad,
                               uint8_t* __restrict__ ext, int32_t* __restrict__ dshift, int* __restrict__ overflow) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_pad) return;
  uint4* row = reinterpret_cast<uint4*>(ext + static_cast<size_t>(n) * 128);
  uint32_t w[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  int ds = 0;
  if (n < N) {
    double t = rint(static_cast<double>(c127[n]) + static_cast<double>(pb[n]) / static_cast<double>(um));
    if (fabs(t) > 500093.0) {
      atomicOr(overflow, 1);
      t = fmin(fmax(t, -500093.0), 500093.0);
    }
    const int ipb = static_cast<int>(t);
    int Q = static_cast<int>(rint(static_cast<double>(ipb) / 127.0));
    if (Q > 3937) Q = 3937;
    if (Q < -3937) Q = -3937;
    const int r = ipb - 127 * Q;  // |r| <= 63 (<= 126 at the clamped ends, still an int8)
    const int base = Q / 31, rem = Q - 31 * base;
    const int step = rem > 0 ? 1 : -1, cnt = rem > 0 ? rem : -rem;
    for (int k = 0; k < 32; k++) {
      const int d = k < 31 ? base + (k < cnt ? step : 0) : r;
      w[k >> 2] |= static_cast<uint32_t>(d & 0xff) << (8 * (k & 3));
    }
    ds = c127[n] - ipb;
  }
  row[0] = make_uint4(w[0], w[1], w[2], w[3]);
  row[1] = make_uint4(w[4], w[5], w[6], w[7]);
  for (int i = 2; i < 8; i++) row[i] = make_uint4(0u, 0u, 0u, 0u);
  dshift[n] = ds;
}

__device__ __forceinline__ unsigned long long pack_best_k(float v, uint32_t idx) {
  if (v == 0.0f) v = 0.0f;
  uint32_t bits = __float_as_uint(v);
  uint32_t key = (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  return (static_cast<unsigned long long>(key) << 32) | static_cast<unsigned long long>(0xFFFFFFFFu - idx);
}

__global__ void argmax_rows_kernel(const float* __restrict__ logits, int cols, unsigned long long* __restrict__ best) {
  const int row = blockIdx.x;
  const float* p = logits + static_cast<size_t>(row) * cols;
  unsigned long long loc = 0ull;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    const unsigned long long k = pack_best_k(p[c], c);
    loc = k > loc ? k : loc;
  }
  atomicMax(best + row, loc);
}

}  // namespace

void launch_embed(const uint32_t* tokens, const int8_t* emb_q, float inv_qm, float sqrt_e, const float* pos, int rows,
                  int T, int E, int pos_from_row, int zero_embed, float* x, QuantOuts q, cudaStream_t stream) {
  const size_t n = static_cast<size_t>(rows) * (E / 4);
  if (n == 0) return;
  embed_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(tokens, emb_q, inv_qm, sqrt_e, pos, rows, T, E,
                                                                         pos_from_row, zero_embed, x, q);
}

void launch_quantize(const float* x, size_t n, QuantOuts q, cudaStream_t stream) {
  const size_t n4 = n / 4;
  if (n4 == 0) return;
  quantize_kernel<<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, stream>>>(x, n4, q);
}

int launch_self_attention(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T, int H,
                          int dh, float* out_f32, QuantOuts q, cudaStream_t stream) {
  if (B == 0) return 0;
  // 1/sqrt(dim_head) evaluated in double then narrowed, as `1.0F / std::sqrt(size_t)` does (Modules.cc:43).
  const float dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
  int threads = ((T + 31) / 32) * 32;
  if (threads > 128) threads = 128;
  const int Tp = T | 1;
  size_t smem = (static_cast<size_t>(2) * T * dh + static_cast<size_t>(threads) * Tp) * sizeof(float);
  while (smem > 200 * 1024 && threads > 32) {
    threads -= 32;
    smem = (static_cast<size_t>(2) * T * dh + static_cast<size_t>(threads) * Tp) * sizeof(float);
  }
  if (smem > 200 * 1024) return 1;  // K, V and one warp's score rows no longer fit: T > 533 (head size 32), T > 319 (64)
  if (dh == 32) {
    ensure_dyn_smem(self_attention_kernel<32>, smem);
    self_attention_kernel<32><<<B * H, threads, smem, stream>>>(Q, K, V, lengths, T, H, dk, out_f32, q);
  } else if (dh == 64) {
    ensure_dyn_smem(self_attention_kernel<64>, smem);
    self_attention_kernel<64><<<B * H, threads, smem, stream>>>(Q, K, V, lengths, T, H, dk, out_f32, q);
  } else {
    return 1;  // the model loader only admits head sizes 32 and 64; reported through the error convention by the caller
  }
  return 0;
}

void launch_ssru_ln(const float* f, const float* wx, float* state, const float* x, const float* ln_scale,
                    const float* ln_bias, float eps, int B, int E, float* h, QuantOuts q, cudaStream_t stream) {
  if (B == 0) return;
  const int wpb = 4;
  const size_t smem = static_cast<size_t>(wpb) * E * sizeof(float);
  ssru_ln_kernel<<<(B + wpb - 1) / wpb, wpb * 32, smem, stream>>>(f, wx, state, x, ln_scale, ln_bias, eps, B, E, h, q);
}

void launch_finalize_step(unsigned long long* best, const uint32_t* shortlist, const uint32_t* forced, int step,
                          uint32_t* step_tokens, uint8_t* done, uint32_t* tgt_len, int* n_done, uint32_t eos_id,
                          const int8_t* emb_q, float inv_qm, float sqrt_e, const float* pos0, int B, int E, float* x,
                          QuantOuts q, cudaStream_t stream) {
  if (B == 0) return;
  launch_pdl(finalize_step_kernel, dim3((B + 7) / 8), dim3(256), 0, stream, best, shortlist, forced, step, step_tokens, done, tgt_len,
             n_done, eos_id, emb_q, inv_qm, sqrt_e, pos0, B, E, x, q);
}

void launch_gather_rows(const int8_t* W, const float* pb, const int32_t* c127, const uint32_t* idx, int n_idx, int K,
                        int8_t* W_sel, float* pb_sel, int32_t* c127_sel, cudaStream_t stream) {
  if (n_idx == 0) return;
  gather_rows_kernel<<<n_idx, 32, 0, stream>>>(W, pb, c127, idx, K, W_sel, pb_sel, c127_sel);
}

void launch_out_bounds(const int32_t* c127, const float* pb, float um, int N, float* dmax, cudaStream_t stream) {
  const int chunks = (N + 31) / 32;
  if (chunks == 0) return;
  out_bounds_kernel<<<(chunks + 7) / 8, 256, 0, stream>>>(c127, pb, um, N, dmax);
}

void launch_out_ipb(const int32_t* c127, const float* pb, float um, int N, int32_t* ipb6, cudaStream_t stream) {
  const int n_pad = (N + 255) / 256 * 256;
  if (n_pad == 0) return;
  out_ipb_kernel<<<(n_pad + 255) / 256, 256, 0, stream>>>(c127, pb, um, N, n_pad, ipb6);
}

void launch_out_ext(const int32_t* c127, const float* pb, float um, int N, uint8_t* ext, int32_t* dshift, int* overflow,
                    cudaStream_t stream) {
  const int n_pad = (N + 255) / 256 * 256;
  if (n_pad == 0) return;
  out_ext_kernel<<<(n_pad + 127) / 128, 128, 0, stream>>>(c127, pb, um, N, n_pad, ext, dshift, overflow);
}

__global__ void transpose_u32_kernel(const uint32_t* __restrict__ src, int rows, int cols, uint32_t* __restrict__ dst,
                                     int dst_stride) {
  __shared__ uint32_t tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? src[static_cast<size_t>(r) * cols + c] : 0u;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) dst[static_cast<size_t>(c) * dst_stride + r] = tile[threadIdx.x][i];
  }
}

void launch_transpose_u32(const uint32_t* src, int rows, int cols, uint32_t* dst, int dst_stride, cudaStream_t stream) {
  if (rows == 0 || cols == 0) return;
  transpose_u32_kernel<<<dim3((cols + 31) / 32, (rows + 31) / 32), dim3(32, 8), 0, stream>>>(src, rows, cols, dst, dst_stride);
}

void launch_argmax_rows(const float* logits, int rows, int cols, unsigned long long* best, cudaStream_t stream) {
  if (rows == 0) return;
  argmax_rows_kernel<<<rows, 256, 0, stream>>>(logits, cols, best);
}

}  // namespace sb
