// See kernels.cuh.  sm_100a; compiled with -fmad=false, all f32 arithmetic spelled with explicit
// round-to-nearest intrinsics in the reference's evaluation order.
#include "kernels.cuh"

#include <stdio.h>

#include "exact_math.cuh"
#include "packed_best.cuh"
#include "ptx.cuh"
#include "sample_rng.cuh"
#include "score_partial.cuh"

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
                             int zero_embed, int shift, float* __restrict__ x, QuantOuts q) {
  const int per_row = E >> 2;
  const size_t gid = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (gid >= static_cast<size_t>(rows) * per_row) return;
  const int r = static_cast<int>(gid / per_row);
  const int e = static_cast<int>(gid % per_row) * 4;
  char4 c = make_char4(0, 0, 0, 0);
  if (!zero_embed && !(shift && r % T == 0)) {
    const uint32_t tok = tokens[shift ? r - 1 : r];
    c = *reinterpret_cast<const char4*>(emb_q + static_cast<size_t>(tok) * E + e);
  }
  const int p = pos_from_row ? (r % T) : 0;
  const float4 ps = *reinterpret_cast<const float4*>(pos + static_cast<size_t>(p) * E + e);
  const float y[4] = {embed1(c.x, inv_qm, sqrt_e, ps.x), embed1(c.y, inv_qm, sqrt_e, ps.y),
                      embed1(c.z, inv_qm, sqrt_e, ps.z), embed1(c.w, inv_qm, sqrt_e, ps.w)};
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
                                      int H, float dk, QuantOuts q) {
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
#pragma unroll
    for (int d = 0; d < DH; d += 4) {
      const float y[4] = {acc[d], acc[d + 1], acc[d + 2], acc[d + 3]};
      store_quant4(q, off + d, y);
    }
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
    const uint32_t word = best_word(best[b], shortlist);
    record_word(word, done[b], tgt_len[b], eos_id, step, B, b, step_tokens, done, tgt_len, n_done, best);
    tok = forced ? forced[static_cast<size_t>(step) * B + b] : word;
  }
  tok = __shfl_sync(0xffffffffu, tok, 0);
  for (int e = lane * 4; e < E; e += 128) {
    const char4 c = *reinterpret_cast<const char4*>(emb_q + static_cast<size_t>(tok) * E + e);
    const float4 ps = *reinterpret_cast<const float4*>(pos0 + e);
    const float y[4] = {embed1(c.x, inv_qm, sqrt_e, ps.x), embed1(c.y, inv_qm, sqrt_e, ps.y),
                        embed1(c.z, inv_qm, sqrt_e, ps.z), embed1(c.w, inv_qm, sqrt_e, ps.w)};
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

__global__ void argmax_rows_kernel(const float* __restrict__ logits, int cols, unsigned long long* __restrict__ best) {
  const int row = blockIdx.x;
  const float* p = logits + static_cast<size_t>(row) * cols;
  unsigned long long loc = 0ull;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    const unsigned long long k = pack_best(p[c], c);
    loc = k > loc ? k : loc;
  }
  atomicMax(best + row, loc);
}

// ------------------------------------------------------------------ token scores
// Logits tap: the partial (m, s) of every 64-column strip of every row, with the same strip_partial as the fused
// scores epilogue.  Thread = (strip, row), rows fastest, so the partial stores are coalesced.  kTemper: the partials of
// the tempered logits fl32(y * inv_t) (sampling at a temperature other than 1).
template <bool kTemper>
__global__ void score_rows_kernel(const float* __restrict__ logits, int B, int N, float2* __restrict__ partials,
                                  float inv_t) {
  const size_t i = static_cast<size_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  const int n_strips = (N + kScoreStrip - 1) / kScoreStrip;
  if (i >= static_cast<size_t>(n_strips) * B) return;
  const int t = static_cast<int>(i / B), b = static_cast<int>(i % B);
  const float ninf = -__int_as_float(0x7f800000);
  const float* p = logits + static_cast<size_t>(b) * N + t * kScoreStrip;
  float y0[32], y1[32];
#pragma unroll
  for (int j = 0; j < 32; j += 4) {  // N % 8 == 0: groups of four are entirely inside or outside
    const int n0 = t * kScoreStrip + j;
    const float4 a = n0 < N ? *reinterpret_cast<const float4*>(p + j) : make_float4(ninf, ninf, ninf, ninf);
    const float4 c = n0 + 32 < N ? *reinterpret_cast<const float4*>(p + 32 + j) : make_float4(ninf, ninf, ninf, ninf);
    y0[j] = a.x, y0[j + 1] = a.y, y0[j + 2] = a.z, y0[j + 3] = a.w;
    y1[j] = c.x, y1[j + 1] = c.y, y1[j + 2] = c.z, y1[j + 3] = c.w;
  }
  if constexpr (kTemper) temper64(y0, y1, inv_t);
  partials[i] = strip_partial(y0, y1);
}

// The exact logit of output column col for row b from the signed int8 operands (the fused GEMM's value, bit for bit).
__device__ __forceinline__ float exact_logit(const ScoreStepArgs& a, int b, int col) {
  const int4* q = reinterpret_cast<const int4*>(a.oq + static_cast<size_t>(b) * a.K);
  const int4* wr = reinterpret_cast<const int4*>(a.w + static_cast<size_t>(col) * a.K);
  int acc = 0;
  for (int k = 0; k < a.K / 16; k++) {
    const int4 x = q[k], v = wr[k];
    acc = __dp4a(x.x, v.x, acc), acc = __dp4a(x.y, v.y, acc), acc = __dp4a(x.z, v.z, acc), acc = __dp4a(x.w, v.w, acc);
  }
  return dequant1(acc + a.c127[col], a.um, a.pb[col]);
}

// Block = 32 rows (lane = row) x 32 warps (warp = a contiguous group of strips).  Both step kernels reduce a row's
// partials in this one order: M = max_t m_t, then group sum sm[w][lane] = sum over warp w's strips t0 <= t < t1, in
// ascending order and in double, of s_t * exp(m_t - M).  The caller sums the 32 groups in ascending order: S, and
// LSE = M + log S.  Returns M.
constexpr int kScoreWarps = 32;
__device__ __forceinline__ float reduce_partials(const float2* __restrict__ partials, int B, int N, int b, int lane,
                                                 int w, float (&mx)[kScoreWarps][32], double (&sm)[kScoreWarps][32]) {
  const float ninf = -__int_as_float(0x7f800000);
  const int n_strips = (N + kScoreStrip - 1) / kScoreStrip;
  const int per = (n_strips + kScoreWarps - 1) / kScoreWarps;
  const int t0 = min(n_strips, w * per), t1 = min(n_strips, t0 + per);
  float m = ninf;
  if (b < B)
    for (int t = t0; t < t1; t++) m = fmaxf(m, partials[static_cast<size_t>(t) * B + b].x);
  mx[w][lane] = m;
  __syncthreads();
  float M = ninf;
#pragma unroll 8
  for (int k = 0; k < kScoreWarps; k++) M = fmaxf(M, mx[k][lane]);
  double s = 0.0;
  if (b < B)
    for (int t = t0; t < t1; t++) {
      const float2 p = partials[static_cast<size_t>(t) * B + b];
      s += static_cast<double>(p.y) * static_cast<double>(score_exp(__fsub_rn(p.x, M)));
    }
  sm[w][lane] = s;
  __syncthreads();
  return M;
}

// The chosen column's logit: the packed best word's value (greedy), or for a forced word its column (binary search in
// the sorted shortlist) evaluated exactly from the int8 operands -- or read from the tap.
__global__ void __launch_bounds__(32 * kScoreWarps) score_step_kernel(ScoreStepArgs a) {
  __shared__ float mx[kScoreWarps][32];
  __shared__ double sm[kScoreWarps][32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int b = blockIdx.x * 32 + lane;
  const int B = a.B;
  pdl_launch_dependents();
  pdl_wait();
  const float ninf = -__int_as_float(0x7f800000);
  const float M = reduce_partials(a.partials, B, a.N, b, lane, w, mx, sm);
  if (w != 0 || b >= B) return;
  double S = 0.0;
  for (int k = 0; k < kScoreWarps; k++) S += sm[k][lane];
  const double lse = static_cast<double>(M) + log(S);
  float y;
  if (a.forced == nullptr) {
    y = best_value(a.best[b]);
  } else {
    const uint32_t word = a.forced[static_cast<size_t>(a.step) * B + b];
    int col = -1;
    if (a.shortlist) {
      int lo = 0, hi = a.N;  // first entry >= word
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a.shortlist[mid] < word) lo = mid + 1;
        else hi = mid;
      }
      if (lo < a.N && a.shortlist[lo] == word) col = lo;
    } else if (word < static_cast<uint32_t>(a.N)) {
      col = static_cast<int>(word);
    }
    if (col < 0) {
      y = ninf;  // not among the output columns: probability 0
    } else if (a.logits) {
      y = a.logits[static_cast<size_t>(b) * a.N + col];
    } else {
      y = exact_logit(a, b, col);
    }
  }
  a.scores[static_cast<size_t>(a.step) * B + b] = static_cast<float>(static_cast<double>(y) - lse);
}

// Sampling (include/slimt_b200.h, DESIGN §4.4b), same block shape.  Over the tempered partials: warp 0 (lane = row)
// draws u and walks the cumulative sums towards u * S -- the 32 group sums, then the chosen group's strip terms, each in
// the order and with the very terms reduce_partials summed -- to a strip; a strip whose running sum passes the target is
// chosen, a term of 0 never is, and when rounding exhausts a level the last nonzero entry of that level is taken.  Every
// warp then evaluates two of the 64 tempered logits z of each row's chosen strip (exactly from the int8 operands, or
// from the tap), and warp 0 walks them in ascending order, accumulating score_exp(z_j - m_t), to the column.
__global__ void __launch_bounds__(32 * kScoreWarps) sample_step_kernel(ScoreStepArgs a) {
  __shared__ float mx[kScoreWarps][32];
  __shared__ double sm[kScoreWarps][32];
  __shared__ float z[32][kScoreStrip + 1];
  __shared__ int strip_of[32];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int b = blockIdx.x * 32 + lane;
  const int B = a.B;
  pdl_launch_dependents();
  pdl_wait();
  const float ninf = -__int_as_float(0x7f800000);
  const float M = reduce_partials(a.partials, B, a.N, b, lane, w, mx, sm);
  const int n_strips = (a.N + kScoreStrip - 1) / kScoreStrip;
  const int per = (n_strips + kScoreWarps - 1) / kScoreWarps;
  double S = 0.0, r = 0.0;  // r: the target left over inside the chosen strip, in units of its exp(m_t - M)
  float m_t = 0.0f;
  if (w == 0) {
    int t = -1;
    if (b < B) {
      for (int k = 0; k < kScoreWarps; k++) S += sm[k][lane];
      const uint64_t key = a.keys ? a.keys[b] : static_cast<uint64_t>(b);
      const double target = sample_uniform(a.seed, key, static_cast<uint32_t>(a.step)) * S;
      double acc = 0.0, before = 0.0;
      int g = -1;
      for (int k = 0; k < kScoreWarps; k++) {
        const double v = sm[k][lane];
        if (v == 0.0) continue;
        g = k, before = acc;
        acc += v;
        if (acc > target) break;
      }
      const double tg = target - before;
      acc = 0.0, before = 0.0;
      const int t0 = g * per, t1 = min(n_strips, t0 + per);
      for (int tt = t0; tt < t1; tt++) {
        const float2 p = a.partials[static_cast<size_t>(tt) * B + b];
        const float e = score_exp(__fsub_rn(p.x, M));
        const double v = static_cast<double>(p.y) * static_cast<double>(e);
        if (v == 0.0) continue;
        t = tt, before = acc, m_t = p.x;
        r = static_cast<double>(e);
        acc += v;
        if (acc > tg) break;
      }
      r = (tg - before) / r;
    }
    strip_of[lane] = t;
  }
  __syncthreads();
  {  // thread (w, lane): columns 2w and 2w + 1 of row lane's strip
    const int t = strip_of[lane];
    for (int j = 2 * w; j < 2 * w + 2; j++) {
      const int col = t * kScoreStrip + j;
      float v = ninf;
      if (t >= 0 && col < a.N)
        v = __fmul_rn(a.logits ? a.logits[static_cast<size_t>(b) * a.N + col] : exact_logit(a, b, col), a.inv_t);
      z[lane][j] = v;
    }
  }
  __syncthreads();
  if (w != 0 || b >= B) return;
  const int t = strip_of[lane];
  double acc = 0.0;
  int c = -1;
  for (int j = 0; j < kScoreStrip; j++) {
    const float e = score_exp(__fsub_rn(z[lane][j], m_t));
    if (e == 0.0f) continue;
    c = j;
    acc += static_cast<double>(e);
    if (acc > r) break;
  }
  const float zc = z[lane][c];
  a.best[b] = pack_best(zc, static_cast<uint32_t>(t * kScoreStrip + c));
  if (a.scores)
    a.scores[static_cast<size_t>(a.step) * B + b] =
        static_cast<float>(static_cast<double>(zc) - (static_cast<double>(M) + log(S)));
}

// ------------------------------------------------------------------ top-k sampling
// One block per row over the row's logits [N] (include/slimt_b200.h, DESIGN §4.4e).  S_k, the first min(k, N) columns
// by (y descending, column ascending), is the set of columns whose 32-bit order key (pack_best's high word) lies above
// a threshold key, plus the first columns equal to it.  The threshold comes from a radix select over the key in three
// digits (12, 10, 10 bits); each digit's histogram is built with shared-memory atomics, whose counts do not depend on
// their order.  After the first digit, every column at or above the boundary bin is compacted, in column order, into a
// shared buffer when it fits there, and the later digits and the final compaction read that buffer instead of the row.
constexpr int kTopkThreads = 512;
constexpr int kTopkStage = 2048;  // staged columns
constexpr int kTopkBins = 4096;   // bins of the first digit

__device__ __forceinline__ uint32_t order_key(float y) { return static_cast<uint32_t>(pack_best(y, 0u) >> 32); }

// Exclusive prefix sum of v over the block's threads in thread order; total receives the block's sum.  Every thread
// calls it.
__device__ __forceinline__ int block_exclusive_scan(int v, int* ws, int& total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = kTopkThreads / 32;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) ws[w] = x;
  __syncthreads();
  if (w == 0) {
    int s = lane < nw ? ws[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, o);
      if (lane >= o) s += y;
    }
    ws[lane] = s;
  }
  __syncthreads();
  const int before = (w > 0 ? ws[w - 1] : 0) + x - v;
  total = ws[nw - 1];
  __syncthreads();
  return before;
}

// The row's columns in ascending order: four consecutive columns per thread and round, float4 loads (N % 8 == 0).
struct TopkRow {
  const float* y;
  int n;
  __device__ __forceinline__ void load4(int i, float (&v)[4], uint32_t (&c)[4]) const {
    const float4 q = *reinterpret_cast<const float4*>(y + i);
    v[0] = q.x, v[1] = q.y, v[2] = q.z, v[3] = q.w;
#pragma unroll
    for (int j = 0; j < 4; j++) c[j] = static_cast<uint32_t>(i + j);
  }
};
// The staged columns, still in ascending order.
struct TopkStaged {
  const float* y;
  const uint32_t* col;
  int n;
  __device__ __forceinline__ void load4(int i, float (&v)[4], uint32_t (&c)[4]) const {
#pragma unroll
    for (int j = 0; j < 4; j++) v[j] = i + j < n ? y[i + j] : 0.0f, c[j] = i + j < n ? col[i + j] : 0u;
  }
};

// Calls f(valid, value, column, key) for every element of src, four per thread and round, every thread the same
// number of times (so f may hold block barriers).
template <class Src, class F>
__device__ __forceinline__ void topk_rounds(const Src& src, F&& f) {
  for (int base = 0; base < src.n; base += 4 * kTopkThreads) {
    const int i = base + 4 * static_cast<int>(threadIdx.x);
    float v[4] = {0.0f, 0.0f, 0.0f, 0.0f};
    uint32_t c[4] = {0u, 0u, 0u, 0u};
    if (i < src.n) src.load4(i, v, c);
    bool ok[4];
    uint32_t key[4];
#pragma unroll
    for (int j = 0; j < 4; j++) ok[j] = i + j < src.n, key[j] = order_key(v[j]);
    f(ok, v, c, key);
  }
}

struct TopkSelect {
  uint32_t prefix, mask;  // the candidates: keys with (key & mask) == prefix
  int need;               // how many of the candidates belong to S_k
};

// One digit of the radix select: the histogram of bits [shift, shift + log2(bins)) over the candidates, and the bin in
// which the need-th largest candidate lies.  The candidates in higher bins all belong to S_k.
template <class Src>
__device__ void topk_digit(const Src& src, int shift, int bins, TopkSelect& s, int* hist, int* ws, int* found) {
  for (int i = threadIdx.x; i < bins; i += kTopkThreads) hist[i] = 0;
  __syncthreads();
  const uint32_t prefix = s.prefix, mask = s.mask, dmask = static_cast<uint32_t>(bins - 1);
  topk_rounds(src, [&](const bool (&ok)[4], const float (&)[4], const uint32_t (&)[4], const uint32_t (&key)[4]) {
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (ok[j] && (key[j] & mask) == prefix) atomicAdd(&hist[(key[j] >> shift) & dmask], 1);
  });
  __syncthreads();
  // thread t owns the chunk of bins kTopkThreads - 1 - t, so its exclusive scan is the count in higher bins
  const int per = bins / kTopkThreads, first = (kTopkThreads - 1 - static_cast<int>(threadIdx.x)) * per;
  int local = 0;
  for (int k = 0; k < per; k++) local += hist[first + k];
  int total;
  int above = block_exclusive_scan(local, ws, total);
  if (above < s.need && above + local >= s.need)
    for (int k = per - 1; k >= 0; k--) {
      if (above + hist[first + k] >= s.need) {
        found[0] = first + k, found[1] = above;
        break;
      }
      above += hist[first + k];
    }
  __syncthreads();
  s.prefix |= static_cast<uint32_t>(found[0]) << shift, s.mask |= dmask << shift, s.need -= found[1];
  __syncthreads();
}

// The last two digits over src, then S_k in ascending column order into (sy, sc): every column whose key is above
// the threshold, and the first `need` columns equal to it.  Returns |S_k|.
template <class Src>
__device__ int topk_finish(const Src& src, TopkSelect s, int* hist, int* ws, int* found, float* sy, uint32_t* sc) {
  topk_digit(src, 10, 1024, s, hist, ws, found);
  topk_digit(src, 0, 1024, s, hist, ws, found);
  const uint32_t thr = s.prefix;
  int eq_before = 0, out_before = 0;
  topk_rounds(src, [&](const bool (&ok)[4], const float (&v)[4], const uint32_t (&c)[4], const uint32_t (&key)[4]) {
    int n_eq = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) n_eq += ok[j] && key[j] == thr;
    int eq_total;
    int rank = eq_before + block_exclusive_scan(n_eq, ws, eq_total);
    bool in[4];
    int n_in = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const bool eq = ok[j] && key[j] == thr;
      in[j] = ok[j] && (key[j] > thr || (eq && rank < s.need));
      rank += eq;
      n_in += in[j];
    }
    int in_total;
    int pos = out_before + block_exclusive_scan(n_in, ws, in_total);
#pragma unroll
    for (int j = 0; j < 4; j++)
      if (in[j]) sy[pos] = v[j], sc[pos] = c[j], pos++;
    eq_before += eq_total, out_before += in_total;
  });
  return out_before;
}

// Per row: S_k (above), then warp 0 tempers its logits and their maximum M, every thread one term score_exp(z - M), and
// thread 0 sums the terms in ascending column order in double, draws u * S and walks the running sum to the word.
__global__ void __launch_bounds__(kTopkThreads) topk_sample_kernel(ScoreStepArgs a, int top_k) {
  __shared__ int hist[kTopkBins];
  __shared__ float stage_y[kTopkStage];
  __shared__ uint32_t stage_c[kTopkStage];
  __shared__ float sy[kMaxTopK], se[kMaxTopK];
  __shared__ uint32_t sc[kMaxTopK];
  __shared__ int ws[32], found[2];
  __shared__ float m_all;
  const int b = blockIdx.x, N = a.N;
  pdl_launch_dependents();
  pdl_wait();
  const TopkRow row{a.logits + static_cast<size_t>(b) * N, N};
  TopkSelect s{0u, 0u, min(top_k, N)};
  topk_digit(row, 20, kTopkBins, s, hist, ws, found);
  // the columns in bins at or above the boundary: those above it and the boundary bin's own
  const int first_bin = static_cast<int>(s.prefix >> 20);
  int staged = 0;
  for (int i = threadIdx.x; i < kTopkBins; i += kTopkThreads) staged += i >= first_bin ? hist[i] : 0;
  int n_stage;
  block_exclusive_scan(staged, ws, n_stage);
  int n;
  if (n_stage <= kTopkStage) {
    int out_before = 0;
    topk_rounds(row, [&](const bool (&ok)[4], const float (&v)[4], const uint32_t (&c)[4], const uint32_t (&key)[4]) {
      bool in[4];
      int n_in = 0;
#pragma unroll
      for (int j = 0; j < 4; j++) in[j] = ok[j] && static_cast<int>(key[j] >> 20) >= first_bin, n_in += in[j];
      int in_total;
      int pos = out_before + block_exclusive_scan(n_in, ws, in_total);
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (in[j]) stage_y[pos] = v[j], stage_c[pos] = c[j], pos++;
      out_before += in_total;
    });
    __syncthreads();
    n = topk_finish(TopkStaged{stage_y, stage_c, n_stage}, s, hist, ws, found, sy, sc);
  } else {  // many equal or nearly equal logits: the later digits read the row again
    n = topk_finish(row, s, hist, ws, found, sy, sc);
  }
  __syncthreads();
  const int t = threadIdx.x;
  const float z = t < n ? __fmul_rn(sy[t], a.inv_t) : -__int_as_float(0x7f800000);
  if (t < 32) {
    float m = z;
    for (int i = t + 32; i < n; i += 32) m = fmaxf(m, __fmul_rn(sy[i], a.inv_t));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (t == 0) m_all = m;
  }
  __syncthreads();
  const float M = m_all;
  if (t < n) se[t] = score_exp(__fsub_rn(z, M));
  __syncthreads();
  if (t != 0) return;
  double S = 0.0;
  for (int i = 0; i < n; i++) S += static_cast<double>(se[i]);
  const uint64_t key = a.keys ? a.keys[b] : static_cast<uint64_t>(b);
  const double target = sample_uniform(a.seed, key, static_cast<uint32_t>(a.step)) * S;
  double acc = 0.0;
  int c = -1;
  for (int i = 0; i < n; i++) {
    if (se[i] == 0.0f) continue;
    c = i;
    acc += static_cast<double>(se[i]);
    if (acc > target) break;
  }
  const float zc = __fmul_rn(sy[c], a.inv_t);
  a.best[b] = pack_best(zc, sc[c]);
  if (a.scores)
    a.scores[static_cast<size_t>(a.step) * a.B + b] =
        static_cast<float>(static_cast<double>(zc) - (static_cast<double>(M) + log(S)));
}

// ------------------------------------------------------------------ beam search
// Candidates are packed as in packed_best.cuh, so a larger key ranks first and equal values go to the lower index.
// top[0..7] holds the largest keys seen, descending (0 = empty); keys are distinct.
__device__ __forceinline__ void top8_insert(unsigned long long (&top)[kMaxBeam], unsigned long long key) {
#pragma unroll
  for (int i = kMaxBeam - 1; i >= 0; i--) {
    const unsigned long long prev = i > 0 ? top[i - 1] : ~0ull;
    if (key > top[i]) top[i] = key < prev ? key : prev;
  }
}

__device__ __forceinline__ unsigned long long warp_max_u64(unsigned long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long u = __shfl_xor_sync(0xffffffffu, v, o);
    v = u > v ? u : v;
  }
  return v;
}

// The warp's largest key over every lane's top list, removed from the list that held it.
__device__ __forceinline__ unsigned long long top8_pop(unsigned long long (&top)[kMaxBeam]) {
  const unsigned long long m = warp_max_u64(top[0]);
  if (m != 0ull && top[0] == m) {
#pragma unroll
    for (int i = 0; i + 1 < kMaxBeam; i++) top[i] = top[i + 1];
    top[kMaxBeam - 1] = 0ull;
  }
  return m;
}

// Block = 32 rows x 32 warps, reduce_partials' shape; then warp w takes row w of the block.
__global__ void __launch_bounds__(32 * kScoreWarps) beam_topk_kernel(BeamStepArgs a) {
  __shared__ float mx[kScoreWarps][32];
  __shared__ double sm[kScoreWarps][32];
  __shared__ double lse_of[32];
  const ScoreStepArgs& s = a.s;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int rows = s.B, K = a.beam;
  pdl_launch_dependents();
  pdl_wait();
  const float M = reduce_partials(s.partials, rows, s.N, blockIdx.x * 32 + lane, lane, w, mx, sm);
  if (w == 0) {
    double S = 0.0;
    for (int k = 0; k < kScoreWarps; k++) S += sm[k][lane];
    lse_of[lane] = static_cast<double>(M) + log(S);
    if (blockIdx.x * 32 + lane < rows) s.best[blockIdx.x * 32 + lane] = 0ull;  // the output GEMM's greedy slot, unused
  }
  __syncthreads();
  const int row = blockIdx.x * 32 + w;
  if (row >= rows) return;
  const int b = row / K, slot = row % K;
  if (slot >= (a.step == 0 ? 1 : static_cast<int>(a.width[b]))) return;
  // the K strips of largest (max, -strip)
  const int n_strips = (s.N + kScoreStrip - 1) / kScoreStrip;
  unsigned long long top[kMaxBeam];
#pragma unroll
  for (int i = 0; i < kMaxBeam; i++) top[i] = 0ull;
  for (int t = lane; t < n_strips; t += 32)
    top8_insert(top, pack_best(s.partials[static_cast<size_t>(t) * rows + row].x, static_cast<uint32_t>(t)));
  int my_strip = -1;  // lane r < K: the r-th strip
  for (int r = 0; r < K; r++) {
    const unsigned long long m = top8_pop(top);
    if (lane == r && m != 0ull) my_strip = static_cast<int>(best_index(m));
  }
  // their 64 * K logits, exactly: lane takes columns lane and lane + 32 of each strip
  const float ninf = -__int_as_float(0x7f800000);
#pragma unroll
  for (int i = 0; i < kMaxBeam; i++) top[i] = 0ull;
  for (int i = 0; i < 2 * K; i++) {
    const int t = __shfl_sync(0xffffffffu, my_strip, i >> 1);
    if (t < 0) break;
    const int col = t * kScoreStrip + lane + 32 * (i & 1);
    top8_insert(top, pack_best(col < s.N ? exact_logit(s, row, col) : ninf, static_cast<uint32_t>(col)));
  }
  const double lse = lse_of[w];
  for (int r = 0; r < K; r++) {
    const unsigned long long m = top8_pop(top);
    if (lane == 0)
      a.cand[static_cast<size_t>(row) * K + r] =
          BeamCand{best_index(m), static_cast<float>(static_cast<double>(best_value(m)) - lse)};
  }
}

// Warp = one sentence, eight per block.  Every lane computes the same choices; lane 0 writes the records.
__global__ void __launch_bounds__(256) beam_merge_kernel(BeamStepArgs a) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * 8 + (threadIdx.x >> 5);
  pdl_launch_dependents();
  pdl_wait();
  if (b >= a.n_sent) return;
  const int K = a.beam, width = a.width[b];
  if (width == 0) return;
  const int live = a.step == 0 ? 1 : width, base = b * K;
  // candidate i = slot * K + rank of the live slots: lanes hold i = lane and lane + 32
  auto key_of = [&](int i) -> unsigned long long {
    if (i >= live * K) return 0ull;
    const float t = __fadd_rn(a.cum[base + i / K], a.cand[static_cast<size_t>(base) * K + i].score);
    return pack_best(t, static_cast<uint32_t>(i));
  };
  unsigned long long k0 = key_of(lane), k1 = key_of(lane + 32);
  int pick[kMaxBeam];
  float total[kMaxBeam];
#pragma unroll
  for (int r = 0; r < kMaxBeam; r++) {
    if (r >= width) break;
    const unsigned long long m = warp_max_u64(k0 > k1 ? k0 : k1);
    if (k0 == m) k0 = 0ull;
    if (k1 == m) k1 = 0ull;
    pick[r] = static_cast<int>(best_index(m));
    total[r] = __fadd_rn(a.cum[base + pick[r] / K], a.cand[static_cast<size_t>(base) * K + pick[r]].score);
  }
  __syncwarp();  // every lane has read cum before it is rewritten
  const size_t rows = static_cast<size_t>(a.n_sent) * K;
  int n_live = 0, n_fin = K - width;
  int parent[kMaxBeam];
  uint32_t word[kMaxBeam];
#pragma unroll
  for (int r = 0; r < kMaxBeam; r++) {
    if (r >= width) break;
    const int k = pick[r] / K;
    const BeamCand c = a.cand[static_cast<size_t>(base) * K + pick[r]];
    const uint32_t wd = a.s.shortlist ? a.s.shortlist[c.col] : c.col;
    if (wd == a.eos_id || a.step == a.last_step) {
      if (lane == 0)
        a.fin[base + n_fin] = BeamFin{static_cast<uint32_t>(a.step), static_cast<uint32_t>(k), wd, c.score, total[r]};
      n_fin++;
    } else {
      if (lane == 0) {
        a.rec[static_cast<size_t>(a.step) * rows + base + n_live] = BeamRec{wd, static_cast<uint32_t>(k), c.score};
        a.cum[base + n_live] = total[r];
      }
      parent[n_live] = k, word[n_live] = wd;
      n_live++;
    }
  }
  if (lane == 0) {
    a.width[b] = static_cast<uint8_t>(n_live);
    if (n_live == 0) atomicAdd(a.n_done, 1);
  }
  const int E = a.E;
#pragma unroll
  for (int n = 0; n < kMaxBeam; n++) {
    if (n >= n_live) break;
    const size_t dst = static_cast<size_t>(base + n) * E, src = static_cast<size_t>(base + parent[n]) * E;
    for (int l = 0; l < a.Ld; l++)
      for (int e = lane * 4; e < E; e += 128)
        *reinterpret_cast<float4*>(a.state_nxt[l] + dst + e) = *reinterpret_cast<const float4*>(a.state_cur[l] + src + e);
    for (int e = lane * 4; e < E; e += 128) {
      const char4 c = *reinterpret_cast<const char4*>(a.emb_q + static_cast<size_t>(word[n]) * E + e);
      const float4 ps = *reinterpret_cast<const float4*>(a.pos0 + e);
      const float y[4] = {embed1(c.x, a.inv_qm, a.sqrt_e, ps.x), embed1(c.y, a.inv_qm, a.sqrt_e, ps.y),
                          embed1(c.z, a.inv_qm, a.sqrt_e, ps.z), embed1(c.w, a.inv_qm, a.sqrt_e, ps.w)};
      *reinterpret_cast<float4*>(a.x + dst + e) = make_float4(y[0], y[1], y[2], y[3]);
      store_quant4(a.q, dst + e, y);
    }
  }
}

}  // namespace

void launch_embed(const uint32_t* tokens, const int8_t* emb_q, float inv_qm, float sqrt_e, const float* pos, int rows,
                  int T, int E, int pos_from_row, int zero_embed, float* x, QuantOuts q, cudaStream_t stream, int shift) {
  const size_t n = static_cast<size_t>(rows) * (E / 4);
  if (n == 0) return;
  embed_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(tokens, emb_q, inv_qm, sqrt_e, pos, rows, T, E,
                                                                         pos_from_row, zero_embed, shift, x, q);
}

void launch_quantize(const float* x, size_t n, QuantOuts q, cudaStream_t stream) {
  const size_t n4 = n / 4;
  if (n4 == 0) return;
  quantize_kernel<<<static_cast<unsigned>((n4 + 255) / 256), 256, 0, stream>>>(x, n4, q);
}

int launch_self_attention(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T, int H,
                          int dh, QuantOuts q, cudaStream_t stream) {
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
    self_attention_kernel<32><<<B * H, threads, smem, stream>>>(Q, K, V, lengths, T, H, dk, q);
  } else if (dh == 64) {
    ensure_dyn_smem(self_attention_kernel<64>, smem);
    self_attention_kernel<64><<<B * H, threads, smem, stream>>>(Q, K, V, lengths, T, H, dk, q);
  } else {
    return 1;  // the model loader only admits head sizes 32 and 64; reported through the error convention by the caller
  }
  return 0;
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

void launch_score_rows(const float* logits, int B, int N, float2* partials, float inv_t, cudaStream_t stream) {
  const size_t n = static_cast<size_t>((N + kScoreStrip - 1) / kScoreStrip) * B;
  if (n == 0) return;
  const unsigned grid = static_cast<unsigned>((n + 255) / 256);
  if (inv_t == 1.0f) score_rows_kernel<false><<<grid, 256, 0, stream>>>(logits, B, N, partials, inv_t);
  else score_rows_kernel<true><<<grid, 256, 0, stream>>>(logits, B, N, partials, inv_t);
}

int launch_score_step(const ScoreStepArgs& a, cudaStream_t stream) {
  if (a.B == 0) return 0;
  return launch_pdl(score_step_kernel, dim3((a.B + 31) / 32), dim3(32 * kScoreWarps), 0, stream, a) != cudaSuccess ? 1 : 0;
}

int launch_sample_step(const ScoreStepArgs& a, cudaStream_t stream) {
  if (a.B == 0) return 0;
  return launch_pdl(sample_step_kernel, dim3((a.B + 31) / 32), dim3(32 * kScoreWarps), 0, stream, a) != cudaSuccess ? 1 : 0;
}

int launch_topk_sample(const ScoreStepArgs& a, int top_k, cudaStream_t stream) {
  if (a.B == 0) return 0;
  if (top_k < 1 || top_k > kMaxTopK || a.logits == nullptr) return 1;
  return launch_pdl(topk_sample_kernel, dim3(a.B), dim3(kTopkThreads), 0, stream, a, top_k) != cudaSuccess ? 1 : 0;
}

int launch_beam_topk(const BeamStepArgs& a, cudaStream_t stream) {
  if (a.s.B == 0) return 0;
  if (a.beam < 1 || a.beam > kMaxBeam || a.Ld > 2) return 1;
  return launch_pdl(beam_topk_kernel, dim3((a.s.B + 31) / 32), dim3(32 * kScoreWarps), 0, stream, a) != cudaSuccess ? 1 : 0;
}

int launch_beam_merge(const BeamStepArgs& a, cudaStream_t stream) {
  if (a.n_sent == 0) return 0;
  if (a.beam < 1 || a.beam > kMaxBeam || a.Ld > 2) return 1;
  return launch_pdl(beam_merge_kernel, dim3((a.n_sent + 7) / 8), dim3(256), 0, stream, a) != cudaSuccess ? 1 : 0;
}

}  // namespace sb
