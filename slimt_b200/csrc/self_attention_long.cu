// Encoder self-attention on f32 Q, K, V for sentences too long for the tiled kernel (self_attention_tiled.cu), whose
// [64][T] score block and whole transposed K no longer fit shared memory beyond T ~ 558 (head size 32) / ~ 400 (64).
// Reference: scaled_dot_product_attention, slimt/Modules.cc:24-86; softmax slimt/TensorOps.cc:282-315.
//
// A block of 256 threads owns 32 query rows of one (sentence, head) and keeps their [32][T] score block in shared
// memory (128 KB at T = 1024); K and then V pass through one 128-key tile buffer.  The arithmetic is the tiled
// kernel's, operation for operation, so the two give the same bits:
//   scores   thread = 4 queries x 4 keys of a 128-key tile, each one fma chain over the head dimension in order, then
//            __fmul_rn(dk, .); Q and the K tile sit transposed ([d][row]) so one 16-byte load brings four rows.
//   softmax  row maxima by shuffle tree (order-free), exp elementwise (exact_math.cuh), the row sums as ONE chain per
//            row in key order (warp 0; the other warps stage the first V tile meanwhile), p = e / sum with the row's
//            reciprocal formed once (div_by_rcp).  No online rescaling: the softmax sees the whole row.
//   P V      thread = 1 query x (head size / 8) dims, one fma chain per output over the keys in order, carried across
//            the V tiles.
// Masked keys (>= the sentence's length) are skipped; padded query rows produce quantize(0).
// Bound: the score block is [32][round_up(T, 128) + 4] floats, which fits the 220 KB budget up to T = 1024.
#include <stdio.h>

#include "exact_math.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kLQB = 32;        // query rows per block
constexpr int kLKT = 128;       // keys per K / V tile
constexpr int kLThreads = 256;
constexpr int kLSQ = kLQB + 4;  // row stride of the transposed Q
constexpr int kLSK = kLKT + 4;  // row stride of the transposed K tile

size_t long_smem_bytes(int T, int dh) {
  const size_t kcap = (static_cast<size_t>(T) + kLKT - 1) / kLKT * kLKT;
  return (static_cast<size_t>(dh) * kLSQ + static_cast<size_t>(dh) * kLSK + kLQB * (kcap + 4) + 2 * kLQB) * sizeof(float);
}

template <int DH>
__global__ void __launch_bounds__(kLThreads, 1) self_attention_long_kernel(
    const float* __restrict__ Q, const float* __restrict__ K, const float* __restrict__ V,
    const uint32_t* __restrict__ lengths, int T, int H, int n_qb, float dk, float* __restrict__ out_f32, QuantOuts qo) {
  extern __shared__ __align__(16) float sm[];
  __shared__ uint64_t exp_tab[32];
  const int tid = threadIdx.x;
  const int qb = blockIdx.x % n_qb;
  const int bh = blockIdx.x / n_qb;
  const int b = bh / H, h = bh % H;
  const int E = H * DH;
  const int len = min(static_cast<int>(lengths[b]), T);
  const int i0 = qb * kLQB;
  const int SK = ((T + kLKT - 1) / kLKT) * kLKT + 4;  // row stride of S: every tile's stores land inside, 16-byte aligned
  float* Qt = sm;                     // [DH][kLSQ]
  float* Kt = Qt + DH * kLSQ;         // K tile [DH][kLSK]; later a V tile [kLKT][DH]
  float* S = Kt + DH * kLSK;          // [kLQB][SK]
  float* rmax = S + kLQB * SK;        // [kLQB]
  float* rsum = rmax + kLQB;          // [kLQB]
  if (tid < 32) exp_tab[tid] = kExp2fTab[tid];

  const size_t base = static_cast<size_t>(b) * T * E + static_cast<size_t>(h) * DH;
  const int rows_here = max(0, min(kLQB, len - i0));
  // V tile staging: keys jb .. jb + 127 below len, row-major [key][DH]
  auto stage_v = [&](int jb, int t0, int nt) {
    const int nk = min(kLKT, len - jb);
    for (int i = t0; i < nk * (DH / 4); i += nt) {
      const int j = i / (DH / 4), c = (i % (DH / 4)) * 4;
      *reinterpret_cast<float4*>(Kt + j * DH + c) = *reinterpret_cast<const float4*>(V + base + static_cast<size_t>(jb + j) * E + c);
    }
  };

  // P V outputs of this thread: query row pr, dims 4 dg + 32 g + (0..3) for g < DH / 32
  constexpr int NG = DH / 32;
  const int pr = tid >> 3, dg = tid & 7;
  float acc[NG][4];
#pragma unroll
  for (int g = 0; g < NG; g++)
#pragma unroll
    for (int k = 0; k < 4; k++) acc[g][k] = 0.0f;

  if (rows_here > 0) {
    // ---- stage Q (this block's rows), transposed; zero beyond the valid rows
    for (int i = tid; i < kLQB * (DH / 4); i += kLThreads) {
      const int r = i / (DH / 4), c = (i % (DH / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows_here) v = *reinterpret_cast<const float4*>(Q + base + static_cast<size_t>(i0 + r) * E + c);
      Qt[(c + 0) * kLSQ + r] = v.x, Qt[(c + 1) * kLSQ + r] = v.y, Qt[(c + 2) * kLSQ + r] = v.z, Qt[(c + 3) * kLSQ + r] = v.w;
    }

    // ---- scores: S[i][j] = dk * (q_i . k_j), each a sequential fma chain over d, one 128-key tile at a time
    const int ty = tid >> 5, tx = tid & 31;  // queries 4 ty .. 4 ty + 3; keys 4 tx .. 4 tx + 3 of the tile
    for (int jb = 0; jb < len; jb += kLKT) {
      __syncthreads();  // the previous tile's readers are done (first pass: Q is staged by the loop below's barrier)
      for (int i = tid; i < kLKT * (DH / 4); i += kLThreads) {
        const int j = i / (DH / 4), c = (i % (DH / 4)) * 4;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (jb + j < len) v = *reinterpret_cast<const float4*>(K + base + static_cast<size_t>(jb + j) * E + c);
        Kt[(c + 0) * kLSK + j] = v.x, Kt[(c + 1) * kLSK + j] = v.y, Kt[(c + 2) * kLSK + j] = v.z, Kt[(c + 3) * kLSK + j] = v.w;
      }
      __syncthreads();
      float a[4][4];
#pragma unroll
      for (int u = 0; u < 4; u++)
#pragma unroll
        for (int w = 0; w < 4; w++) a[u][w] = 0.0f;
#pragma unroll 4
      for (int d = 0; d < DH; d++) {
        const float4 q4 = *reinterpret_cast<const float4*>(Qt + d * kLSQ + 4 * ty);
        const float4 k4 = *reinterpret_cast<const float4*>(Kt + d * kLSK + 4 * tx);
        const float qv[4] = {q4.x, q4.y, q4.z, q4.w};
        const float kv[4] = {k4.x, k4.y, k4.z, k4.w};
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
          for (int w = 0; w < 4; w++) a[u][w] = fmaf(qv[u], kv[w], a[u][w]);
      }
#pragma unroll
      for (int u = 0; u < 4; u++)
        *reinterpret_cast<float4*>(S + (4 * ty + u) * SK + jb + 4 * tx) =
            make_float4(__fmul_rn(dk, a[u][0]), __fmul_rn(dk, a[u][1]), __fmul_rn(dk, a[u][2]), __fmul_rn(dk, a[u][3]));
    }
    __syncthreads();

    // ---- row maxima over the valid keys: eight threads per row, shuffle tree
    {
      const int r = tid >> 3, part = tid & 7;
      float mx = -3.402823466e+38f;
      for (int j = part; j < len; j += 8) mx = fmaxf(mx, S[r * SK + j]);
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
      if (part == 0) rmax[r] = mx;
    }
    __syncthreads();
    // ---- e = exp(s - max), elementwise
    {
      const int r = tid >> 3, part = tid & 7;
      const float mx = rmax[r];
      if (r < rows_here)
        for (int j = part; j < len; j += 8) S[r * SK + j] = expf_glibc_nonpos_tab(__fsub_rn(S[r * SK + j], mx), exp_tab);
    }
    __syncthreads();
    // ---- row sums in key order (warp 0, one chain per row) while the other warps stage the first V tile (K is dead)
    if (tid < kLQB) {
      if (tid < rows_here) {
        const float* srow = S + tid * SK;
        float sum = 0.0f;
        int j = 0;
        for (; j + 4 <= len; j += 4) {
          const float4 e4 = *reinterpret_cast<const float4*>(srow + j);
          sum = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(sum, e4.x), e4.y), e4.z), e4.w);
        }
        for (; j < len; j++) sum = __fadd_rn(sum, srow[j]);
        rsum[tid] = sum;
      }
    } else {
      stage_v(0, tid - kLQB, kLThreads - kLQB);
    }
    __syncthreads();
    // ---- p = e / sum, elementwise
    {
      const int r = tid >> 3, part = tid & 7;
      if (r < rows_here) {
        const float sum = rsum[r];
        const float rc = rcp_refined(sum), lo = div_guard_lo(sum);
        for (int j = part; j < len; j += 8) S[r * SK + j] = div_by_rcp(S[r * SK + j], sum, rc, lo);
      }
    }
    __syncthreads();

    // ---- P V, one 128-key V tile at a time (tile 0 is already staged)
    for (int jb = 0; jb < len; jb += kLKT) {
      if (jb > 0) {
        __syncthreads();
        stage_v(jb, tid, kLThreads);
        __syncthreads();
      }
      if (pr < rows_here) {
        const float* prow = S + pr * SK + jb;
        const int nk = min(kLKT, len - jb);
        int j = 0;
        for (; j + 4 <= nk; j += 4) {
          const float4 p4 = *reinterpret_cast<const float4*>(prow + j);
          const float pv[4] = {p4.x, p4.y, p4.z, p4.w};
#pragma unroll
          for (int e = 0; e < 4; e++) {
#pragma unroll
            for (int g = 0; g < NG; g++) {
              const float4 v4 = *reinterpret_cast<const float4*>(Kt + (j + e) * DH + 32 * g + 4 * dg);
              acc[g][0] = fmaf(pv[e], v4.x, acc[g][0]);
              acc[g][1] = fmaf(pv[e], v4.y, acc[g][1]);
              acc[g][2] = fmaf(pv[e], v4.z, acc[g][2]);
              acc[g][3] = fmaf(pv[e], v4.w, acc[g][3]);
            }
          }
        }
        for (; j < nk; j++) {
          const float p = prow[j];
#pragma unroll
          for (int g = 0; g < NG; g++) {
            const float4 v4 = *reinterpret_cast<const float4*>(Kt + j * DH + 32 * g + 4 * dg);
            acc[g][0] = fmaf(p, v4.x, acc[g][0]);
            acc[g][1] = fmaf(p, v4.y, acc[g][1]);
            acc[g][2] = fmaf(p, v4.z, acc[g][2]);
            acc[g][3] = fmaf(p, v4.w, acc[g][3]);
          }
        }
      }
    }
  }

  // ---- outputs: padded query rows carry zeros
  const int i = i0 + pr;
  if (i >= T) return;
  const bool live = pr < rows_here;
#pragma unroll
  for (int g = 0; g < NG; g++) {
    const size_t off = base + static_cast<size_t>(i) * E + 32 * g + 4 * dg;
    float y[4];
#pragma unroll
    for (int k = 0; k < 4; k++) y[k] = live ? acc[g][k] : 0.0f;
    if (out_f32) *reinterpret_cast<float4*>(out_f32 + off) = make_float4(y[0], y[1], y[2], y[3]);
    for (int k = 0; k < qo.n; k++) {
      const float aq = qo.aq[k];
      *reinterpret_cast<uint32_t*>(qo.ptr[k] + off) = pack4(quantize1(y[0], aq), quantize1(y[1], aq), quantize1(y[2], aq), quantize1(y[3], aq));
    }
  }
}

}  // namespace

bool self_attention_long_supported(int T, int dh) {
  return (dh == 32 || dh == 64) && T >= 1 && long_smem_bytes(T, dh) <= 220 * 1024;
}

int launch_self_attention_long(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T, int H,
                               int dh, float* out_f32, QuantOuts q, cudaStream_t stream) {
  if (B == 0) return 0;
  if (!self_attention_long_supported(T, dh)) return 1;
  // 1/sqrt(dim_head) evaluated in double then narrowed, as `1.0F / std::sqrt(size_t)` does (Modules.cc:43)
  const float dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
  const int n_qb = (T + kLQB - 1) / kLQB;
  const size_t smem = long_smem_bytes(T, dh);
  const long blocks = static_cast<long>(B) * H * n_qb;
  if (blocks > 0x7fffffffL) return 1;
  if (dh == 32) {
    if (ensure_dyn_smem(self_attention_long_kernel<32>, smem) != cudaSuccess) return 1;
    self_attention_long_kernel<32><<<static_cast<unsigned>(blocks), kLThreads, smem, stream>>>(Q, K, V, lengths, T, H, n_qb, dk, out_f32, q);
  } else {
    if (ensure_dyn_smem(self_attention_long_kernel<64>, smem) != cudaSuccess) return 1;
    self_attention_long_kernel<64><<<static_cast<unsigned>(blocks), kLThreads, smem, stream>>>(Q, K, V, lengths, T, H, n_qb, dk, out_f32, q);
  }
  return 0;
}

}  // namespace sb
