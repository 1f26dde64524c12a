// Encoder self-attention on f32 Q, K, V for the shapes the fused kernel (enc_attention.cu) does not take: sentences
// longer than 64 tokens and head size 64 (reference: scaled_dot_product_attention, slimt/Modules.cc:24-86, with
// split_heads / join_heads :88-143 folded into the addressing; softmax slimt/TensorOps.cc:282-315).
//
// The first kernel for these shapes (self_attention_kernel in kernels.cu, kept as SLIMT_B200_SELFATTN=rowwise) gave each
// query row to one thread: every K and V element a thread needs then arrives as a broadcast shared-memory load that
// feeds four FMAs, the score row of every thread lives in shared memory (131 KB at T = 256), and one block of four
// warps fills an SM.  It ran at 3 % of the HBM roofline and took 28 % of the mixed-length workload.
//
// Here a block of 256 threads owns 64 query rows of one (sentence, head) and works like a register-tiled SGEMM whose
// every output is still accumulated by ONE thread in index order, so each dot product is the reference's sequential
// fma chain and nothing is re-associated:
//   scores   thread = 4 queries x 8 keys per 128-key tile; Q and K sit transposed in shared memory ([d][row]) so that
//            one 16-byte load brings four rows' values of a dimension: 32 FMAs per three loads instead of 4 per one.
//   softmax  row maxima by shuffle tree (a maximum does not depend on order), exp elementwise over the 64 x T block by
//            all threads, the row sums as one sequential chain per row in key order (64 threads; the other warps load V
//            meanwhile), p = e / sum elementwise (the row's reciprocal formed once, exact_math.cuh: div_by_rcp).
//   P V      thread = 2 queries x 4 dims (x 8 for head size 64), one fma chain per output over the keys in order.
// Masked keys (>= the sentence's length) contribute exactly +0 in the reference (exp(-99999999 + s) underflows to 0), so
// they are skipped; padded query rows produce quantize(0) like the row-wise kernel.
#include <stdio.h>

#include "exact_math.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kQB = 64;        // query rows per block
constexpr int kTThreads = 256;

template <int DH>
__global__ void __launch_bounds__(kTThreads) self_attention_tiled_kernel(
    const float* __restrict__ Q, const float* __restrict__ K, const float* __restrict__ V,
    const uint32_t* __restrict__ lengths, int T, int H, int n_qb, float dk, float* __restrict__ out_f32, QuantOuts qo) {
  extern __shared__ __align__(16) float sm[];
  __shared__ uint64_t exp_tab[32];
  const int tid = threadIdx.x, lane = tid & 31;
  const int qb = blockIdx.x % n_qb;
  const int bh = blockIdx.x / n_qb;
  const int b = bh / H, h = bh % H;
  const int E = H * DH;
  const int len = min(static_cast<int>(lengths[b]), T);
  const int i0 = qb * kQB;
  const int Tk = (T + 3) & ~3;      // key capacity of the tile buffers (multiple of 4)
  const int SK = Tk + 4;            // row stride of S and of the transposed K: keeps 16-byte alignment
  constexpr int SQ = kQB + 4;       // row stride of the transposed Q
  float* Qt = sm;                                  // [DH][SQ]
  float* Kt = Qt + DH * SQ;                        // [DH][SK], later V as [Tk][DH]
  const int kv_floats = DH * SK > Tk * DH ? DH * SK : Tk * DH;
  float* S = Kt + kv_floats;                       // [kQB][SK]
  float* rmax = S + kQB * SK;                      // [kQB]
  float* rsum = rmax + kQB;                        // [kQB]
  if (tid < 32) exp_tab[tid] = kExp2fTab[tid];

  const size_t base = static_cast<size_t>(b) * T * E + static_cast<size_t>(h) * DH;
  const int rows_here = max(0, min(kQB, len - i0));  // valid query rows of this block

  if (rows_here > 0) {
    // ---- stage Q (this block's rows) and K (the sentence's valid keys), transposed; zero beyond the valid range
    for (int i = tid; i < kQB * (DH / 4); i += kTThreads) {
      const int r = i / (DH / 4), c = (i % (DH / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < rows_here) v = *reinterpret_cast<const float4*>(Q + base + static_cast<size_t>(i0 + r) * E + c);
      Qt[(c + 0) * SQ + r] = v.x, Qt[(c + 1) * SQ + r] = v.y, Qt[(c + 2) * SQ + r] = v.z, Qt[(c + 3) * SQ + r] = v.w;
    }
    const int kcap = (len + 127) & ~127;  // keys the score loop touches: whole 128-key tiles (capped by Tk below)
    for (int i = tid; i < min(kcap, Tk) * (DH / 4); i += kTThreads) {
      const int j = i / (DH / 4), c = (i % (DH / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j < len) v = *reinterpret_cast<const float4*>(K + base + static_cast<size_t>(j) * E + c);
      Kt[(c + 0) * SK + j] = v.x, Kt[(c + 1) * SK + j] = v.y, Kt[(c + 2) * SK + j] = v.z, Kt[(c + 3) * SK + j] = v.w;
    }
    __syncthreads();

    // ---- scores: S[i][j] = dk * (q_i . k_j), each a sequential fma chain over d
    {
      const int ty = tid >> 4, tx = tid & 15;  // queries 4 ty .. 4 ty + 3; keys 4 tx .. + 3 of each 64-key half tile
      for (int jb = 0; jb < len; jb += 128) {
        const int ja = jb + 4 * tx, jc = ja + 64;
        const bool second = jc < Tk;
        float acc[4][8];
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
          for (int w = 0; w < 8; w++) acc[u][w] = 0.0f;
        if (ja < Tk) {
#pragma unroll 4
          for (int d = 0; d < DH; d++) {
            const float4 q4 = *reinterpret_cast<const float4*>(Qt + d * SQ + 4 * ty);
            const float4 ka = *reinterpret_cast<const float4*>(Kt + d * SK + ja);
            const float4 kc = second ? *reinterpret_cast<const float4*>(Kt + d * SK + jc) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float qv[4] = {q4.x, q4.y, q4.z, q4.w};
            const float kv[8] = {ka.x, ka.y, ka.z, ka.w, kc.x, kc.y, kc.z, kc.w};
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
              for (int w = 0; w < 8; w++) acc[u][w] = fmaf(qv[u], kv[w], acc[u][w]);
          }
#pragma unroll
          for (int u = 0; u < 4; u++) {
            float* srow = S + (4 * ty + u) * SK;
            *reinterpret_cast<float4*>(srow + ja) = make_float4(__fmul_rn(dk, acc[u][0]), __fmul_rn(dk, acc[u][1]),
                                                                 __fmul_rn(dk, acc[u][2]), __fmul_rn(dk, acc[u][3]));
            if (second)
              *reinterpret_cast<float4*>(srow + jc) = make_float4(__fmul_rn(dk, acc[u][4]), __fmul_rn(dk, acc[u][5]),
                                                                   __fmul_rn(dk, acc[u][6]), __fmul_rn(dk, acc[u][7]));
          }
        }
      }
    }
    __syncthreads();

    // ---- row maxima over the valid keys: four threads per row, shuffle tree
    {
      const int r = tid >> 2, part = tid & 3;
      float mx = -3.402823466e+38f;
      for (int j = part; j < len; j += 4) mx = fmaxf(mx, S[r * SK + j]);
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
      if (part == 0) rmax[r] = mx;
    }
    __syncthreads();
    // ---- e = exp(s - max), elementwise (four threads per row, interleaved keys)
    {
      const int r = tid >> 2, part = tid & 3;
      const float mx = rmax[r];
      if (r < rows_here)
        for (int j = part; j < len; j += 4) S[r * SK + j] = expf_glibc_nonpos_tab(__fsub_rn(S[r * SK + j], mx), exp_tab);
    }
    __syncthreads();
    // ---- row sums in key order (threads 0..63, one chain each) while the other warps bring V in (K is dead)
    if (tid < kQB) {
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
      float* Vs = Kt;  // [len][DH]
      for (int i = tid - kQB; i < len * (DH / 4); i += kTThreads - kQB) {
        const int j = i / (DH / 4), c = (i % (DH / 4)) * 4;
        *reinterpret_cast<float4*>(Vs + j * DH + c) = *reinterpret_cast<const float4*>(V + base + static_cast<size_t>(j) * E + c);
      }
    }
    __syncthreads();
    // ---- p = e / sum, elementwise
    {
      const int r = tid >> 2, part = tid & 3;
      if (r < rows_here) {
        const float sum = rsum[r];
        const float rc = rcp_refined(sum), lo = div_guard_lo(sum);
        for (int j = part; j < len; j += 4) S[r * SK + j] = div_by_rcp(S[r * SK + j], sum, rc, lo);
      }
    }
    __syncthreads();
  }

  // ---- P V: thread = 2 queries x (DH / 8) dims... laid out as 32 query pairs x 8 dim groups
  {
    constexpr int DG = DH / 8;  // dims per thread: 4 (head size 32) or 8 (head size 64)
    const int pr = tid >> 3, dg = tid & 7;
    const int r0 = 2 * pr, d0 = dg * DG;
    float acc[2][DG];
#pragma unroll
    for (int u = 0; u < 2; u++)
#pragma unroll
      for (int w = 0; w < DG; w++) acc[u][w] = 0.0f;
    if (r0 < rows_here) {
      const float* Vs = Kt;
      const float* p0 = S + r0 * SK;
      const float* p1 = p0 + SK;
      for (int j = 0; j < len; j++) {
        const float a0 = p0[j], a1 = p1[j];
#pragma unroll
        for (int w = 0; w < DG; w += 4) {
          const float4 v4 = *reinterpret_cast<const float4*>(Vs + j * DH + d0 + w);
          acc[0][w] = fmaf(a0, v4.x, acc[0][w]), acc[1][w] = fmaf(a1, v4.x, acc[1][w]);
          acc[0][w + 1] = fmaf(a0, v4.y, acc[0][w + 1]), acc[1][w + 1] = fmaf(a1, v4.y, acc[1][w + 1]);
          acc[0][w + 2] = fmaf(a0, v4.z, acc[0][w + 2]), acc[1][w + 2] = fmaf(a1, v4.z, acc[1][w + 2]);
          acc[0][w + 3] = fmaf(a0, v4.w, acc[0][w + 3]), acc[1][w + 3] = fmaf(a1, v4.w, acc[1][w + 3]);
        }
      }
    }
#pragma unroll
    for (int u = 0; u < 2; u++) {
      const int i = i0 + r0 + u;
      if (i >= T) continue;
      const bool live = r0 + u < rows_here;  // padded query rows (and a row pair's odd tail) carry zeros
      const size_t off = base + static_cast<size_t>(i) * E + d0;
#pragma unroll
      for (int w = 0; w < DG; w += 4) {
        float y[4];
#pragma unroll
        for (int k = 0; k < 4; k++) y[k] = live ? acc[u][w + k] : 0.0f;
        if (out_f32) *reinterpret_cast<float4*>(out_f32 + off + w) = make_float4(y[0], y[1], y[2], y[3]);
        for (int k = 0; k < qo.n; k++) {
          const float aq = qo.aq[k];
          *reinterpret_cast<uint32_t*>(qo.ptr[k] + off + w) =
              pack4(quantize1(y[0], aq), quantize1(y[1], aq), quantize1(y[2], aq), quantize1(y[3], aq));
        }
      }
    }
  }
  (void)lane;
}

}  // namespace

namespace {
size_t tiled_smem_bytes(int T, int dh) {
  const int Tk = (T + 3) & ~3, SK = Tk + 4;
  const size_t kv = static_cast<size_t>(std::max(dh * SK, Tk * dh));
  return (static_cast<size_t>(dh) * (kQB + 4) + kv + static_cast<size_t>(kQB) * SK + 2 * kQB) * sizeof(float);
}
}  // namespace

bool self_attention_tiled_supported(int T, int dh) {
  return (dh == 32 || dh == 64) && T >= 1 && tiled_smem_bytes(T, dh) <= 220 * 1024;
}

int launch_self_attention_tiled(const float* Q, const float* K, const float* V, const uint32_t* lengths, int B, int T, int H,
                                int dh, float* out_f32, QuantOuts q, cudaStream_t stream) {
  if (B == 0) return 0;
  // 1/sqrt(dim_head) evaluated in double then narrowed, as `1.0F / std::sqrt(size_t)` does (Modules.cc:43)
  const float dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
  const int n_qb = (T + kQB - 1) / kQB;
  const size_t smem = tiled_smem_bytes(T, dh);
  const long blocks = static_cast<long>(B) * H * n_qb;
  if (!self_attention_tiled_supported(T, dh) || blocks > 0x7fffffffL) return 1;
  if (dh == 32) {
    if (ensure_dyn_smem(self_attention_tiled_kernel<32>, smem) != cudaSuccess) return 1;
    self_attention_tiled_kernel<32><<<static_cast<unsigned>(blocks), kTThreads, smem, stream>>>(Q, K, V, lengths, T, H, n_qb, dk, out_f32, q);
  } else if (dh == 64) {
    if (ensure_dyn_smem(self_attention_tiled_kernel<64>, smem) != cudaSuccess) return 1;
    self_attention_tiled_kernel<64><<<static_cast<unsigned>(blocks), kTThreads, smem, stream>>>(Q, K, V, lengths, T, H, n_qb, dk, out_f32, q);
  } else {
    return 1;
  }
  return 0;
}

}  // namespace sb
