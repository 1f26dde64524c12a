// Building blocks shared by the row-tile kernels (fused_rows.cu, rows_ffn.cu): the weight-tile TMA ring, the
// single-thread MMA consumer, the swizzled operand addressing and the bit-exact LayerNorm pieces.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "exact_math.cuh"
#include "fused_rows.cuh"
#include "ptx.cuh"

namespace sb {
namespace rows {

constexpr int kWTile = 128 * 128;     // one weight tile: 128 features x 128-byte k-block
constexpr int kEpiWarps = 16;
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kThreads = 128 + kEpiThreads;  // warp0 TMA, warps 1 and 3 MMA issuers, warp2 TMEM alloc, warps 4-19 epilogue

// byte offset of element (row r, k index kk) inside a K-major 128B-swizzled operand made of [R x 128 B] k-blocks
template <int R>
__device__ __forceinline__ uint32_t opnd_off(int r, int kk) {
  return static_cast<uint32_t>((kk >> 7) * (R * 128) + r * 128 + ((((kk & 127) >> 4) ^ (r & 7)) << 4) + (kk & 15));
}

// clamp(rne(x * aq), -127, 127) + 127 (exact_math.cuh: quantize1), optionally as the signed value
__device__ __forceinline__ uint8_t quant_byte(float x, float aq, bool sgn) {
  const int q = quantize1(x, aq);
  return static_cast<uint8_t>(sgn ? q - 127 : q);
}

// LayerNorm statistics of one row parked in xs (slimt/TensorOps.cc:542-580: sequential sums in element order,
// population variance, eps inside the square root).  Thread = row; rows are E + 1 floats apart (bank-conflict free).
template <int E>
__device__ __forceinline__ void ln_stats_row(const float* xr, float* mean_out, float* sigma_out, float eps) {
  // The two sums are strict left-to-right chains (4 cycles per add); the loads of the next 16 elements are issued
  // before the current 16 are added so that the chain never waits for shared memory.
  constexpr int kB = 16;
  static_assert(E % (2 * kB) == 0, "row length");
  float a[kB], b[kB];
#pragma unroll
  for (int i = 0; i < kB; i++) a[i] = xr[i];
  float sum = 0.0f;
#pragma unroll 1
  for (int e = 0; e < E; e += 2 * kB) {
#pragma unroll
    for (int i = 0; i < kB; i++) b[i] = xr[e + kB + i];
#pragma unroll
    for (int i = 0; i < kB; i++) sum = __fadd_rn(sum, a[i]);
    const int nx = (e + 2 * kB < E) ? e + 2 * kB : 0;  // the last prefetch wraps to the row start: reused by pass 2
#pragma unroll
    for (int i = 0; i < kB; i++) a[i] = xr[nx + i];
#pragma unroll
    for (int i = 0; i < kB; i++) sum = __fadd_rn(sum, b[i]);
  }
  const float mean = __fdiv_rn(sum, static_cast<float>(E));
  float sq = 0.0f;
#pragma unroll 1
  for (int e = 0; e < E; e += 2 * kB) {
#pragma unroll
    for (int i = 0; i < kB; i++) b[i] = xr[e + kB + i];
#pragma unroll
    for (int i = 0; i < kB; i++) {
      const float d = __fsub_rn(a[i], mean);
      sq = __fadd_rn(sq, __fmul_rn(d, d));
    }
    const int nx = (e + 2 * kB < E) ? e + 2 * kB : 0;
#pragma unroll
    for (int i = 0; i < kB; i++) a[i] = xr[nx + i];
#pragma unroll
    for (int i = 0; i < kB; i++) {
      const float d = __fsub_rn(b[i], mean);
      sq = __fadd_rn(sq, __fmul_rn(d, d));
    }
  }
  *mean_out = mean;
  *sigma_out = __fsqrt_rn(__fadd_rn(__fdiv_rn(sq, static_cast<float>(E)), eps));
}

__device__ __forceinline__ float ln_apply(float x, float mean, float sigma, float g, float b) {
  return __fadd_rn(__fmul_rn(g, __fdiv_rn(__fsub_rn(x, mean), sigma)), b);
}

// LayerNorm statistics of R rows parked in xs (row stride E + 1 floats), all kEpiWarps warps cooperating: a warp owns
// rows ew, ew + 16, ...; its lanes stride over the features and meet in a shuffle tree.  stats[row] = mean,
// stats[R + row] = 1 / sqrt(var + eps) (the exact path stores sigma there and divides).
template <int E, int R>
__device__ __forceinline__ void ln_stats_fast(const float* xs, float* stats, float eps, int ew, int lane) {
  constexpr int kPer = E / 32;
  for (int row = ew; row < R; row += kEpiWarps) {
    const float* xr = xs + row * (E + 1);
    float v[kPer];
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < kPer; i++) {
      v[i] = xr[lane + 32 * i];
      s += v[i];
    }
    const float mean = warp_sum(s) * (1.0f / static_cast<float>(E));
    float sq = 0.0f;
#pragma unroll
    for (int i = 0; i < kPer; i++) {
      const float d = v[i] - mean;
      sq = fmaf(d, d, sq);
    }
    sq = warp_sum(sq);
    if (lane == 0) {
      stats[row] = mean;
      stats[R + row] = rsqrtf(fmaf(sq, 1.0f / static_cast<float>(E), eps));
    }
  }
}
template <bool kFast>
__device__ __forceinline__ float ln_apply_t(float x, float mean, float sigma_or_rstd, float g, float b) {
  if constexpr (kFast) return fmaf((x - mean) * sigma_or_rstd, g, b);
  else return ln_apply(x, mean, sigma_or_rstd, g, b);
}
// Streams one weight tile per call through the ring (producer side).
struct RingProducer {
  uint8_t* ring;
  uint64_t* full;
  uint64_t* empty;
  uint32_t it;
  int stages;
  __device__ __forceinline__ void load(const CUtensorMap* map, int kb, int mb) {
    const uint32_t s = it % stages, ph = (it / stages) & 1;
    mbar_wait(&empty[s], ph ^ 1);
    mbar_expect_tx(&full[s], kWTile);
    tma_load_2d(ring + s * kWTile, map, &full[s], kb * 128, mb * 128);
    it++;
  }
};

// Consumes one weight tile per call (MMA side): four K = 32 MMAs of [128 features] x [R rows].
template <int R>
struct RingConsumer {
  uint8_t* ring;
  uint64_t* full;
  uint64_t* empty;
  uint32_t it;
  int stages;
  __device__ __forceinline__ void mma(uint32_t tmem_d, const uint8_t* opnd_kblock, bool first) {
    constexpr uint32_t idesc = make_idesc_i8_wa(128, R);
    const uint32_t s = it % stages, ph = (it / stages) & 1;
    mbar_wait(&full[s], ph);
    tc_fence_after();
    const uint64_t da = make_kmajor_sw128_desc(smem_u32(ring + s * kWTile));
    const uint64_t db = make_kmajor_sw128_desc(smem_u32(opnd_kblock));
#pragma unroll
    for (int k = 0; k < 4; k++) umma_i8(tmem_d, da + 2 * k, db + 2 * k, idesc, (first && k == 0) ? 0u : 1u);
    umma_commit(&empty[s]);
    it++;
  }
};

// TMEM -> registers: this warp's 32 lanes x N consecutive columns (N = 8 or 32), no wait.
template <int N>
__device__ __forceinline__ void tmem_ldn_nowait(uint32_t taddr, uint32_t (&v)[N]);
template <>
__device__ __forceinline__ void tmem_ldn_nowait<8>(uint32_t taddr, uint32_t (&v)[8]) { tmem_ld8_nowait(taddr, v); }
template <>
__device__ __forceinline__ void tmem_ldn_nowait<32>(uint32_t taddr, uint32_t (&v)[32]) { tmem_ld32_nowait(taddr, v); }

}  // namespace rows
}  // namespace sb
