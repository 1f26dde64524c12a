// Decoder cross-attention over the cached encoder K/V (reference: Attention::forward with
// q = one decoder row per sentence, slimt/Modules.cc:287-319, scaled_dot_product_attention :24-86).
//
// HBM-bound: every decode step streams the whole f32 K and V cache of the batch once
// (2 * S * E * 4 bytes per sentence per layer).  A persistent CTA per SM walks sentences; a producer
// warp keeps a ring of TMA box loads (one 128-byte-swizzled [32 keys x 32 floats] tile per head) in
// flight while H consumer warps (warp = head) compute from shared memory.  The arithmetic order is
// the reference's: per-key sequential fma chains over the head dimension (ruy's sgemm), then the
// scalar softmax of slimt/TensorOps.cc:282-315 (max, exp, sum in key order, divide), then the
// probability-weighted sum of V in key order.
#include <stdio.h>

#include "exact_math.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kRegKeyChunks = 8;   // S <= 256: every lane keeps its keys' scores in registers
constexpr int kMaxKeyChunks = 32;  // S <= 1024: the scores are parked in the warp's shared memory instead

// NC = compile-time bound on 32-key chunks per sentence (ceil(S / 32) rounded up to 1, 2, 4, 8 or 32).  Above 8 chunks
// the score array would spill; each lane then keeps score c of key 32 c + lane at sc_smem[32 c + lane] of its warp's
// block (written and read back by the same lane only), and the chunk loops are not unrolled.
template <int DH, int H, int NC>
__global__ void __launch_bounds__((H + 1) * 32, 3)
    cross_attention_kernel(const __grid_constant__ CUtensorMap mapK, const __grid_constant__ CUtensorMap mapV,
                           const float* __restrict__ Qr, const uint32_t* __restrict__ lengths, int B, int S,
                           int box_rows, int stages, float dk, float* __restrict__ out_f32, QuantOuts q,
                           float* __restrict__ attn_head0) {
  constexpr int E = H * DH;
  constexpr int kSub = DH / 32;  // 128-byte column tiles per head
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  const uint32_t tile_bytes = static_cast<uint32_t>(box_rows) * 128u;
  const uint32_t chunk_bytes = tile_bytes * H * kSub;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + static_cast<size_t>(stages) * chunk_bytes);
  uint64_t* empty_bar = full_bar + stages;
  uint64_t* exp_tab = empty_bar + stages;
  float* sq_all = reinterpret_cast<float*>(exp_tab + 32);
  constexpr bool kSmemScores = NC > kRegKeyChunks;
  constexpr int kUnroll = kSmemScores ? 1 : NC;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x >= 32 && threadIdx.x < 64) exp_tab[threadIdx.x - 32] = kExp2fTab[threadIdx.x - 32];
  if (threadIdx.x == 0) {
    tma_prefetch_desc(&mapK);
    tma_prefetch_desc(&mapV);
    for (int s = 0; s < stages; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], H);
    }
    fence_barrier_init();
  }
  __syncthreads();

  if (warp == H) {
    // ===== producer: one thread issues every TMA load of this CTA's sentences =====
    if (lane == 0) {
      uint32_t it = 0;
      for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const int len = min(static_cast<int>(lengths[b]), S);
        const int nc = (len + 31) >> 5;
        for (int pass = 0; pass < 2; pass++) {
          const CUtensorMap* map = pass == 0 ? &mapK : &mapV;
          for (int c = 0; c < nc; c++, it++) {
            const uint32_t s = it % stages;
            const uint32_t ph = (it / stages) & 1;
            mbar_wait(&empty_bar[s], ph ^ 1);
            mbar_expect_tx(&full_bar[s], chunk_bytes);
            uint8_t* dst = smem + static_cast<size_t>(s) * chunk_bytes;
#pragma unroll
            for (int t = 0; t < H * kSub; t++) {
              tma_load_2d(dst + t * tile_bytes, map, &full_bar[s], t * 32, b * S + c * 32);
            }
          }
        }
      }
    }
    return;
  }

  // ===== consumers: warp = head =====
  const int h = warp;
  float* sq = sq_all + h * DH;
  float* sp = sq_all + H * DH + h * 32;  // this warp's probabilities of the current 32-key chunk
  float* sc_smem = sq_all + H * (DH + 32) + h * (kSmemScores ? NC * 32 : 0);
  // Per-lane byte offsets inside a swizzled [rows][128 B] tile.  Score pass: lane = key row, 16-byte
  // chunk g sits at ((g ^ (row & 7)) << 4).  Value pass: lane = head dimension, row l of the tile holds
  // it at (((lane >> 2) ^ (l & 7)) << 4) + (lane & 3) * 4.
  uint32_t voff[8];
#pragma unroll
  for (int r = 0; r < 8; r++) voff[r] = ((((lane >> 2) ^ r) << 4) + ((lane & 3) << 2));
  uint32_t it = 0;
  for (int b = blockIdx.x; b < B; b += gridDim.x) {
    const int len = min(static_cast<int>(lengths[b]), S);
    const int nc = (len + 31) >> 5;
    __syncwarp();
    for (int d = lane; d < DH; d += 32) sq[d] = Qr[static_cast<size_t>(b) * E + h * DH + d];
    __syncwarp();
    float sc_reg[kSmemScores ? 1 : NC];
    auto sc = [&](int c) -> float& {
      if constexpr (kSmemScores) return sc_smem[c * 32 + lane];
      else return sc_reg[c];
    };
    float mx = -3.402823466e+38f;
#pragma unroll kUnroll
    for (int c = 0; c < NC; c++) {
      sc(c) = 0.0f;
      if (c < nc) {
        const uint32_t s = it % stages;
        const uint32_t ph = (it / stages) & 1;
        it++;
        mbar_wait(&full_bar[s], ph);
        const uint8_t* tile = smem + static_cast<size_t>(s) * chunk_bytes + (h * kSub) * tile_bytes + lane * 128;
        float acc = 0.0f;
#pragma unroll
        for (int u = 0; u < kSub; u++) {
#pragma unroll
          for (int g = 0; g < 8; g++) {
            const float4 kk = *reinterpret_cast<const float4*>(tile + u * tile_bytes + ((g ^ (lane & 7)) << 4));
            const float4 qq = *reinterpret_cast<const float4*>(sq + u * 32 + g * 4);
            acc = fmaf(qq.x, kk.x, acc);
            acc = fmaf(qq.y, kk.y, acc);
            acc = fmaf(qq.z, kk.z, acc);
            acc = fmaf(qq.w, kk.w, acc);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
        if (c * 32 + lane < len) {
          acc = __fmul_rn(dk, acc);
          sc(c) = acc;
          mx = fmaxf(mx, acc);
        }
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.0f;
#pragma unroll kUnroll
    for (int c = 0; c < NC; c++) {
      if (c < nc) {
        const int j = c * 32 + lane;
        sc(c) = (j < len) ? expf_glibc_nonpos_tab(__fsub_rn(sc(c), mx), exp_tab) : 0.0f;
        // sum in key order (slimt/TensorOps.cc:296-314): exp of a masked key is +0 and adding it is exact
        __syncwarp();
        sp[lane] = sc(c);
        __syncwarp();
#pragma unroll
        for (int l = 0; l < 32; l += 4) {
          const float4 e = *reinterpret_cast<const float4*>(sp + l);
          sum = __fadd_rn(sum, e.x);
          sum = __fadd_rn(sum, e.y);
          sum = __fadd_rn(sum, e.z);
          sum = __fadd_rn(sum, e.w);
        }
      }
    }
#pragma unroll kUnroll
    for (int c = 0; c < NC; c++) {
      if (c < nc) sc(c) = __fdiv_rn(sc(c), sum);
    }
    if (attn_head0 != nullptr && h == 0) {
#pragma unroll kUnroll
      for (int c = 0; c < NC; c++) {
        const int j = c * 32 + lane;
        if (j < S) attn_head0[static_cast<size_t>(b) * S + j] = (j < len) ? sc(c) : 0.0f;
      }
    }

    float acc[kSub];
#pragma unroll
    for (int u = 0; u < kSub; u++) acc[u] = 0.0f;
#pragma unroll kUnroll
    for (int c = 0; c < NC; c++) {
      if (c < nc) {
        const uint32_t s = it % stages;
        const uint32_t ph = (it / stages) & 1;
        it++;
        __syncwarp();
        sp[lane] = sc(c);
        __syncwarp();
        mbar_wait(&full_bar[s], ph);
        const uint8_t* tile = smem + static_cast<size_t>(s) * chunk_bytes + (h * kSub) * tile_bytes;
        const int lim = min(32, len - c * 32);
        if (lim == 32) {
#pragma unroll
          for (int l = 0; l < 32; l += 4) {
            const float4 p = *reinterpret_cast<const float4*>(sp + l);
            const float pv[4] = {p.x, p.y, p.z, p.w};
#pragma unroll
            for (int e = 0; e < 4; e++) {
#pragma unroll
              for (int u = 0; u < kSub; u++) {
                acc[u] = fmaf(pv[e], *reinterpret_cast<const float*>(tile + u * tile_bytes + (l + e) * 128 + voff[(l + e) & 7]),
                              acc[u]);
              }
            }
          }
        } else {
          // ragged tail: the reference's remaining keys carry probability +0 and change nothing
          for (int l = 0; l < lim; l++) {
            const float pl = sp[l];
            const uint32_t o = l * 128 + ((((lane >> 2) ^ (l & 7)) << 4) + ((lane & 3) << 2));
#pragma unroll
            for (int u = 0; u < kSub; u++) acc[u] = fmaf(pl, *reinterpret_cast<const float*>(tile + u * tile_bytes + o), acc[u]);
          }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty_bar[s]);
      }
    }
    const size_t off = static_cast<size_t>(b) * E + h * DH;
#pragma unroll
    for (int u = 0; u < kSub; u++) {
      if (out_f32) out_f32[off + u * 32 + lane] = acc[u];
      for (int k = 0; k < q.n; k++) q.ptr[k][off + u * 32 + lane] = static_cast<int8_t>(quantize1(acc[u], q.aq[k]));
    }
  }
}

}  // namespace

int cross_attention_box_rows(int S) { return S >= 32 ? 32 : ((S + 7) & ~7); }

int launch_cross_attention(const CUtensorMap& mapK, const CUtensorMap& mapV, const float* Qr, const uint32_t* lengths,
                           int B, int S, int H, int dh, int num_sms, float* out_f32, QuantOuts q, float* attn_head0,
                           cudaStream_t stream) {
  if (B == 0) return 0;
  if (S > 32 * kMaxKeyChunks || H != 8 || (dh != 32 && dh != 64)) return 1;
  const float dk = static_cast<float>(1.0 / std::sqrt(static_cast<double>(dh)));
  const int box_rows = cross_attention_box_rows(S);
  const size_t chunk = static_cast<size_t>(box_rows) * 128 * H * (dh / 32);
  // Two ring stages per CTA (a sentence's K chunk is consumed while its V chunk lands) and as many CTAs
  // per SM as shared memory allows: the per-head instruction stream is a latency chain, so the bytes in
  // flight come from co-resident CTAs.
  int stages = 2;
  if (chunk <= 8 * 1024) stages = 4;
  const int nc = (S + 31) / 32;
  const size_t sc_park = nc > kRegKeyChunks ? static_cast<size_t>(H) * kMaxKeyChunks * 32 * sizeof(float) : 0;
  const size_t smem = 1024 + stages * chunk + stages * 16 + 256 + static_cast<size_t>(H) * (dh + 32) * sizeof(float) + sc_park;
  int per_sm = static_cast<int>((220 * 1024) / (smem + 1024));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 3) per_sm = 3;
  const int grid = B < num_sms * per_sm ? B : num_sms * per_sm;
  const int threads = (H + 1) * 32;
#define SB_CA_LAUNCH(DH_, NC_)                                                                                   \
  do {                                                                                                           \
    auto kern = cross_attention_kernel<DH_, 8, NC_>;                                                             \
    if (ensure_dyn_smem(kern, smem) != cudaSuccess) return 1;                                                    \
    kern<<<grid, threads, smem, stream>>>(mapK, mapV, Qr, lengths, B, S, box_rows, stages, dk, out_f32, q,      \
                                          attn_head0);                                                           \
  } while (0)
  if (dh == 32) {
    if (nc <= 1) SB_CA_LAUNCH(32, 1);
    else if (nc <= 2) SB_CA_LAUNCH(32, 2);
    else if (nc <= 4) SB_CA_LAUNCH(32, 4);
    else if (nc <= 8) SB_CA_LAUNCH(32, 8);
    else SB_CA_LAUNCH(32, 32);
  } else {
    if (nc <= 1) SB_CA_LAUNCH(64, 1);
    else if (nc <= 2) SB_CA_LAUNCH(64, 2);
    else if (nc <= 4) SB_CA_LAUNCH(64, 4);
    else if (nc <= 8) SB_CA_LAUNCH(64, 8);
    else SB_CA_LAUNCH(64, 32);
  }
#undef SB_CA_LAUNCH
  return 0;
}

}  // namespace sb
