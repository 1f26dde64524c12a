// See gemm_i8.cuh for the contract.  sm_100a only.
#include "gemm_i8.cuh"

#include <stdio.h>

#include "exact_math.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kThreads = 256;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 constants, warps4-7 epilogue

template <int BN>
struct TileCfg {
  static constexpr int kSub = BN > 256 ? BN / 256 : 1;  // MMAs per k-step along N (UMMA N <= 256)
  static constexpr int kUmmaN = BN > 256 ? 256 : BN;
  static constexpr int kABytes = kBM * kBK;
  static constexpr int kBBytes = BN * kBK;
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr uint32_t kTmemCols = BN < 32 ? 32 : BN;
};

template <int BN, int STAGES, int EPI>
__global__ void __launch_bounds__(kThreads) gemm_i8_kernel(const __grid_constant__ GemmBatch batch) {
  using Cfg = TileCfg<BN>;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // 1024-byte alignment is required by the 128B swizzle atoms.
  uint8_t* smem = smem_align1024(smem_raw);

  const GemmProblem& P = batch.prob[blockIdx.z];
  const int M = batch.M, N = batch.N, K = batch.K;
  const int n0 = blockIdx.x * BN;
  const int m0 = blockIdx.y * kBM;
  const int num_kb = (K + kBK - 1) / kBK;

  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + STAGES * Cfg::kABytes;
  uint8_t* tail = smem + STAGES * Cfg::kStageBytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* accum_bar = empty_bar + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_bar + 1);
  float* s_pb = reinterpret_cast<float*>(tail + 128);
  float* s_scale = s_pb + BN;
  float* s_bias = s_scale + BN;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&P.tma_a);
    tma_prefetch_desc(&P.tma_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(accum_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) {
    tmem_alloc<Cfg::kTmemCols>(tmem_slot);
  }
  if (warp == 3) {
    for (int i = lane; i < BN; i += 32) {
      int n = n0 + i;
      bool ok = n < N;
      s_pb[i] = ok ? P.pb[n] : 0.0f;
      if constexpr (EPI == EPI_RES_LN) {
        s_scale[i] = ok ? P.ln_scale[n] : 0.0f;
        s_bias[i] = ok ? P.ln_bias[n] : 0.0f;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one()) {
      for (int kb = 0; kb < num_kb; kb++) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        mbar_expect_tx(&full_bar[s], Cfg::kStageBytes);
        tma_load_2d(smem_a + s * Cfg::kABytes, &P.tma_a, &full_bar[s], kb * kBK, m0);
#pragma unroll
        for (int j = 0; j < Cfg::kSub; j++) {
          tma_load_2d(smem_b + s * Cfg::kBBytes + j * Cfg::kUmmaN * kBK, &P.tma_b, &full_bar[s], kb * kBK,
                      n0 + j * Cfg::kUmmaN);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (single thread) =====
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_i8(kBM, Cfg::kUmmaN);
      for (int kb = 0; kb < num_kb; kb++) {
        const int s = kb % STAGES;
        const uint32_t ph = (kb / STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint64_t da = make_kmajor_sw128_desc(smem_u32(smem_a + s * Cfg::kABytes));
#pragma unroll
        for (int j = 0; j < Cfg::kSub; j++) {
          const uint64_t db = make_kmajor_sw128_desc(smem_u32(smem_b + s * Cfg::kBBytes + j * Cfg::kUmmaN * kBK));
#pragma unroll
          for (int k = 0; k < kBK / 32; k++) {
            // advance 32 bytes (= UMMA_K int8 elements) inside the swizzle atom: +2 in 16-byte units
            umma_i8(tmem_base + j * Cfg::kUmmaN, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          }
        }
        umma_commit(&empty_bar[s]);  // frees this smem stage when the MMAs above retire
      }
      umma_commit(accum_bar);  // accumulator complete
    }
  } else if (warp >= 4) {
    // ===== epilogue: thread <-> TMEM lane <-> output row =====
    const int q = warp & 3;
    const int row = m0 + q * 32 + lane;
    const bool row_ok = row < M;
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    mbar_wait(accum_bar, 0);
    tc_fence_after();
    const float um = P.um;
    uint32_t v[32];

    if constexpr (EPI == EPI_F32 || EPI == EPI_ACC) {
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        tmem_ld32(taddr + c * 32, v);
        const int nb = n0 + c * 32;
        if (row_ok && nb < N) {
          if constexpr (EPI == EPI_ACC) {
            int32_t* o = static_cast<int32_t*>(P.out) + static_cast<size_t>(row) * P.ldo + nb;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (nb + j < N) {
                int4 w = make_int4((int)v[j], (int)v[j + 1], (int)v[j + 2], (int)v[j + 3]);
                *reinterpret_cast<int4*>(o + j) = w;
              }
            }
          } else {
            float* o = static_cast<float*>(P.out) + static_cast<size_t>(row) * P.ldo + nb;
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              if (nb + j < N) {
                float y[4];
#pragma unroll
                for (int e = 0; e < 4; e++) {
                  y[e] = dequant1((int)v[j + e], um, s_pb[c * 32 + j + e]);
                  if (P.relu) y[e] = y[e] > 0.0f ? y[e] : 0.0f;  // std::max<float>(0, a), TensorOps.cc:163
                }
                *reinterpret_cast<float4*>(o + j) = make_float4(y[0], y[1], y[2], y[3]);
              }
            }
          }
        }
      }
    } else if constexpr (EPI == EPI_QUANT) {
      const float aq = P.aq_out[0];
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        tmem_ld32(taddr + c * 32, v);
        const int nb = n0 + c * 32;
        if (row_ok && nb < N) {
          uint32_t w[8];
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            int qv[4];
#pragma unroll
            for (int e = 0; e < 4; e++) {
              float y = dequant1((int)v[j + e], um, s_pb[c * 32 + j + e]);
              if (P.relu) y = y > 0.0f ? y : 0.0f;
              qv[e] = quantize1(y, aq);
            }
            w[j / 4] = pack4(qv[0], qv[1], qv[2], qv[3]);
          }
          int8_t* o = P.qout[0] + static_cast<size_t>(row) * N + nb;
          if (nb + 32 <= N) {
            *reinterpret_cast<uint4*>(o) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(o + 16) = make_uint4(w[4], w[5], w[6], w[7]);
          } else {
            for (int j = 0; j < 8 && nb + j * 4 < N; j++) *reinterpret_cast<uint32_t*>(o + j * 4) = w[j];
          }
        }
      }
    } else if constexpr (EPI == EPI_RES_LN) {
      // LayerNorm(y + residual): reference slimt/TensorOps.cc:542-580 (sequential sums, population
      // variance, eps inside sqrt).  The f32 row is parked back in TMEM between the three passes.
      const float* res = P.residual + static_cast<size_t>(row_ok ? row : 0) * N;
      float sum = 0.0f;
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        tmem_ld32(taddr + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          float4 r4 = *reinterpret_cast<const float4*>(res + c * 32 + j);
          float r[4] = {r4.x, r4.y, r4.z, r4.w};
#pragma unroll
          for (int e = 0; e < 4; e++) {
            float y = dequant1((int)v[j + e], um, s_pb[c * 32 + j + e]);
            float x = __fadd_rn(y, r[e]);
            sum = __fadd_rn(sum, x);
            v[j + e] = __float_as_uint(x);
          }
        }
        tmem_st32(taddr + c * 32, v);
      }
      const float cols = static_cast<float>(N);
      const float mean = __fdiv_rn(sum, cols);
      float sq = 0.0f;
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        tmem_ld32(taddr + c * 32, v);
#pragma unroll
        for (int j = 0; j < 32; j++) {
          float d = __fsub_rn(__uint_as_float(v[j]), mean);
          sq = __fadd_rn(sq, __fmul_rn(d, d));
        }
      }
      const float sigma = __fsqrt_rn(__fadd_rn(__fdiv_rn(sq, cols), P.ln_eps));
#pragma unroll 1
      for (int c = 0; c < BN / 32; c++) {
        tmem_ld32(taddr + c * 32, v);
        float y[32];
#pragma unroll
        for (int j = 0; j < 32; j++) {
          float t = __fdiv_rn(__fsub_rn(__uint_as_float(v[j]), mean), sigma);
          y[j] = __fadd_rn(__fmul_rn(s_scale[c * 32 + j], t), s_bias[c * 32 + j]);
        }
        if (row_ok) {
          if (P.out != nullptr) {
            float* o = static_cast<float*>(P.out) + static_cast<size_t>(row) * N + c * 32;
#pragma unroll
            for (int j = 0; j < 32; j += 4) *reinterpret_cast<float4*>(o + j) = make_float4(y[j], y[j + 1], y[j + 2], y[j + 3]);
          }
          for (int k = 0; k < P.n_qout; k++) {
            const float aq = P.aq_out[k];
            const int sh = ((P.qout_signed >> k) & 1) ? 127 : 0;
            uint32_t w[8];
#pragma unroll
            for (int j = 0; j < 32; j += 4)
              w[j / 4] = pack4(quantize1(y[j], aq) - sh, quantize1(y[j + 1], aq) - sh, quantize1(y[j + 2], aq) - sh,
                               quantize1(y[j + 3], aq) - sh);
            int8_t* o = P.qout[k] + static_cast<size_t>(row) * N + c * 32;
            *reinterpret_cast<uint4*>(o) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4*>(o + 16) = make_uint4(w[4], w[5], w[6], w[7]);
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tmem_dealloc<Cfg::kTmemCols>(tmem_base);
  }
}

template <int BN, int STAGES, int EPI>
void launch_one(const GemmBatch& b, int n_problems, cudaStream_t stream) {
  const size_t smem = gemm_smem_bytes(BN, STAGES);
  auto kern = gemm_i8_kernel<BN, STAGES, EPI>;
  ensure_dyn_smem(kern, smem);  // per (device, kernel): a process may drive several GPUs
  dim3 grid((b.N + BN - 1) / BN, (b.M + kBM - 1) / kBM, n_problems);
  kern<<<grid, kThreads, smem, stream>>>(b);
}

template <int EPI>
void dispatch_bn(const GemmBatch& b, int n_problems, int BN, cudaStream_t stream) {
  const bool deep = b.K > 2 * kBK;
  switch (BN) {
    case 64:
      return launch_one<64, 4, EPI>(b, n_problems, stream);
    case 128:
      return launch_one<128, 4, EPI>(b, n_problems, stream);
    case 256:
      if (deep) return launch_one<256, 4, EPI>(b, n_problems, stream);
      return launch_one<256, 2, EPI>(b, n_problems, stream);
    case 512:
      return launch_one<512, 2, EPI>(b, n_problems, stream);
    default:
      fprintf(stderr, "slimt_b200: unsupported GEMM tile BN=%d\n", BN);
      abort();
  }
}

}  // namespace

size_t gemm_smem_bytes(int BN, int stages) {
  // stages * (A + B) + barriers (128 B) + pb/scale/bias (12 B per column) + 1024 B alignment slack
  return static_cast<size_t>(stages) * (kBM * kBK + BN * kBK) + 128 + static_cast<size_t>(BN) * 12 + 1024;
}

void launch_gemm_i8(const GemmBatch& batch, int n_problems, int epilogue, int BN, cudaStream_t stream) {
  switch (epilogue) {
    case EPI_F32:
      return dispatch_bn<EPI_F32>(batch, n_problems, BN, stream);
    case EPI_QUANT:
      return dispatch_bn<EPI_QUANT>(batch, n_problems, BN, stream);
    case EPI_RES_LN:
      return dispatch_bn<EPI_RES_LN>(batch, n_problems, BN, stream);
    case EPI_ACC:
      return dispatch_bn<EPI_ACC>(batch, n_problems, BN, stream);
    default:
      fprintf(stderr, "slimt_b200: unknown epilogue %d\n", epilogue);
      abort();
  }
}

}  // namespace sb
