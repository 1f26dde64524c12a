// int8 x int8 -> int32 GEMM on the 5th-gen tensor cores (tcgen05.mma kind::i8)
// with TMA-fed shared memory, int32 accumulators in TMEM and fused epilogues.
//
// Replaces, for slimt's hot path, the whole of qmm::affine / dot /
// affine_with_select (reference slimt/QMM.cc:37-75, qmm/Intgemm.inl.cc:8-243 ==
// qmm/Gemmology.inl.cc:33-281): PrepareA is done by the PRODUCER of the
// activation (it emits int8), PrepareBias is precomputed at load, Multiply is the
// MMA, UnquantizeAndAddBiasAndWrite (+ReLU / +requantize / +residual+LayerNorm)
// is the epilogue; the output projection's fused argmax is out_argmax.cu.
//
// Layouts: A = quantized activations as the reference's PrepareA emits them, u8 = qa + 127, [M][K] row-major
// (K contiguous), so the u8 x s8 MMA forms Int8Shift::Multiply's shifted accumulator directly;
// B = weights in the STORED model layout B^T, int8 [N][K] (K contiguous) -- i.e.
// both operands are "K-major" for UMMA, no re-tiling at load.  One CTA computes
// one [128 x BN] output tile; K is consumed in 128-byte blocks (one 128B-swizzle
// atom row per matrix row) through a STAGES-deep TMA/mbarrier ring.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace sb {

constexpr int kBM = 128;   // rows per CTA tile == TMEM lanes
constexpr int kBK = 128;   // int8 elements (= bytes) per k-block
constexpr int kMaxQuantOut = 4;

enum Epilogue : int {
  EPI_F32 = 0,     // y (optionally ReLU) -> f32 [M][N]
  EPI_QUANT = 1,   // relu?(y) -> requantize with aq_out[0] -> int8 [M][N]
  EPI_RES_LN = 2,  // LayerNorm(y + residual) -> f32 (optional) + up to 4 int8 copies; needs BN == N
  EPI_ACC = 4,     // raw shifted int32 accumulators -> s32 [M][N] (parity/debug tap)
};

struct GemmProblem {
  CUtensorMap tma_a;  // int8 [M][K]
  CUtensorMap tma_b;  // int8 [N][K]
  const float* pb;      // [N] prepared bias: colsum*(-127/(aq*bq)) + bias  (Intgemm.inl.cc:112-128)
  float um;             // 1/(aq*bq)
  int relu;
  // EPI_F32 / EPI_ACC
  void* out;            // f32 or s32 [M][ldo]
  int ldo;
  // EPI_QUANT / EPI_RES_LN
  int8_t* qout[kMaxQuantOut];
  float aq_out[kMaxQuantOut];
  int n_qout;
  int qout_signed;  // bit k set: qout[k] receives the signed qa instead of the u8 (qa + 127)
  // EPI_RES_LN
  const float* residual;  // f32 [M][N]
  const float* ln_scale;  // [N]
  const float* ln_bias;   // [N]
  float ln_eps;
};

struct GemmBatch {
  GemmProblem prob[3];
  int M, N, K;
};

size_t gemm_smem_bytes(int BN, int stages);

// Launches grid (ceil(N/BN), ceil(M/128), n_problems).
void launch_gemm_i8(const GemmBatch& batch, int n_problems, int epilogue, int BN, cudaStream_t stream);

}  // namespace sb
