// Row-tile kernel of the attention-output + feed-forward half of a layer (encoder and decoder):
//   y = LN1(res + Wo a + bo);   z = LN2(y + W2 relu(W1 y + b1) + b2)
// Reference: Attention::forward tail (slimt/Modules.cc:308-316) + FFN block of EncoderLayer / DecoderLayer
// (:326-331, :251-257).  See fused_rows.cuh for the tile design.  R = rows per CTA tile: 32 for the decoder
// step (latency: one tile per SM at B = 4096), 128 for the encoder (throughput: full-rate N = 128 MMAs and a
// quarter of the weight re-streaming).
//
// GEMM 1 (FFN1) and GEMM 2 (FFN2) are interleaved per 128-feature block: block j of relu(W1 y + b1) is
// requantised by the epilogue warps into a ring of operand k-blocks and consumed by FFN2's k-step j while the
// tensor core already works on block j + 2, so the F-wide intermediate never exists in full.
#include <stdio.h>

#include "rows_common.cuh"

namespace sb {

namespace {

using namespace rows;

constexpr int kLook = 2;  // FFN1 feature blocks issued ahead of the FFN2 k-step that consumes them

template <int E, int F, int R>
struct FfnPlan {
  static constexpr int EK = E / 128, EM = E / 128, FM = F / 128;
  static constexpr int kOpK = R * 128;                                    // one operand k-block
  // two weight rings, one per MMA-issuing thread: ring A streams Wo and W1, ring B streams W2
  static constexpr int kStagesA = (R == 32) ? ((E == 256) ? 4 : 2) : 2;
  static constexpr int kStagesB = (R == 32) ? ((E == 256) ? 4 : 2) : 2;
  static constexpr int kStages = kStagesA + kStagesB;
  static constexpr int kTS = (R == 32) ? 8 : 2;                            // TMEM slots for FFN1 blocks
  static constexpr int kFS = (R == 32) ? FM : 4;                           // operand ring slots for relu(W1 y) blocks
  static constexpr bool kParkY = (R != 32);                                // y parked in global (xs aliases the f ring)
  static constexpr int XS = E + 1;
  static constexpr int ring = 0;
  static constexpr int opnd_a = ring + kStages * kWTile;                   // attention-output operand, then y operand
  static constexpr int opnd_y = kParkY ? opnd_a : opnd_a + EK * kOpK;      // R = 128: y reuses the a buffer
  static constexpr int opnd_f = opnd_y + EK * kOpK;
  static constexpr int xs_bytes = R * XS * 4;
  static constexpr int f_bytes = kFS * kOpK;
  static constexpr int xs = kParkY ? opnd_f : opnd_f + f_bytes;            // R = 128: xs aliases the f ring
  static constexpr int after = kParkY ? opnd_f + (xs_bytes > f_bytes ? xs_bytes : f_bytes) : xs + xs_bytes;
  static constexpr int stats = (after + 15) & ~15;                         // mean[R], sigma[R]
  static constexpr int bars = stats + 2 * R * 4;
  // full[kStages] empty[kStages] (ring A's stages first) a_full g0_done yq_ready g2_done slot_full[kTS] slot_empty[kTS]
  // fq_full[kFS] fq_free[kFS]
  static constexpr int n_bars = 2 * kStages + 4 + 2 * kTS + 2 * kFS;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
  static_assert(EM * R + kTS * R <= 512, "TMEM columns");
  static_assert(total <= 227 * 1024, "shared memory");
};

template <int E, int F, int R, bool kFast>
__global__ void __launch_bounds__(kThreads, 1) rows_ffn_kernel(const __grid_constant__ RowsFfnArgs a) {
  using L = FfnPlan<E, F, R>;
  constexpr int EK = L::EK, EM = L::EM, FM = L::FM, XS = L::XS, kOpK = L::kOpK;
  constexpr int RPW = R / 4;  // rows (TMEM columns) per epilogue warp: 16 warps = 4 lane quadrants x 4 column groups
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* ring = smem + L::ring;
  uint8_t* opnd_a = smem + L::opnd_a;
  uint8_t* opnd_y = smem + L::opnd_y;
  uint8_t* opnd_f = smem + L::opnd_f;
  float* xs = reinterpret_cast<float*>(smem + L::xs);
  float* stats = reinterpret_cast<float*>(smem + L::stats);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint64_t* full = bars;
  uint64_t* empty = full + L::kStages;
  uint64_t* a_full = empty + L::kStages;
  uint64_t* g0_done = a_full + 1;
  uint64_t* yq_ready = g0_done + 1;
  uint64_t* g2_done = yq_ready + 1;
  uint64_t* slot_full = g2_done + 1;
  uint64_t* slot_empty = slot_full + L::kTS;
  uint64_t* fq_full = slot_empty + L::kTS;
  uint64_t* fq_free = fq_full + L::kFS;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.map_a);
    tma_prefetch_desc(&a.map_wo);
    tma_prefetch_desc(&a.map_w1);
    tma_prefetch_desc(&a.map_w2);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < L::kStages; s++) mbar_init(&full[s], 1), mbar_init(&empty[s], 1);
    mbar_init(a_full, 1);
    mbar_init(g0_done, 1);
    mbar_init(yq_ready, kEpiWarps);
    mbar_init(g2_done, 1);
    for (int s = 0; s < L::kTS; s++) mbar_init(&slot_full[s], 1), mbar_init(&slot_empty[s], kEpiWarps);
    for (int s = 0; s < L::kFS; s++) mbar_init(&fq_full[s], kEpiWarps), mbar_init(&fq_free[s], 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_acc = tmem;             // EM blocks x R columns: accumulators of the Wo GEMM, then of FFN2
  const uint32_t tmem_ring = tmem + EM * R;   // kTS slots x R columns: FFN1 feature blocks

  const int n_tiles = (a.M + R - 1) / R;
  uint32_t iter = 0;     // tile iterations of this CTA (phase of the once-per-tile barriers)
  uint32_t blocks = 0;   // FFN1 feature blocks so far: position in the TMEM slot ring and the operand ring (per role)
  // Ring A feeds warp 1 (Wo, W1), ring B feeds warp 3 (W2); each consumer object lives in its own warp's leader.
  uint8_t* ring_b = ring + L::kStagesA * kWTile;
  RingProducer prod_a{ring, full, empty, 0, L::kStagesA};
  RingProducer prod_b{ring_b, full + L::kStagesA, empty + L::kStagesA, 0, L::kStagesB};
  RingConsumer<R> cons = (warp == 3) ? RingConsumer<R>{ring_b, full + L::kStagesA, empty + L::kStagesA, 0, L::kStagesB}
                                     : RingConsumer<R>{ring, full, empty, 0, L::kStagesA};

  // One leader lane per warp, elected once (elect.sync also tells the compiler the branch is single-threaded, so
  // descriptors and addresses stay in uniform registers: no per-MMA waterfall loop as with `lane == 0`).  The ring
  // positions live in the leader's registers across tiles, hence a single election.
  const bool leader = elect_one();
  pdl_wait();  // everything above overlapped the previous kernel's tail; its outputs are visible from here on
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, iter++) {
    const int row0 = tile * R;
    const uint32_t tph = iter & 1;
    if (warp == 0) {
      // ===== TMA producer: the tile's input operand, then every weight tile in consumption order (Wo and W1 through
      // ring A, W2 through ring B)
      if (leader) {
        mbar_expect_tx(a_full, EK * kOpK);
        for (int kb = 0; kb < EK; kb++) tma_load_2d(opnd_a + kb * kOpK, &a.map_a, a_full, kb * 128, row0);
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) prod_a.load(&a.map_wo, kb, mb);
        for (int st = 0; st < FM + kLook; st++) {
          if (st < FM)
            for (int kb = 0; kb < EK; kb++) prod_a.load(&a.map_w1, kb, st);
          if (st >= kLook)
            for (int mb = 0; mb < EM; mb++) prod_b.load(&a.map_w2, st - kLook, mb);
        }
      }
    } else if (warp == 1) {
      // ===== MMA issuer A: the Wo GEMM and the FFN1 feature blocks.  The FFN2 k-steps are issued by warp 3, so that
      // neither stream waits behind the other's barrier / fence / commit latencies (a single issuing thread needed
      // ~2200 cycles per block for ~700 cycles of tensor-pipe work).  Each has its own weight ring.
      if (leader) {
        mbar_wait(a_full, tph);
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) cons.mma(tmem_acc + mb * R, opnd_a + kb * kOpK, kb == 0);
        umma_commit(g0_done);
        mbar_wait(yq_ready, tph);
        tc_fence_after();
        for (int st = 0; st < FM + kLook; st++) {
          if (st < FM) {  // FFN1 feature block st -> TMEM slot
            const uint32_t n = blocks + st;
            const uint32_t s = n % L::kTS, ph = (n / L::kTS) & 1;
            mbar_wait(&slot_empty[s], ph ^ 1);
            tc_fence_after();
            for (int kb = 0; kb < EK; kb++) cons.mma(tmem_ring + s * R, opnd_y + kb * kOpK, kb == 0);
            umma_commit(&slot_full[s]);
          }
        }
        blocks += FM;
      }
    } else if (warp == 3) {
      // ===== MMA issuer B: FFN2 k-step kb2 = st - kLook, fed by the requantised block kb2.  Its first MMA overwrites
      // the Wo accumulators: fq_full of block 0 is only reached after every epilogue warp has drained them.
      if (leader) {
        for (int st = kLook; st < FM + kLook; st++) {
          {
            const int kb2 = st - kLook;
            const uint32_t n = blocks + kb2;
            const uint32_t s = n % L::kFS, ph = (n / L::kFS) & 1;
            mbar_wait(&fq_full[s], ph);
            tc_fence_after();
            for (int mb = 0; mb < EM; mb++) cons.mma(tmem_acc + mb * R, opnd_f + s * kOpK, kb2 == 0);
            umma_commit(&fq_free[s]);
          }
        }
        umma_commit(g2_done);
        blocks += FM;
      }
    } else if (warp >= 4) {
      // ===== epilogue warps: TMEM lane = output feature, TMEM column = row of the tile
      const int ew = warp - 4;
      const int q = warp & 3;            // TMEM lane quadrant of this warp
      const int cg = ew >> 2;            // column group: rows [cg * RPW, cg * RPW + RPW)
      const int et = threadIdx.x - 128;  // 0..511
      const uint32_t lane_sel = static_cast<uint32_t>(q * 32) << 16;
      const int kk = q * 32 + lane;      // feature index inside a 128-feature block
      // swizzled byte offset of (row, kk) inside an operand k-block is row * 128 + xo[row & 7]
      uint32_t xo[8];
#pragma unroll
      for (int i = 0; i < 8; i++) xo[i] = static_cast<uint32_t>((((kk >> 4) ^ i) << 4) + (kk & 15));
      // LayerNorm apply phases: thread = (feature, contiguous block of rows)
      constexpr int kParts = kEpiThreads / E;
      constexpr int kRowsPer = R / kParts;
      const int nf = et % E;
      const int nr0 = (et / E) * kRowsPer;
      uint32_t xn[8];
#pragma unroll
      for (int i = 0; i < 8; i++) xn[i] = static_cast<uint32_t>((nf >> 7) * kOpK + ((((nf & 127) >> 4) ^ i) << 4) + (nf & 15));

      // ---- epilogue 0: x = (Wo a + bo) + res -> xs
      mbar_wait(g0_done, tph);
      tc_fence_after();
#pragma unroll 1
      for (int mb = 0; mb < EM; mb++) {
        uint32_t v[RPW];
        tmem_ldn_nowait<RPW>(tmem_acc + lane_sel + mb * R + cg * RPW, v);
        const int f = mb * 128 + kk;
        const float pb = a.pb_o[f];
        float res[RPW];
#pragma unroll
        for (int r = 0; r < RPW; r++) {
          const int grow = row0 + cg * RPW + r;
          res[r] = grow < a.M ? a.res[static_cast<size_t>(grow) * E + f] : 0.0f;
        }
        tmem_ld_wait();
#pragma unroll
        for (int r = 0; r < RPW; r++)
          xs[(cg * RPW + r) * XS + f] = __fadd_rn(dequant<kFast>(static_cast<int>(v[r]), a.um_o, pb), res[r]);
      }
      named_bar_sync(1, kEpiThreads);
      if constexpr (kFast) ln_stats_fast<E, R>(xs, stats, a.eps, ew, lane);
      else if (et < R) ln_stats_row<E>(xs + et * XS, &stats[et], &stats[R + et], a.eps);
      named_bar_sync(1, kEpiThreads);
      // y = LN1(x): residual of the FFN block (kept in xs, or parked in global when xs is about to be reused by
      // the operand ring) and the u8 operand of W1
      {
        const float g = a.ln1_scale[nf], b = a.ln1_bias[nf];
        uint8_t* dst = opnd_y + nr0 * 128;
#pragma unroll 8
        for (int r = 0; r < kRowsPer; r++) {
          const int row = nr0 + r;
          const float y = ln_apply_t<kFast>(xs[row * XS + nf], stats[row], stats[R + row], g, b);
          if constexpr (L::kParkY) {
            const int grow = row0 + row;
            if (grow < a.M) a.y_park[static_cast<size_t>(grow) * E + nf] = y;
          } else {
            xs[row * XS + nf] = y;
          }
          dst[r * 128 + xn[r & 7]] = static_cast<uint8_t>(quantize<kFast>(y, a.aq_1));
        }
      }
      fence_proxy_async();
      if constexpr (L::kParkY) named_bar_sync(1, kEpiThreads);  // xs is dead from here: the operand ring may overwrite it
      __syncwarp();
      if (lane == 0) mbar_arrive(yq_ready);

      // ---- epilogue 1: per FFN1 feature block, relu + requantise -> operand ring slot
#pragma unroll 1
      for (int j = 0; j < FM; j++) {
        const uint32_t n = blocks + j;
        const uint32_t ts = n % L::kTS, tph2 = (n / L::kTS) & 1;
        const uint32_t fs = n % L::kFS, fph = (n / L::kFS) & 1;
        mbar_wait(&slot_full[ts], tph2);
        tc_fence_after();
        uint32_t v[RPW];
        tmem_ldn_nowait<RPW>(tmem_ring + lane_sel + ts * R + cg * RPW, v);
        const float pb = a.pb_1[j * 128 + kk];
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&slot_empty[ts]);
        mbar_wait(&fq_free[fs], fph ^ 1);  // FFN2 has consumed the block that last lived in this slot
        uint8_t* dst = opnd_f + fs * kOpK + cg * RPW * 128;
#pragma unroll
        for (int r = 0; r < RPW; r++) {
          float y = dequant<kFast>(static_cast<int>(v[r]), a.um_1, pb);
          y = fmaxf(y, 0.0f);  // std::max<float>(0, a), TensorOps.cc:163 (NaN -> 0 and -0 -> +0 either way)
          dst[r * 128 + xo[r & 7]] = static_cast<uint8_t>(quantize<kFast>(y, a.aq_2));
        }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&fq_full[fs]);
      }
      blocks += FM;

      // ---- epilogue 2: x = (W2 f + b2) + y -> xs; z = LN2(x) -> global
      mbar_wait(g2_done, tph);
      tc_fence_after();
#pragma unroll 1
      for (int mb = 0; mb < EM; mb++) {
        uint32_t v[RPW];
        tmem_ldn_nowait<RPW>(tmem_acc + lane_sel + mb * R + cg * RPW, v);
        const int f = mb * 128 + kk;
        const float pb = a.pb_2[f];
        float yv[RPW];
#pragma unroll
        for (int r = 0; r < RPW; r++) {
          if constexpr (L::kParkY) {
            const int grow = row0 + cg * RPW + r;
            yv[r] = grow < a.M ? a.y_park[static_cast<size_t>(grow) * E + f] : 0.0f;
          } else {
            yv[r] = xs[(cg * RPW + r) * XS + f];
          }
        }
        tmem_ld_wait();
#pragma unroll
        for (int r = 0; r < RPW; r++)
          xs[(cg * RPW + r) * XS + f] = __fadd_rn(dequant<kFast>(static_cast<int>(v[r]), a.um_2, pb), yv[r]);
      }
      tc_fence_before();
      named_bar_sync(1, kEpiThreads);
      if constexpr (kFast) ln_stats_fast<E, R>(xs, stats, a.eps, ew, lane);
      else if (et < R) ln_stats_row<E>(xs + et * XS, &stats[et], &stats[R + et], a.eps);
      named_bar_sync(1, kEpiThreads);
      {
        const float g = a.ln2_scale[nf], b = a.ln2_bias[nf];
        // consumers' quantised copies: pointers and multipliers in registers, sign handling decided once
        uint8_t* zp[4];
        float za[4];
        int zsub[4];
#pragma unroll
        for (int k = 0; k < 4; k++) {
          zp[k] = k < a.n_zq ? a.zq[k] + static_cast<size_t>(row0) * E + nf : nullptr;
          za[k] = k < a.n_zq ? a.zaq[k] : 0.0f;
          zsub[k] = ((a.zq_signed >> k) & 1) ? 127 : 0;
        }
        float* zo = a.z_out ? a.z_out + static_cast<size_t>(row0) * E + nf : nullptr;
        const int rows_here = min(kRowsPer, a.M - row0 - nr0);
#pragma unroll 4
        for (int r = 0; r < rows_here; r++) {
          const int row = nr0 + r;
          const float z = ln_apply_t<kFast>(xs[row * XS + nf], stats[row], stats[R + row], g, b);
          const size_t o = static_cast<size_t>(row) * E;
          if (zo) zo[o] = z;
#pragma unroll
          for (int k = 0; k < 4; k++)
            if (zp[k]) zp[k][o] = static_cast<uint8_t>(quantize<kFast>(z, za[k]) - zsub[k]);
        }
      }
    }
    // all roles meet before the tile's buffers and once-per-tile barriers are reused
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (warp == 2) tmem_dealloc<512>(tmem);
}

template <int E, int F, int R, bool kFast>
int launch(const RowsFfnArgs& a, cudaStream_t stream) {
  using L = FfnPlan<E, F, R>;
  const int tiles = (a.M + R - 1) / R;
  if (tiles == 0) return 0;
  if (L::kParkY && a.y_park == nullptr) return 1;
  auto kern = rows_ffn_kernel<E, F, R, kFast>;
  ensure_dyn_smem(kern, L::total);
  int sms = 148, dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (launch_pdl(kern, dim3(tiles < sms ? tiles : sms), dim3(kThreads), L::total, stream, a) != cudaSuccess) return 1;
  return 0;
}

}  // namespace

int launch_rows_ffn(const RowsFfnArgs& a, int E, int F, int rows_per_tile, bool fast, cudaStream_t stream) {
  if (E == 256 && F == 1536 && rows_per_tile == 32) return fast ? launch<256, 1536, 32, true>(a, stream) : launch<256, 1536, 32, false>(a, stream);
  if (E == 256 && F == 1536 && rows_per_tile == 128) return fast ? launch<256, 1536, 128, true>(a, stream) : launch<256, 1536, 128, false>(a, stream);
  if (E == 512 && F == 2048 && rows_per_tile == 32) return fast ? launch<512, 2048, 32, true>(a, stream) : launch<512, 2048, 32, false>(a, stream);
  return 1;
}

}  // namespace sb
