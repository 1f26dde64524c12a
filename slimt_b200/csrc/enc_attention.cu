// Encoder self-attention fused with its three input projections (reference: Attention::forward,
// slimt/Modules.cc:287-319 -- linear q/k/v via qmm::affine, split_heads, scaled_dot_product_attention :24-86,
// join_heads; softmax slimt/TensorOps.cc:282-315).  The split path (gemm_i8.cu + self_attention_kernel) writes Q, K
// and V as f32 [R][E] to HBM and reads them back: 24 bytes per element against 3 bytes of u8 input and 1 byte of u8
// output.  Here Q, K and V never leave the SM.
//
// One persistent CTA per SM walks tiles of 128 rows = G = floor(128 / T) whole sentences.  The three quantised copies
// of x (each projection has its own a_quant) sit in shared memory for the whole tile (A operands, M = 128 rows); the
// weights stream head by head through a TMA ring (32 output features of Wq, Wk and Wv per head: B operands, N = 32).
// For head h the MMA thread forms D_q | D_k | D_v in one of four 96-column TMEM regions; TMEM lane = row, so a
// consumer thread owns one query row: it dequantises its row of Q (registers), K and V (parked in a padded f32
// staging tile shared by the four warps of its slot) and then runs the reference's arithmetic unchanged: sequential
// fma chains over the head dimension, scalar softmax in key order, probability-weighted V sum in key order.  Two
// slots of four warps work on alternate heads; a region is handed back to the MMA thread as soon as its
// accumulators are in registers, so the projections of the next heads overlap the attention arithmetic.
//
// Supported: E = 256, 8 heads of 32, T <= 64 (scores are kept in registers).  Everything else takes the split path.
// enc_attention_kernel below takes 33 <= T <= 64; enc_attention_warp_kernel, further down, takes T <= 32.
#include <stdio.h>

#include "exact_math.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kE = 256, kH = 8, kDH = 32;
constexpr int kTileRows = 128;
constexpr int kWStages = 2;
constexpr int kSlots = 2;
constexpr int kConsWarps = 4 * kSlots;
constexpr int kThreadsEa = 128 + 32 * kConsWarps;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 tables, 4.. consumers
constexpr int kTMax = 64;                          // longest sentence enc_attention_kernel holds
constexpr int kStride = 36;                        // floats per staged K / V row: 16-byte aligned, conflict-free
constexpr int kStageRows = kTileRows + 4;          // the score loop reads keys in groups of four
constexpr int kStageBytes = kStageRows * kStride * 4;

struct Smem {
  static constexpr int a = 0;                                  // 3 operands x 2 k-blocks x [128 rows x 128 B]
  static constexpr int w = a + 3 * 32768;                      // ring: 3 matrices x 2 k-blocks x [32 features x 128 B]
  static constexpr int kv = w + kWStages * 24576;              // per slot: K then V staging tiles
  static constexpr int pb = kv + kSlots * 2 * kStageBytes;     // f32 [3][256]
  static constexpr int exp_tab = pb + 3 * kE * 4;              // u64 [32]
  static constexpr int bars = exp_tab + 32 * 8;
  // a_full a_free w_full[kWStages] w_free[kWStages] acc_full[4] acc_free[4]
  static constexpr int n_bars = 2 + 2 * kWStages + 8;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
};
static_assert(Smem::total <= 227 * 1024, "shared memory budget");

__global__ void __launch_bounds__(kThreadsEa, 1) enc_attention_kernel(const __grid_constant__ EncAttnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* s_a = smem + Smem::a;
  uint8_t* s_w = smem + Smem::w;
  float* s_pb = reinterpret_cast<float*>(smem + Smem::pb);
  uint64_t* exp_tab = reinterpret_cast<uint64_t*>(smem + Smem::exp_tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::bars);
  uint64_t* a_full = bars;
  uint64_t* a_free = bars + 1;
  uint64_t* w_full = bars + 2;
  uint64_t* w_free = w_full + kWStages;
  uint64_t* acc_full = w_free + kWStages;
  uint64_t* acc_free = acc_full + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Smem::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.map_aq), tma_prefetch_desc(&a.map_ak), tma_prefetch_desc(&a.map_av);
    tma_prefetch_desc(&a.map_wq), tma_prefetch_desc(&a.map_wk), tma_prefetch_desc(&a.map_wv);
  }
  if (warp == 1 && lane == 0) {
    mbar_init(a_full, 1), mbar_init(a_free, 1);
    for (int i = 0; i < kWStages; i++) mbar_init(&w_full[i], 1), mbar_init(&w_free[i], 1);
    for (int i = 0; i < 4; i++) mbar_init(&acc_full[i], 1), mbar_init(&acc_free[i], 4);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  if (warp == 3) {
    exp_tab[lane] = kExp2fTab[lane];
    for (int i = lane; i < kE; i += 32) {
      s_pb[i] = a.pb_q[i];
      s_pb[kE + i] = a.pb_k[i];
      s_pb[2 * kE + i] = a.pb_v[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();  // the previous kernel's outputs (the quantised x copies) are visible from here on
  const uint32_t tmem = *tmem_slot;

  const int T = a.T;
  const int G = kTileRows / T;  // whole sentences per tile
  const int n_tiles = (a.B + G - 1) / G;

  if (warp == 0) {
    // ===== TMA producer
    if (elect_one()) {
      const CUtensorMap* map_a[3] = {&a.map_aq, &a.map_ak, &a.map_av};
      const CUtensorMap* map_w[3] = {&a.map_wq, &a.map_wk, &a.map_wv};
      uint32_t hc = 0, it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        const int row0 = tile * G * T;
        mbar_wait(a_free, (it & 1) ^ 1);
        mbar_expect_tx(a_full, 3 * 32768);
        for (int m = 0; m < 3; m++)
          for (int kb = 0; kb < 2; kb++) tma_load_2d(s_a + m * 32768 + kb * 16384, map_a[m], a_full, kb * 128, row0);
        for (int h = 0; h < kH; h++, hc++) {
          const uint32_t s = hc % kWStages, ph = (hc / kWStages) & 1;
          mbar_wait(&w_free[s], ph ^ 1);
          mbar_expect_tx(&w_full[s], 24576);
          for (int m = 0; m < 3; m++)
            for (int kb = 0; kb < 2; kb++)
              tma_load_2d(s_w + s * 24576 + m * 8192 + kb * 4096, map_w[m], &w_full[s], kb * 128, h * kDH);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: per head, D_q | D_k | D_v = (x quantised for that projection) x (the head's 32 features)
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_i8(kTileRows, kDH);  // A = u8 rows, B = s8 weights
      uint32_t hc = 0, it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        mbar_wait(a_full, it & 1);
        for (int h = 0; h < kH; h++, hc++) {
          const uint32_t s = hc % kWStages;
          const uint32_t reg = hc & 3;
          mbar_wait(&w_full[s], (hc / kWStages) & 1);
          mbar_wait(&acc_free[reg], ((hc >> 2) & 1) ^ 1);
          tc_fence_after();
#pragma unroll
          for (int m = 0; m < 3; m++) {
#pragma unroll
            for (int kb = 0; kb < 2; kb++) {
              const uint64_t da = make_kmajor_sw128_desc(smem_u32(s_a + m * 32768 + kb * 16384));
              const uint64_t db = make_kmajor_sw128_desc(smem_u32(s_w + s * 24576 + m * 8192 + kb * 4096));
#pragma unroll
              for (int k = 0; k < 4; k++) umma_i8(tmem + reg * 128 + m * 32, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
            }
          }
          umma_commit(&w_free[s]);
          umma_commit(&acc_full[reg]);
        }
        umma_commit(a_free);
      }
    }
  } else if (warp >= 4) {
    // ===== consumers: thread = query row of the tile
    const int slot = (warp - 4) >> 2;
    const int qd = warp & 3;
    const int r = qd * 32 + lane;
    const uint32_t lane_sel = static_cast<uint32_t>(qd * 32) << 16;
    float* Ks = reinterpret_cast<float*>(smem + Smem::kv + slot * 2 * kStageBytes);
    float* Vs = Ks + kStageRows * kStride;
    const float ninf = -3.402823466e+38f;
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
      const int j = r / T, i = r - j * T;
      const int b = tile * G + j;
      const bool sent_ok = j < G && b < a.B;
      const int len = sent_ok ? min(static_cast<int>(__ldg(a.lengths + b)), T) : 0;
      const int krow0 = sent_ok ? j * T : 0;
      int wmax = len;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
      const bool row_live = sent_ok && i < len;
      uint8_t* out_row = a.out_q + (static_cast<size_t>(tile) * G * T + r) * kE;

#pragma unroll 1
      for (int hh = 0; hh < kH / kSlots; hh++) {
        const int h = hh * kSlots + slot;
        const uint32_t reg = h & 3;
        const uint32_t use = it * 2 + (h >> 2);
        float q[kDH];
        {
          uint32_t vq[32], vk[32], vv[32];
          mbar_wait(&acc_full[reg], use & 1);
          tc_fence_after();
          const uint32_t taddr = tmem + lane_sel + reg * 128;
          tmem_ld32_nowait(taddr + 32, vk);
          tmem_ld32_nowait(taddr + 64, vv);
          tmem_ld32_nowait(taddr, vq);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_free[reg]);
          named_bar_sync(1 + slot, 128);  // the slot's warps are done reading the previous head's K and V
          const float* pbk = s_pb + kE + h * kDH;
          const float* pbv = s_pb + 2 * kE + h * kDH;
          float* kr = Ks + r * kStride;
          float* vr = Vs + r * kStride;
#pragma unroll
          for (int d = 0; d < kDH; d += 4) {
            const float4 pk = *reinterpret_cast<const float4*>(pbk + d);
            const float4 pv = *reinterpret_cast<const float4*>(pbv + d);
            *reinterpret_cast<float4*>(kr + d) =
                make_float4(dequant1(static_cast<int>(vk[d]), a.um_k, pk.x), dequant1(static_cast<int>(vk[d + 1]), a.um_k, pk.y),
                            dequant1(static_cast<int>(vk[d + 2]), a.um_k, pk.z), dequant1(static_cast<int>(vk[d + 3]), a.um_k, pk.w));
            *reinterpret_cast<float4*>(vr + d) =
                make_float4(dequant1(static_cast<int>(vv[d]), a.um_v, pv.x), dequant1(static_cast<int>(vv[d + 1]), a.um_v, pv.y),
                            dequant1(static_cast<int>(vv[d + 2]), a.um_v, pv.z), dequant1(static_cast<int>(vv[d + 3]), a.um_v, pv.w));
          }
          const float* pbq = s_pb + h * kDH;
#pragma unroll
          for (int d = 0; d < kDH; d += 4) {
            const float4 pq = *reinterpret_cast<const float4*>(pbq + d);
            q[d] = dequant1(static_cast<int>(vq[d]), a.um_q, pq.x);
            q[d + 1] = dequant1(static_cast<int>(vq[d + 1]), a.um_q, pq.y);
            q[d + 2] = dequant1(static_cast<int>(vq[d + 2]), a.um_q, pq.z);
            q[d + 3] = dequant1(static_cast<int>(vq[d + 3]), a.um_q, pq.w);
          }
          named_bar_sync(1 + slot, 128);  // K and V of every row of the tile are staged
        }

        // scores: four keys at a time (independent chains); each chain is the reference's sequential fma order
        float S[kTMax];
        float mx = ninf;
#pragma unroll
        for (int j0 = 0; j0 < kTMax; j0 += 4) {
          if (j0 < wmax) {
            const float* kp = Ks + (krow0 + j0) * kStride;
            float s0 = 0.0f, s1 = 0.0f, s2 = 0.0f, s3 = 0.0f;
#pragma unroll
            for (int d = 0; d < kDH; d += 4) {
              const float4 k0 = *reinterpret_cast<const float4*>(kp + d);
              const float4 k1 = *reinterpret_cast<const float4*>(kp + kStride + d);
              const float4 k2 = *reinterpret_cast<const float4*>(kp + 2 * kStride + d);
              const float4 k3 = *reinterpret_cast<const float4*>(kp + 3 * kStride + d);
              s0 = fmaf(q[d], k0.x, s0), s1 = fmaf(q[d], k1.x, s1), s2 = fmaf(q[d], k2.x, s2), s3 = fmaf(q[d], k3.x, s3);
              s0 = fmaf(q[d + 1], k0.y, s0), s1 = fmaf(q[d + 1], k1.y, s1), s2 = fmaf(q[d + 1], k2.y, s2), s3 = fmaf(q[d + 1], k3.y, s3);
              s0 = fmaf(q[d + 2], k0.z, s0), s1 = fmaf(q[d + 2], k1.z, s1), s2 = fmaf(q[d + 2], k2.z, s2), s3 = fmaf(q[d + 2], k3.z, s3);
              s0 = fmaf(q[d + 3], k0.w, s0), s1 = fmaf(q[d + 3], k1.w, s1), s2 = fmaf(q[d + 3], k2.w, s2), s3 = fmaf(q[d + 3], k3.w, s3);
            }
            S[j0] = j0 < len ? __fmul_rn(a.dk, s0) : ninf;
            S[j0 + 1] = j0 + 1 < len ? __fmul_rn(a.dk, s1) : ninf;
            S[j0 + 2] = j0 + 2 < len ? __fmul_rn(a.dk, s2) : ninf;
            S[j0 + 3] = j0 + 3 < len ? __fmul_rn(a.dk, s3) : ninf;
            mx = fmaxf(fmaxf(fmaxf(mx, S[j0]), fmaxf(S[j0 + 1], S[j0 + 2])), S[j0 + 3]);
          } else {
            S[j0] = S[j0 + 1] = S[j0 + 2] = S[j0 + 3] = ninf;
          }
        }
        // softmax (TensorOps.cc:282-315): exp(s - max), sum in key order; masked keys contribute exactly +0
        float sum = 0.0f;
#pragma unroll
        for (int j0 = 0; j0 < kTMax; j0 += 4) {
          if (j0 < wmax) {
#pragma unroll
            for (int u = 0; u < 4; u++) {
              const float e = j0 + u < len ? expf_glibc_nonpos_tab(__fsub_rn(S[j0 + u], mx), exp_tab) : 0.0f;
              S[j0 + u] = e;
              sum = __fadd_rn(sum, e);
            }
          }
        }
        float acc[kDH];
#pragma unroll
        for (int d = 0; d < kDH; d++) acc[d] = 0.0f;
        // every probability of the row divides by `sum`: reciprocal once, three FFMAs per key (exact_math.cuh)
        const float sum_rcp = rcp_refined(sum);
        const float sum_lo = div_guard_lo(sum);
#pragma unroll
        for (int j0 = 0; j0 < kTMax; j0 += 4) {
          if (j0 < wmax) {
#pragma unroll
            for (int u = 0; u < 4; u++) {
              if (j0 + u < wmax) {
                const float p = j0 + u < len ? div_by_rcp(S[j0 + u], sum, sum_rcp, sum_lo) : 0.0f;
                const float* vp = Vs + (krow0 + j0 + u) * kStride;
#pragma unroll
                for (int d = 0; d < kDH; d += 4) {
                  const float4 v4 = *reinterpret_cast<const float4*>(vp + d);
                  acc[d] = fmaf(p, v4.x, acc[d]);
                  acc[d + 1] = fmaf(p, v4.y, acc[d + 1]);
                  acc[d + 2] = fmaf(p, v4.z, acc[d + 2]);
                  acc[d + 3] = fmaf(p, v4.w, acc[d + 3]);
                }
              }
            }
          }
        }
        if (sent_ok) {
          // padded query rows never reach a valid output; like the split path they carry quantize(0)
          uint32_t wq[8];
#pragma unroll
          for (int d = 0; d < kDH; d += 4)
            wq[d >> 2] = row_live ? pack4(quantize1(acc[d], a.aq_out), quantize1(acc[d + 1], a.aq_out),
                                          quantize1(acc[d + 2], a.aq_out), quantize1(acc[d + 3], a.aq_out))
                                  : 0x7f7f7f7fu;
          uint4* o = reinterpret_cast<uint4*>(out_row + h * kDH);
          o[0] = make_uint4(wq[0], wq[1], wq[2], wq[3]);
          o[1] = make_uint4(wq[4], wq[5], wq[6], wq[7]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// ---------------------------------------------------------------------------------------------------------------------
// T <= 32: one WARP per (sentence, head), register-tiled.  In the kernel above every K and V element reaches a thread
// as a broadcast 16-byte shared-memory load that feeds four FMAs, and that load -- eight issue cycles per scheduler --
// is what the inner loops cost.  At T <= 32 this kernel takes 241 us per layer, where one thread per query row took 347
// and two threads per row 313 (DESIGN.md 4.3).  Here a tile is four sentences, each in its own 32-row slot of
// the A operands (its own TMA box), so TMEM lane quadrant qd = sentence qd and the warp that drains a quadrant owns the
// whole attention of that sentence for the head: no barrier wider than the warp.  The warp parks Q and K transposed
// ([d][row], conflict-free scalar stores), then works like a register-tiled SGEMM whose every output is still ONE
// thread's chain in index order:
//   scores   thread = 4 queries x 8 keys: three 16-byte loads (q quad, two k quads) per 32 FMAs, chains over d;
//   softmax  a row's 32 keys live in the four adjacent lanes of its query group: max by two shuffles (order-free), exp
//            elementwise, the row sum handed from lane to lane so that it is one chain in key order, p = e / sum;
//   P V      P parked transposed in K's place, V (drained from TMEM only now) in Q's place; thread = 4 queries x 8 dims,
//            three loads per 32 FMAs, chains over the valid keys in order (a masked key adds exactly +0: skipped).
// Bit-identical to the kernel above and to the split path (test_fused_encoder_attention_equals_split_path).
// Twelve consumer warps (three per scheduler: the phases of a unit are latency chains, the third warp fills their gaps)
// take the CTA's (tile, head) units round-robin.  That many staging tiles only fit because they are unpadded
// ([32][32] floats with XOR-swizzled 16-byte chunks where a padded row used to avoid the bank conflicts) and the weight
// ring has ONE stage: the MMA of a head is ~1 k cycles of a ~9 k-cycle unit, its weights need no prefetch distance.
// (The two FMA loops are unrolled by 2 only: twelve warps walk the unit's code at different places, and at 8 / 4 its body
// no longer fitted the instruction cache -- ncu: no_instruction the second-largest stall, 256 vs 241 us.  Giving the four
// query rows turns in one copy of the softmax code shrank it further but cost more in lost overlap: 259 us.)
constexpr int kWSlots = 3;
constexpr int kWWarps = 4 * kWSlots;
constexpr int kThreadsW = 128 + 32 * kWWarps;
constexpr int kWarpBuf = 32 * 32;  // floats: one [32][32] staging tile

struct SmemW {
  static constexpr int a = 0;                              // 3 operands x 2 k-blocks x [128 rows x 128 B]
  static constexpr int w = a + 3 * 32768;                  // 3 matrices x 2 k-blocks x [32 features x 128 B], one stage
  static constexpr int kv = w + 24576;                     // per warp: two staging tiles
  static constexpr int pb = kv + kWWarps * 2 * kWarpBuf * 4;  // f32 [3][256]
  static constexpr int exp_tab = pb + 3 * kE * 4;          // u64 [32]
  static constexpr int bars = exp_tab + 32 * 8;
  // a_full a_free w_full w_free acc_full[4] acc_free[4]
  static constexpr int n_bars = 4 + 8;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
};
static_assert(SmemW::total <= 227 * 1024, "shared memory budget");

__global__ void __launch_bounds__(kThreadsW, 1) enc_attention_warp_kernel(const __grid_constant__ EncAttnArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* s_a = smem + SmemW::a;
  uint8_t* s_w = smem + SmemW::w;
  float* s_pb = reinterpret_cast<float*>(smem + SmemW::pb);
  uint64_t* exp_tab = reinterpret_cast<uint64_t*>(smem + SmemW::exp_tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SmemW::bars);
  uint64_t* a_full = bars;
  uint64_t* a_free = bars + 1;
  uint64_t* w_full = bars + 2;
  uint64_t* w_free = bars + 3;
  uint64_t* acc_full = bars + 4;
  uint64_t* acc_free = acc_full + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SmemW::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.map_aq32), tma_prefetch_desc(&a.map_ak32), tma_prefetch_desc(&a.map_av32);
    tma_prefetch_desc(&a.map_wq), tma_prefetch_desc(&a.map_wk), tma_prefetch_desc(&a.map_wv);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 4; i++) mbar_init(&bars[i], 1);
    for (int i = 0; i < 4; i++) mbar_init(&acc_full[i], 1), mbar_init(&acc_free[i], 4);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  if (warp == 3) {
    exp_tab[lane] = kExp2fTab[lane];
    for (int i = lane; i < kE; i += 32) {
      s_pb[i] = a.pb_q[i];
      s_pb[kE + i] = a.pb_k[i];
      s_pb[2 * kE + i] = a.pb_v[i];
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();  // the previous kernel's outputs (the quantised x copies) are visible from here on
  const uint32_t tmem = *tmem_slot;

  const int T = a.T;
  constexpr int G = 4;  // sentences per tile, one per 32-row slot
  const int n_tiles = (a.B + G - 1) / G;

  if (warp == 0) {
    // ===== TMA producer: every sentence's rows into its own slot (rows past the sentence are the next sentence's, or
    // zero fill past the tensor: they are masked as keys and never stored as queries)
    if (elect_one()) {
      const CUtensorMap* map_a[3] = {&a.map_aq32, &a.map_ak32, &a.map_av32};
      const CUtensorMap* map_w[3] = {&a.map_wq, &a.map_wk, &a.map_wv};
      uint32_t hc = 0, it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        mbar_wait(a_free, (it & 1) ^ 1);
        mbar_expect_tx(a_full, 3 * 32768);
        for (int m = 0; m < 3; m++)
          for (int kb = 0; kb < 2; kb++)
            for (int j = 0; j < G; j++)
              tma_load_2d(s_a + m * 32768 + kb * 16384 + j * 4096, map_a[m], a_full, kb * 128, (tile * G + j) * T);
        for (int h = 0; h < kH; h++, hc++) {
          mbar_wait(w_free, (hc & 1) ^ 1);
          mbar_expect_tx(w_full, 24576);
          for (int m = 0; m < 3; m++)
            for (int kb = 0; kb < 2; kb++) tma_load_2d(s_w + m * 8192 + kb * 4096, map_w[m], w_full, kb * 128, h * kDH);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer: per head, D_q | D_k | D_v = (x quantised for that projection) x (the head's 32 features)
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_i8(kTileRows, kDH);
      uint32_t hc = 0, it = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, it++) {
        mbar_wait(a_full, it & 1);
        for (int h = 0; h < kH; h++, hc++) {
          const uint32_t reg = hc & 3;
          mbar_wait(w_full, hc & 1);
          mbar_wait(&acc_free[reg], ((hc >> 2) & 1) ^ 1);
          tc_fence_after();
#pragma unroll
          for (int m = 0; m < 3; m++) {
#pragma unroll
            for (int kb = 0; kb < 2; kb++) {
              const uint64_t da = make_kmajor_sw128_desc(smem_u32(s_a + m * 32768 + kb * 16384));
              const uint64_t db = make_kmajor_sw128_desc(smem_u32(s_w + m * 8192 + kb * 4096));
#pragma unroll
              for (int k = 0; k < 4; k++) umma_i8(tmem + reg * 128 + m * 32, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
            }
          }
          umma_commit(w_free);
          umma_commit(&acc_full[reg]);
        }
        umma_commit(a_free);
      }
    }
  } else if (warp >= 4) {
    // ===== consumers: warp = (slot, sentence qd of the tile); slot s takes the CTA's units s, s + 3, s + 6, ...
    // (unit u = head u % 8 of the CTA's tile u / 8; its accumulators sit in TMEM region u % 4)
    const int slot = (warp - 4) >> 2;
    const int qd = warp & 3;
    const uint32_t lane_sel = static_cast<uint32_t>(qd * 32) << 16;
    float* buf0 = reinterpret_cast<float*>(smem + SmemW::kv) + (warp - 4) * 2 * kWarpBuf;  // Q^T, later V
    float* buf1 = buf0 + kWarpBuf;                                                          // K^T, later P^T
    const int ty = lane >> 2, tx = lane & 3;
    const float ninf = -3.402823466e+38f;
    const int my_tiles = blockIdx.x < static_cast<unsigned>(n_tiles) ? (n_tiles - 1 - static_cast<int>(blockIdx.x)) / static_cast<int>(gridDim.x) + 1 : 0;
    const int n_units = my_tiles * kH;
    auto sentence_of = [&](int u) { return (static_cast<int>(blockIdx.x) + (u >> 3) * static_cast<int>(gridDim.x)) * G + qd; };
    // the next unit's sentence length is requested a unit ahead (raw; clamped at use)
    int len_nx = 0;
    if (slot < n_units) {
      const int b = sentence_of(slot);
      len_nx = b < a.B ? static_cast<int>(__ldg(a.lengths + b)) : 0;
    }
#pragma unroll 1
    for (int u = slot; u < n_units; u += kWSlots) {
      const int h = u & 7;
      const uint32_t reg = u & 3;
      const int b = sentence_of(u);
      const int len = min(len_nx, T);
      if (u + kWSlots < n_units) {
        const int bn = sentence_of(u + kWSlots);
        len_nx = bn < a.B ? static_cast<int>(__ldg(a.lengths + bn)) : 0;
      }
      uint8_t* out_base = a.out_q + static_cast<size_t>(b) * T * kE;
      const uint32_t taddr = tmem + lane_sel + reg * 128;
      mbar_wait(&acc_full[reg], (u >> 2) & 1);
      tc_fence_after();
      if (len == 0) {  // no sentence in this slot (or an empty one): hand the region back untouched
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_free[reg]);
        if (b < a.B)  // an empty sentence: its padded query rows carry quantize(0)
          for (int i = ty; i < T; i += 8)
            *reinterpret_cast<uint2*>(out_base + static_cast<size_t>(i) * kE + h * kDH + 8 * tx) = make_uint2(0x7f7f7f7fu, 0x7f7f7f7fu);
        continue;
      }
      {
        // ---- Q and K of this lane's row -> f32, parked transposed ([d][row]: a row's value of dimension d)
        uint32_t vq[32], vk[32];
        tmem_ld32_nowait(taddr, vq);
        tmem_ld32_nowait(taddr + 32, vk);
        tmem_ld_wait();
        const float* pbq = s_pb + h * kDH;
        const float* pbk = s_pb + kE + h * kDH;
#pragma unroll
        for (int d = 0; d < kDH; d += 4) {
          const float4 pq = *reinterpret_cast<const float4*>(pbq + d);
          const float4 pk = *reinterpret_cast<const float4*>(pbk + d);
          buf0[(d + 0) * 32 + lane] = dequant1(static_cast<int>(vq[d]), a.um_q, pq.x);
          buf0[(d + 1) * 32 + lane] = dequant1(static_cast<int>(vq[d + 1]), a.um_q, pq.y);
          buf0[(d + 2) * 32 + lane] = dequant1(static_cast<int>(vq[d + 2]), a.um_q, pq.z);
          buf0[(d + 3) * 32 + lane] = dequant1(static_cast<int>(vq[d + 3]), a.um_q, pq.w);
          buf1[(d + 0) * 32 + lane] = dequant1(static_cast<int>(vk[d]), a.um_k, pk.x);
          buf1[(d + 1) * 32 + lane] = dequant1(static_cast<int>(vk[d + 1]), a.um_k, pk.y);
          buf1[(d + 2) * 32 + lane] = dequant1(static_cast<int>(vk[d + 2]), a.um_k, pk.z);
          buf1[(d + 3) * 32 + lane] = dequant1(static_cast<int>(vk[d + 3]), a.um_k, pk.w);
        }
      }
      __syncwarp();

      // ---- scores: queries 4 ty .. + 3 against keys 8 tx .. + 7, each a sequential fma chain over d
      float sc[4][8];
#pragma unroll
      for (int x = 0; x < 4; x++)
#pragma unroll
        for (int w = 0; w < 8; w++) sc[x][w] = 0.0f;
#pragma unroll 2
      for (int d = 0; d < kDH; d++) {
        const float4 q4 = *reinterpret_cast<const float4*>(buf0 + d * 32 + 4 * ty);
        const float4 ka = *reinterpret_cast<const float4*>(buf1 + d * 32 + 8 * tx);
        const float4 kb = *reinterpret_cast<const float4*>(buf1 + d * 32 + 8 * tx + 4);
        const float qv[4] = {q4.x, q4.y, q4.z, q4.w};
        const float kv[8] = {ka.x, ka.y, ka.z, ka.w, kb.x, kb.y, kb.z, kb.w};
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
          for (int w = 0; w < 8; w += 2) ffma2(sc[x][w], sc[x][w + 1], qv[x], qv[x], kv[w], kv[w + 1]);
      }
      // ---- softmax per query row (TensorOps.cc:282-315): masked keys score -inf and contribute exactly +0
      float mx[4], sum[4];
#pragma unroll
      for (int x = 0; x < 4; x++) {
        mx[x] = ninf;
#pragma unroll
        for (int w = 0; w < 8; w++) {
          sc[x][w] = 8 * tx + w < len ? __fmul_rn(a.dk, sc[x][w]) : ninf;
          mx[x] = fmaxf(mx[x], sc[x][w]);
        }
        mx[x] = fmaxf(mx[x], __shfl_xor_sync(0xffffffffu, mx[x], 1));
        mx[x] = fmaxf(mx[x], __shfl_xor_sync(0xffffffffu, mx[x], 2));
      }
#pragma unroll
      for (int w = 0; w < 8; w++) {
        if (8 * tx + w < len) {
#pragma unroll
          for (int x = 0; x < 4; x++) sc[x][w] = expf_glibc_nonpos_tab(__fsub_rn(sc[x][w], mx[x]), exp_tab);
        } else {
#pragma unroll
          for (int x = 0; x < 4; x++) sc[x][w] = 0.0f;
        }
      }
      // the row sum in key order: lane tx = 0 adds keys 0..7, hands the partial sum to tx = 1, and so on
#pragma unroll
      for (int x = 0; x < 4; x++) sum[x] = 0.0f;
#pragma unroll
      for (int t = 0; t < 4; t++) {
#pragma unroll
        for (int x = 0; x < 4; x++) {
          const float in = __shfl_sync(0xffffffffu, sum[x], (lane & ~3) | (t > 0 ? t - 1 : 0));
          if (tx == t) {
            float acc1 = t == 0 ? 0.0f : in;
#pragma unroll
            for (int w = 0; w < 8; w++) acc1 = __fadd_rn(acc1, sc[x][w]);
            sum[x] = acc1;
          }
        }
      }
      __syncwarp();  // every lane is done reading K^T: its place takes P^T
#pragma unroll
      for (int x = 0; x < 4; x++) {
        sum[x] = __shfl_sync(0xffffffffu, sum[x], (lane & ~3) | 3);
        const float rc = rcp_refined(sum[x]), lo = div_guard_lo(sum[x]);
#pragma unroll
        for (int w = 0; w < 8; w++) sc[x][w] = div_by_rcp(sc[x][w], sum[x], rc, lo);
      }
      // P^T[key][query quad]: quad ty of key row j sits at chunk ty ^ 2 (j / 8) (conflict-free stores and loads)
#pragma unroll
      for (int w = 0; w < 8; w++)
        *reinterpret_cast<float4*>(buf1 + (8 * tx + w) * 32 + 4 * (ty ^ (2 * tx))) = make_float4(sc[0][w], sc[1][w], sc[2][w], sc[3][w]);
      {
        // ---- V of this lane's key row -> f32 in Q^T's place ([key][d], 16-byte chunk c at position c ^ (key & 7)); the
        // TMEM region is free after this
        uint32_t vv[32];
        tmem_ld32_nowait(taddr + 64, vv);
        tmem_ld_wait();
        tc_fence_before();
        const float* pbv = s_pb + 2 * kE + h * kDH;
#pragma unroll
        for (int d = 0; d < kDH; d += 4) {
          const float4 pv = *reinterpret_cast<const float4*>(pbv + d);
          *reinterpret_cast<float4*>(buf0 + lane * 32 + 4 * ((d >> 2) ^ (lane & 7))) =
              make_float4(dequant1(static_cast<int>(vv[d]), a.um_v, pv.x), dequant1(static_cast<int>(vv[d + 1]), a.um_v, pv.y),
                          dequant1(static_cast<int>(vv[d + 2]), a.um_v, pv.z), dequant1(static_cast<int>(vv[d + 3]), a.um_v, pv.w));
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&acc_free[reg]);

      // ---- P V: queries 4 ty .. + 3, dims 8 tx .. + 7, one chain per output over the valid keys in order
      float acc[4][8];
#pragma unroll
      for (int x = 0; x < 4; x++)
#pragma unroll
        for (int w = 0; w < 8; w++) acc[x][w] = 0.0f;
#pragma unroll 2
      for (int j = 0; j < len; j++) {
        const float4 p4 = *reinterpret_cast<const float4*>(buf1 + j * 32 + 4 * (ty ^ (2 * (j >> 3))));
        const float4 va = *reinterpret_cast<const float4*>(buf0 + j * 32 + 4 * ((2 * tx) ^ (j & 7)));
        const float4 vb = *reinterpret_cast<const float4*>(buf0 + j * 32 + 4 * ((2 * tx + 1) ^ (j & 7)));
        const float pv[4] = {p4.x, p4.y, p4.z, p4.w};
        const float vv[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
#pragma unroll
        for (int x = 0; x < 4; x++)
#pragma unroll
          for (int w = 0; w < 8; w += 2) ffma2(acc[x][w], acc[x][w + 1], pv[x], pv[x], vv[w], vv[w + 1]);
      }
      // ---- Wo's operand: 8 bytes per (query row, thread); padded query rows carry quantize(0) like the split path
#pragma unroll
      for (int x = 0; x < 4; x++) {
        const int i = 4 * ty + x;
        if (i < T) {
          uint2 o = make_uint2(0x7f7f7f7fu, 0x7f7f7f7fu);
          if (i < len) {
            o.x = pack4(quantize1(acc[x][0], a.aq_out), quantize1(acc[x][1], a.aq_out), quantize1(acc[x][2], a.aq_out),
                        quantize1(acc[x][3], a.aq_out));
            o.y = pack4(quantize1(acc[x][4], a.aq_out), quantize1(acc[x][5], a.aq_out), quantize1(acc[x][6], a.aq_out),
                        quantize1(acc[x][7], a.aq_out));
          }
          *reinterpret_cast<uint2*>(out_base + static_cast<size_t>(i) * kE + h * kDH + 8 * tx) = o;
        }
      }
      __syncwarp();  // the staging tiles are rewritten by the next unit
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

}  // namespace

bool enc_attention_supported(int E, int H, int dh, int T) { return E == kE && H == kH && dh == kDH && T >= 1 && T <= kTMax; }

int launch_enc_attention(const EncAttnArgs& a, int num_sms, cudaStream_t stream) {
  if (a.B == 0) return 0;
  if (a.T <= 32) {
    const int tiles = (a.B + 3) / 4;
    if (ensure_dyn_smem(enc_attention_warp_kernel, SmemW::total) != cudaSuccess) return 1;
    return launch_pdl(enc_attention_warp_kernel, dim3(tiles < num_sms ? tiles : num_sms), dim3(kThreadsW), SmemW::total, stream,
                      a) != cudaSuccess;
  }
  const int G = kTileRows / a.T;
  const int tiles = (a.B + G - 1) / G;
  if (ensure_dyn_smem(enc_attention_kernel, Smem::total) != cudaSuccess) return 1;
  return launch_pdl(enc_attention_kernel, dim3(tiles < num_sms ? tiles : num_sms), dim3(kThreadsEa), Smem::total, stream, a) !=
         cudaSuccess;
}

}  // namespace sb
