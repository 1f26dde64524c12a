// Decoder cross-attention with recomputed K / V for LONG source sentences (65 .. 256 tokens): the sentence-at-a-time
// sibling of cross_attention_rc.cu (reference: Attention::forward, slimt/Modules.cc:287-319 — K and V re-projected on
// every step, :244-249 — and scaled_dot_product_attention :24-86; softmax slimt/TensorOps.cc:282-315).
//
// The cached kernel (cross_attention.cu) streams 2 * len * E * 4 bytes of f32 K / V per sentence, layer and step and sits
// at 90 % of the HBM roofline on the mixed-length workload; this kernel reads the projections' INPUT instead — the u8
// PrepareA bytes of the encoder output, 4x fewer bytes — and rebuilds K = dequant(qa_k Wk), V = dequant(qa_v Wv) with
// tcgen05.mma kind::i8: exact int32 accumulators, the same two roundings, so every float is the one the cache held.
//
// One persistent CTA per SM takes whole sentences (b = blockIdx.x, += gridDim.x).  A sentence is ng = ceil(len / 128)
// GROUPS of 128 key rows (the 128 TMEM lanes); its operand tiles travel through a two-stage 32 KB ring in consumption
// order  K(0) .. K(ng-1), V(0) .. V(ng-1):
//   K group   D_k[key][feature] = qa_k tile (A, M = 128) x Wk (B, N = 256).  Consumer warp (lane quadrant qd, head
//             pair sub): lane = key, the reference's sequential fma chain of two heads against q; scores stay in
//             registers until every group of the sentence is in.
//   softmax   per head over ALL the sentence's keys: block maxima meet in shared memory (a maximum has no order), the
//             exponentials are parked, ONE warp per head forms the sum in key order, every thread divides its own.
//   V group   D_v[feature][key] = Wv (A, 2 x M = 128) x qa_v tile (B, N = 128).  lane = output feature: one chain over
//             the sentence's keys in order, carried across the groups.  256 features = 8 warps; the other 8 wait (a
//             chain cannot be split, and two warps per scheduler already fill the issue slots of this phase).
// Keys past the sentence's length have probability exactly 0 and change no chain (x + 0 * v = x).
// Supported: E = 256, 8 heads of 32, S <= 256, bit-exact arithmetic mode.
#include <stdio.h>

#include "exact_math.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kE = 256, kH = 8, kDH = 32;
constexpr int kKeys = 32;         // key rows per TMA box
constexpr int kGKeys = 128;       // key rows per group
constexpr int kMaxS = 256;
constexpr int kMaxGroups = kMaxS / kGKeys;
constexpr int kConsWarps = 16;
constexpr int kConsThreads = kConsWarps * 32;
constexpr int kThreadsL = 128 + kConsThreads;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 tables, 4..19 consumers
constexpr int kTile = 32 * 1024;               // one operand tile: 2 k-blocks x [128 key rows x 128 B]

struct SmemL {
  static constexpr int wk = 0;                        // 2 k-blocks x [256 features x 128 B]
  static constexpr int wv = wk + 64 * 1024;
  static constexpr int ring = wv + 64 * 1024;         // 2 operand tiles
  static constexpr int qs = ring + 2 * kTile;         // f32 [2 buffers][256]
  static constexpr int ps = qs + 2 * kE * 4;          // f32 [8 heads][256 keys]
  static constexpr int pbk = ps + kH * kMaxS * 4;     // f32 [256]
  static constexpr int pmax = pbk + kE * 4;           // f32 [4 key blocks][8 heads]
  static constexpr int psum = pmax + 4 * kH * 4;      // f32 [8 heads]
  static constexpr int exp_tab = psum + kH * 4;       // u64 [32]
  static constexpr int bars = exp_tab + 32 * 8;
  // w_full full[2] empty[2] k_done v_done k_drained v_drained
  static constexpr int n_bars = 9;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
  static_assert(total <= 227 * 1024, "shared memory");
};

__device__ __forceinline__ int groups_of(int len) { return len > kGKeys ? 2 : 1; }

__global__ void __launch_bounds__(kThreadsL, 1) cross_attention_rcl_kernel(const __grid_constant__ CrossRcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* s_wk = smem + SmemL::wk;
  uint8_t* s_wv = smem + SmemL::wv;
  uint8_t* s_ring = smem + SmemL::ring;
  float* s_q_all = reinterpret_cast<float*>(smem + SmemL::qs);
  float* s_p = reinterpret_cast<float*>(smem + SmemL::ps);
  float* s_pbk = reinterpret_cast<float*>(smem + SmemL::pbk);
  float* s_pmax = reinterpret_cast<float*>(smem + SmemL::pmax);
  float* s_psum = reinterpret_cast<float*>(smem + SmemL::psum);
  uint64_t* exp_tab = reinterpret_cast<uint64_t*>(smem + SmemL::exp_tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SmemL::bars);
  uint64_t* w_full = bars;
  uint64_t* full = bars + 1;
  uint64_t* empty = bars + 3;
  uint64_t* k_done = bars + 5;
  uint64_t* v_done = bars + 6;
  uint64_t* k_drained = bars + 7;
  uint64_t* v_drained = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SmemL::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.map_ak);
    tma_prefetch_desc(&a.map_av);
    tma_prefetch_desc(&a.map_wk);
    tma_prefetch_desc(&a.map_wv);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 7; i++) mbar_init(&bars[i], 1);
    mbar_init(k_drained, kConsWarps);
    mbar_init(v_drained, kConsWarps / 2);  // the eight warps that own output features
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  if (warp == 3) {
    exp_tab[lane] = kExp2fTab[lane];
    for (int i = lane; i < kE; i += 32) s_pbk[i] = a.pb_k[i];
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();  // everything above overlapped the previous kernel's tail; its outputs are visible from here on
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_k = tmem;        // 256 columns: features
  const uint32_t tmem_v = tmem + 256;  // 2 blocks x 128 columns: key rows of the group

  auto length_of = [&](int b) { return max(1, min(static_cast<int>(__ldg(a.lengths + b)), a.T)); };

  if (warp == 0) {
    // ===== TMA producer: Wk, Wv once, then every sentence's operand tiles in consumption order
    if (elect_one()) {
      mbar_expect_tx(w_full, 128 * 1024);
      for (int kb = 0; kb < 2; kb++)
        for (int half = 0; half < 2; half++) {
          tma_load_2d(s_wk + kb * 32768 + half * 16384, &a.map_wk, w_full, kb * 128, half * 128);
          tma_load_2d(s_wv + kb * 32768 + half * 16384, &a.map_wv, w_full, kb * 128, half * 128);
        }
      uint32_t tile = 0;
      for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        const int ng = groups_of(length_of(b));
        for (int pass = 0; pass < 2; pass++) {
          const CUtensorMap* map = pass == 0 ? &a.map_ak : &a.map_av;
          for (int gi = 0; gi < ng; gi++, tile++) {
            const uint32_t s = tile & 1, ph = (tile >> 1) & 1;
            mbar_wait(&empty[s], ph ^ 1);
            mbar_expect_tx(&full[s], kTile);
            // rows past the sentence (the next sentence's, or zero fill past the tensor) are masked by the consumers
            for (int kb = 0; kb < 2; kb++)
              for (int slot = 0; slot < 4; slot++)
                tma_load_2d(s_ring + s * kTile + kb * 16384 + slot * 4096, map, &full[s], kb * 128,
                            b * a.T + gi * kGKeys + slot * kKeys);
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer
    if (elect_one()) {
      constexpr uint32_t idesc_k = make_idesc_i8(128, 256);     // A = u8 key rows, B = s8 Wk
      constexpr uint32_t idesc_v = make_idesc_i8_wa(128, 128);  // A = s8 Wv block, B = u8 key rows
      mbar_wait(w_full, 0);
      uint32_t tile = 0, ck = 0, cv = 0;
      for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        const int ng = groups_of(length_of(b));
        for (int gi = 0; gi < ng; gi++, tile++, ck++) {
          const uint32_t s = tile & 1, ph = (tile >> 1) & 1;
          mbar_wait(&full[s], ph);
          mbar_wait(k_drained, (ck & 1) ^ 1);
          tc_fence_after();
          for (int kb = 0; kb < 2; kb++) {
            const uint64_t da = make_kmajor_sw128_desc(smem_u32(s_ring + s * kTile + kb * 16384));
            const uint64_t db = make_kmajor_sw128_desc(smem_u32(s_wk + kb * 32768));
#pragma unroll
            for (int k = 0; k < 4; k++) umma_i8(tmem_k, da + 2 * k, db + 2 * k, idesc_k, (kb | k) ? 1u : 0u);
          }
          umma_commit(k_done);
          umma_commit(&empty[s]);
        }
        for (int gi = 0; gi < ng; gi++, tile++, cv++) {
          const uint32_t s = tile & 1, ph = (tile >> 1) & 1;
          mbar_wait(&full[s], ph);
          mbar_wait(v_drained, (cv & 1) ^ 1);
          tc_fence_after();
          for (int mb = 0; mb < 2; mb++)
            for (int kb = 0; kb < 2; kb++) {
              const uint64_t da = make_kmajor_sw128_desc(smem_u32(s_wv + kb * 32768 + mb * 16384));
              const uint64_t db = make_kmajor_sw128_desc(smem_u32(s_ring + s * kTile + kb * 16384));
#pragma unroll
              for (int k = 0; k < 4; k++) umma_i8(tmem_v + mb * 128, da + 2 * k, db + 2 * k, idesc_v, (kb | k) ? 1u : 0u);
            }
          umma_commit(v_done);
          umma_commit(&empty[s]);
        }
      }
    }
  } else if (warp >= 4) {
    // ===== consumers
    const int cw = warp - 4;
    const int qd = warp & 3;  // TMEM lane quadrant of this warp: key block of a K group, feature block of a V group
    const int sub = cw >> 2;  // K phase: head pair; V phase: sub < 2 owns the features of block sub
    const int ct = threadIdx.x - 128;
    const uint32_t lane_sel = static_cast<uint32_t>(qd * 32) << 16;
    const int h0 = sub * 2;
    const bool v_active = sub < 2;
    const int v_mb = sub & 1;
    const int v_feat = v_mb * 128 + qd * 32 + lane;
    const int v_head = v_mb * 4 + qd;
    const float pbv = a.pb_v[v_feat];
    const uint32_t sq_u32 = smem_u32(s_q_all);
    // the next sentence's query row travels global -> shared with cp.async while this one is processed
    auto fetch_q = [&](int b, uint32_t buf) {
      if (ct < kE) cp_async4(sq_u32 + (buf * kE + ct) * 4, a.q + static_cast<size_t>(b < a.B ? b : 0) * kE + ct, b < a.B);
      cp_async_commit();
    };
    fetch_q(blockIdx.x, 0);
    int len_nx = static_cast<int>(blockIdx.x) < a.B ? static_cast<int>(__ldg(a.lengths + blockIdx.x)) : 1;  // raw, clamped at use
    uint32_t it = 0, ck = 0, cv = 0;
    for (int b = blockIdx.x; b < a.B; b += gridDim.x, it++) {
      const float* s_q = s_q_all + (it & 1) * kE;
      const int len = max(1, min(len_nx, a.T));
      const int ng = groups_of(len);
      cp_async_wait_all();
      {
        const int bn = b + static_cast<int>(gridDim.x);
        fetch_q(bn, (it & 1) ^ 1);
        len_nx = bn < a.B ? static_cast<int>(__ldg(a.lengths + bn)) : 1;
      }
      named_bar_sync(1, kConsThreads);  // q row visible; the previous sentence's probabilities are no longer read

      // ---- K groups: lane = key, two heads per warp; scores stay in registers
      float sc[kMaxGroups][2];
      bool valid[kMaxGroups];
#pragma unroll
      for (int gi = 0; gi < kMaxGroups; gi++) {
        sc[gi][0] = sc[gi][1] = 0.0f;
        valid[gi] = false;
        if (gi < ng) {
          mbar_wait(k_done, ck & 1);
          ck++;
          tc_fence_after();
          uint32_t v0[32], v1[32];
          tmem_ld32_nowait(tmem_k + lane_sel + h0 * 32, v0);
          tmem_ld32_nowait(tmem_k + lane_sel + h0 * 32 + 32, v1);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(k_drained);
          // the two heads' fma chains advance together (source order is what the in-order issue sees)
          const float* qh = s_q + h0 * kDH;
          const float* pbh = s_pbk + h0 * kDH;
          float acc0 = 0.0f, acc1 = 0.0f;
#pragma unroll
          for (int d = 0; d < kDH; d += 4) {
            const float4 q0 = *reinterpret_cast<const float4*>(qh + d);
            const float4 q1 = *reinterpret_cast<const float4*>(qh + kDH + d);
            const float4 p0 = *reinterpret_cast<const float4*>(pbh + d);
            const float4 p1 = *reinterpret_cast<const float4*>(pbh + kDH + d);
            acc0 = fmaf(q0.x, dequant1(static_cast<int>(v0[d]), a.um_k, p0.x), acc0);
            acc1 = fmaf(q1.x, dequant1(static_cast<int>(v1[d]), a.um_k, p1.x), acc1);
            acc0 = fmaf(q0.y, dequant1(static_cast<int>(v0[d + 1]), a.um_k, p0.y), acc0);
            acc1 = fmaf(q1.y, dequant1(static_cast<int>(v1[d + 1]), a.um_k, p1.y), acc1);
            acc0 = fmaf(q0.z, dequant1(static_cast<int>(v0[d + 2]), a.um_k, p0.z), acc0);
            acc1 = fmaf(q1.z, dequant1(static_cast<int>(v1[d + 2]), a.um_k, p1.z), acc1);
            acc0 = fmaf(q0.w, dequant1(static_cast<int>(v0[d + 3]), a.um_k, p0.w), acc0);
            acc1 = fmaf(q1.w, dequant1(static_cast<int>(v1[d + 3]), a.um_k, p1.w), acc1);
          }
          sc[gi][0] = __fmul_rn(a.dk, acc0);
          sc[gi][1] = __fmul_rn(a.dk, acc1);
          valid[gi] = gi * kGKeys + qd * kKeys + lane < len;
        }
      }

      // ---- softmax of the two heads over all the sentence's keys (slimt/TensorOps.cc:282-315): max, exp, sum in key
      // order, divide.  The four warps of a head pair (one per key block) meet at named barrier 2 + sub.
      float mx[2], e[kMaxGroups][2];
#pragma unroll
      for (int hh = 0; hh < 2; hh++) {
        mx[hh] = -3.402823466e+38f;
#pragma unroll
        for (int gi = 0; gi < kMaxGroups; gi++)
          if (valid[gi]) mx[hh] = fmaxf(mx[hh], sc[gi][hh]);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int hh = 0; hh < 2; hh++) mx[hh] = fmaxf(mx[hh], __shfl_xor_sync(0xffffffffu, mx[hh], o));
      }
      if (lane < 2) s_pmax[qd * kH + h0 + lane] = mx[lane];
      named_bar_sync(2 + sub, 4 * 32);
#pragma unroll
      for (int hh = 0; hh < 2; hh++)
#pragma unroll
        for (int o = 0; o < 4; o++) mx[hh] = fmaxf(mx[hh], s_pmax[o * kH + h0 + hh]);
#pragma unroll
      for (int gi = 0; gi < kMaxGroups; gi++) {
        if (gi < ng) {
#pragma unroll
          for (int hh = 0; hh < 2; hh++) e[gi][hh] = expf_glibc_nonpos_tab(__fsub_rn(sc[gi][hh], mx[hh]), exp_tab);
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            e[gi][hh] = valid[gi] ? e[gi][hh] : 0.0f;
            s_p[(h0 + hh) * kMaxS + gi * kGKeys + qd * kKeys + lane] = e[gi][hh];
          }
        } else {
          e[gi][0] = e[gi][1] = 0.0f;
        }
      }
      named_bar_sync(2 + sub, 4 * 32);
      if (qd < 2) {  // this warp forms the row sum of head h0 + qd: one chain over the keys in order
        const float* prow = s_p + (h0 + qd) * kMaxS;
        const int n = (len + 3) & ~3;  // the parked exponentials past the length are exactly 0 (x + 0 = x)
        float sum = 0.0f;
#pragma unroll 4
        for (int l = 0; l < n; l += 4) {
          const float4 t = *reinterpret_cast<const float4*>(prow + l);
          sum = __fadd_rn(sum, t.x);
          sum = __fadd_rn(sum, t.y);
          sum = __fadd_rn(sum, t.z);
          sum = __fadd_rn(sum, t.w);
        }
        if (lane == 0) s_psum[h0 + qd] = sum;
      }
      named_bar_sync(2 + sub, 4 * 32);
#pragma unroll
      for (int gi = 0; gi < kMaxGroups; gi++) {
        if (gi < ng) {
          const int key = gi * kGKeys + qd * kKeys + lane;
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            const float p = valid[gi] ? __fdiv_rn(e[gi][hh], s_psum[h0 + hh]) : 0.0f;
            s_p[(h0 + hh) * kMaxS + key] = p;
            if (a.attn_head0 != nullptr && h0 + hh == 0 && key < a.T) a.attn_head0[static_cast<size_t>(b) * a.T + key] = p;
          }
        } else if (a.attn_head0 != nullptr && h0 == 0) {  // padded keys of a group this sentence never reaches
          const int key = gi * kGKeys + qd * kKeys + lane;
          if (key < a.T) a.attn_head0[static_cast<size_t>(b) * a.T + key] = 0.0f;
        }
      }
      named_bar_sync(1, kConsThreads);

      // ---- V groups: lane = output feature, one chain over the sentence's keys in order
      if (v_active) {
        float acc = 0.0f;
        for (int gi = 0; gi < ng; gi++, cv++) {
          mbar_wait(v_done, cv & 1);
          tc_fence_after();
#pragma unroll
          for (int half = 0; half < 2; half++) {
            uint32_t v0[32], v1[32];
            tmem_ld32_nowait(tmem_v + lane_sel + v_mb * 128 + half * 64, v0);
            tmem_ld32_nowait(tmem_v + lane_sel + v_mb * 128 + half * 64 + 32, v1);
            tmem_ld_wait();
            if (half == 1) {
              tc_fence_before();
              __syncwarp();
              if (lane == 0) mbar_arrive(v_drained);
            }
            const float* pr = s_p + v_head * kMaxS + gi * kGKeys + half * 64;
            // keys past the length have probability exactly 0 and leave the chain unchanged: whole 32-key blocks of them are
            // skipped (a finer test inside the unrolled chain costs more than the skipped FMAs)
            const int left = len - gi * kGKeys - half * 64;
            if (left > 0) {
#pragma unroll
              for (int l = 0; l < kKeys; l += 4) {
                const float4 p = *reinterpret_cast<const float4*>(pr + l);
                acc = fmaf(p.x, dequant1(static_cast<int>(v0[l]), a.um_v, pbv), acc);
                acc = fmaf(p.y, dequant1(static_cast<int>(v0[l + 1]), a.um_v, pbv), acc);
                acc = fmaf(p.z, dequant1(static_cast<int>(v0[l + 2]), a.um_v, pbv), acc);
                acc = fmaf(p.w, dequant1(static_cast<int>(v0[l + 3]), a.um_v, pbv), acc);
              }
            }
            if (left > kKeys) {
#pragma unroll
              for (int l = 0; l < kKeys; l += 4) {
                const float4 p = *reinterpret_cast<const float4*>(pr + kKeys + l);
                acc = fmaf(p.x, dequant1(static_cast<int>(v1[l]), a.um_v, pbv), acc);
                acc = fmaf(p.y, dequant1(static_cast<int>(v1[l + 1]), a.um_v, pbv), acc);
                acc = fmaf(p.z, dequant1(static_cast<int>(v1[l + 2]), a.um_v, pbv), acc);
                acc = fmaf(p.w, dequant1(static_cast<int>(v1[l + 3]), a.um_v, pbv), acc);
              }
            }
          }
        }
        const size_t off = static_cast<size_t>(b) * kE + v_feat;
        if (a.qo.n == 1) a.qo.ptr[0][off] = static_cast<int8_t>(quantize<false>(acc, a.qo.aq[0]));
        else
          for (int k = 0; k < a.qo.n; k++) a.qo.ptr[k][off] = static_cast<int8_t>(quantize<false>(acc, a.qo.aq[k]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

}  // namespace

bool cross_attention_rcl_supported(int E, int H, int dh, int S) {
  return E == kE && H == kH && dh == kDH && S >= 1 && S <= kMaxS;
}

int launch_cross_attention_rcl(const CrossRcArgs& a, int num_sms, cudaStream_t stream) {
  if (a.B == 0) return 0;
  auto kern = cross_attention_rcl_kernel;
  if (ensure_dyn_smem(kern, SmemL::total) != cudaSuccess) return 1;
  return launch_pdl(kern, dim3(a.B < num_sms ? a.B : num_sms), dim3(kThreadsL), SmemL::total, stream, a) != cudaSuccess;
}

}  // namespace sb
