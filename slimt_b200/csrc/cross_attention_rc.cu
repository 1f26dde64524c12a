// Decoder cross-attention that RECOMPUTES the key/value projections on the tensor cores every step instead of
// streaming an f32 K/V cache from HBM (reference: Attention::forward, slimt/Modules.cc:287-319 — which also
// re-projects K and V on every step, :244-249 — and scaled_dot_product_attention :24-86).
//
// Why: at tiny11 sizes the cached path reads 2 * S * E * 4 = 64 KB per sentence per layer per step and is pinned to
// the HBM roofline.  The projections' INPUT, the encoder output quantised for Wk and Wv (PrepareA bytes), is 4x
// smaller (2 * S * E bytes), the int8 MMAs that rebuild K = dequant(qa_k Wk) and V = dequant(qa_v Wv) are nearly
// free on tcgen05, and the f32 values they produce are the very ones the cache would have held: the int32
// accumulators are exact and the dequantisation is the same two roundings.
//
// Two kernels, one per range of source lengths, built from the shared stages below (set-up, resident weights, MMA
// issue, the exact score and weighted-sum chains, the quantised output, teardown): cross_attention_rc_kernel for
// S <= 64 walks groups of sentences, cross_attention_rcl_kernel for 65 .. 256 tokens walks one sentence at a time.
//
// cross_attention_rc_kernel: one persistent CTA per SM walks groups of 4 sentences (4 x 32 key rows = the 128 TMEM
// lanes); Wk and Wv (64 KB each) stay resident in shared memory for the whole launch.
//   K phase   D_k[key row][feature]   = qa_k tile (A, M = 128) x Wk (B, N = 256): TMEM lane = key, so a consumer
//             thread dequantises its key's 32 features of a head and runs the reference's sequential fma chain
//             against q; softmax across the 32 lanes of the warp (max by shuffle, sum in key order).
//   V phase   D_v[feature][key row]   = Wv (A, M = 128 per block) x qa_v tile (B, N = 128): TMEM lane = feature, so
//             a thread accumulates its output feature over the keys in order, probabilities broadcast from smem.
// The MMA of the next phase overlaps the drain of the current one (D_k and D_v are separate TMEM regions).
// Sentences longer than 32 tokens (template parameter KB = 2: up to 64) take two 32-key blocks of the group's 128 lanes,
// so a group holds 4 / KB sentences: the softmax maximum and the key-ordered sum then span the KB warps that hold a
// sentence's blocks (partial maxima and the exponentials meet in shared memory under a barrier of just those warps),
// and a V-phase thread runs ONE chain over the sentence's 32 * KB keys instead of two sentences' chains.
// Supported: E = 256, 8 heads of 32, S <= 64 (S <= 256 for the sentence-at-a-time kernel).  Everything else uses the
// cached kernel (cross_attention.cu).
#include <stdio.h>

#include "exact_math.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kE = 256, kH = 8, kDH = 32;
constexpr int kKeys = 32;                  // key rows per TMA box, and per TMEM lane quadrant
constexpr int kConsWarps = 16;
constexpr int kConsThreads = kConsWarps * 32;
constexpr int kThreads = 128 + kConsThreads;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 tables, 4..19 consumers
constexpr int kTile = 32 * 1024;           // one operand tile: 2 k-blocks x [128 key rows x 128 B]

// Both kernels' shared memory begins with the resident weights; the rest of each layout is its own.
struct SmemHead {
  static constexpr int wk = 0;                        // 2 k-blocks x [256 features x 128 B]
  static constexpr int wv = wk + 64 * 1024;
  static constexpr int tiles = wv + 64 * 1024;        // 2 operand tiles
};

// Everything before the first TMA or MMA: tensor-map prefetch, the 9 barriers (bars[0..6] single-arrival, k_drained =
// bars[7] counts every consumer warp, v_drained = bars[8] the v_drainers warps that drain D_v), 512 TMEM columns, the
// exp table and Wk's prepared bias in shared memory, then the PDL hand-over.  Returns the TMEM base.
__device__ __forceinline__ uint32_t rc_prologue(const CrossRcArgs& a, uint64_t* bars, uint32_t* tmem_slot,
                                                uint64_t* exp_tab, float* s_pbk, int warp, int lane, int v_drainers) {
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.map_ak);
    tma_prefetch_desc(&a.map_av);
    tma_prefetch_desc(&a.map_wk);
    tma_prefetch_desc(&a.map_wv);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 7; i++) mbar_init(&bars[i], 1);
    mbar_init(bars + 7, kConsWarps);
    mbar_init(bars + 8, v_drainers);
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
  return *tmem_slot;
}

// Wk and Wv (64 KB each), loaded once per launch
__device__ __forceinline__ void load_weights(const CrossRcArgs& a, uint8_t* s_wk, uint8_t* s_wv, uint64_t* w_full) {
  mbar_expect_tx(w_full, 128 * 1024);
  for (int kb = 0; kb < 2; kb++)
    for (int half = 0; half < 2; half++) {
      tma_load_2d(s_wk + kb * 32768 + half * 16384, &a.map_wk, w_full, kb * 128, half * 128);
      tma_load_2d(s_wv + kb * 32768 + half * 16384, &a.map_wv, w_full, kb * 128, half * 128);
    }
}

// D_k[key row][feature] = a_tile (u8 key rows, M = 128) x Wk (s8, N = 256)
__device__ __forceinline__ void mma_k(uint32_t tmem_k, const uint8_t* a_tile, const uint8_t* s_wk) {
  constexpr uint32_t idesc_k = make_idesc_i8(128, 256);  // A = u8 key rows, B = s8 Wk
  for (int kb = 0; kb < 2; kb++) {
    const uint64_t da = make_kmajor_sw128_desc(smem_u32(a_tile + kb * 16384));
    const uint64_t db = make_kmajor_sw128_desc(smem_u32(s_wk + kb * 32768));
#pragma unroll
    for (int k = 0; k < 4; k++) umma_i8(tmem_k, da + 2 * k, db + 2 * k, idesc_k, (kb | k) ? 1u : 0u);
  }
}

// D_v[feature][key row] = Wv (s8, 2 blocks of M = 128 features) x b_tile (u8 key rows, N = 128)
__device__ __forceinline__ void mma_v(uint32_t tmem_v, const uint8_t* s_wv, const uint8_t* b_tile) {
  constexpr uint32_t idesc_v = make_idesc_i8_wa(128, 128);  // A = s8 Wv block, B = u8 key rows
  for (int mb = 0; mb < 2; mb++)
    for (int kb = 0; kb < 2; kb++) {
      const uint64_t da = make_kmajor_sw128_desc(smem_u32(s_wv + kb * 32768 + mb * 16384));
      const uint64_t db = make_kmajor_sw128_desc(smem_u32(b_tile + kb * 16384));
#pragma unroll
      for (int k = 0; k < 4; k++) umma_i8(tmem_v + mb * 128, da + 2 * k, db + 2 * k, idesc_v, (kb | k) ? 1u : 0u);
    }
}

// The scores of one key for heads h0 and h0 + 1 (qh: the query from head h0 on; v0, v1: the key's int32 accumulators of
// the two heads): the reference's sequential fma chain of q against the dequantised K, scaled by dk.  The two heads'
// chains advance together (source order is what the in-order issue sees).
__device__ __forceinline__ void exact_scores2(float (&sc)[2], const float* qh, const float* s_pbk, int h0,
                                              const uint32_t (&v0)[32], const uint32_t (&v1)[32], float um_k,
                                              float dk) {
  const float* pbh = s_pbk + h0 * kDH;
  float acc0 = 0.0f, acc1 = 0.0f;
#pragma unroll
  for (int d = 0; d < kDH; d += 4) {
    const float4 q0 = *reinterpret_cast<const float4*>(qh + d);
    const float4 q1 = *reinterpret_cast<const float4*>(qh + kDH + d);
    const float4 p0 = *reinterpret_cast<const float4*>(pbh + d);
    const float4 p1 = *reinterpret_cast<const float4*>(pbh + kDH + d);
    acc0 = fmaf(q0.x, dequant1(static_cast<int>(v0[d]), um_k, p0.x), acc0);
    acc1 = fmaf(q1.x, dequant1(static_cast<int>(v1[d]), um_k, p1.x), acc1);
    acc0 = fmaf(q0.y, dequant1(static_cast<int>(v0[d + 1]), um_k, p0.y), acc0);
    acc1 = fmaf(q1.y, dequant1(static_cast<int>(v1[d + 1]), um_k, p1.y), acc1);
    acc0 = fmaf(q0.z, dequant1(static_cast<int>(v0[d + 2]), um_k, p0.z), acc0);
    acc1 = fmaf(q1.z, dequant1(static_cast<int>(v1[d + 2]), um_k, p1.z), acc1);
    acc0 = fmaf(q0.w, dequant1(static_cast<int>(v0[d + 3]), um_k, p0.w), acc0);
    acc1 = fmaf(q1.w, dequant1(static_cast<int>(v1[d + 3]), um_k, p1.w), acc1);
  }
  sc[0] = __fmul_rn(dk, acc0);
  sc[1] = __fmul_rn(dk, acc1);
}

// The weighted sum of one output feature carried over 32 more keys in order: acc += p[key] * dequant(v[key]).
__device__ __forceinline__ float v_chain32(float acc, const float* pr, const uint32_t (&v)[32], float um_v, float pbv) {
#pragma unroll
  for (int l = 0; l < kKeys; l += 4) {
    const float4 p = *reinterpret_cast<const float4*>(pr + l);
    acc = fmaf(p.x, dequant1(static_cast<int>(v[l]), um_v, pbv), acc);
    acc = fmaf(p.y, dequant1(static_cast<int>(v[l + 1]), um_v, pbv), acc);
    acc = fmaf(p.z, dequant1(static_cast<int>(v[l + 2]), um_v, pbv), acc);
    acc = fmaf(p.w, dequant1(static_cast<int>(v[l + 3]), um_v, pbv), acc);
  }
  return acc;
}

// Output feature `feat` of sentence b, quantised for each consumer.  The usual case is one consumer (Wo): constant
// indices keep its multiplier and pointer in the constant bank.
template <bool kFast>
__device__ __forceinline__ void emit(const CrossRcArgs& a, int b, int feat, float acc) {
  const size_t off = static_cast<size_t>(b) * kE + feat;
  if (a.qo.n == 1) a.qo.ptr[0][off] = static_cast<int8_t>(quantize<kFast>(acc, a.qo.aq[0]));
  else
    for (int k = 0; k < a.qo.n; k++) a.qo.ptr[k][off] = static_cast<int8_t>(quantize<kFast>(acc, a.qo.aq[k]));
}

// Every role is done with TMEM before the warp that allocated it frees it.
__device__ __forceinline__ void rc_teardown(uint32_t tmem, int warp) {
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// ================================================ groups of sentences, S <= 64

constexpr int kGroup = 4;                  // sentences per group

struct Smem : SmemHead {
  static constexpr int ak = tiles;
  static constexpr int av = ak + kTile;
  static constexpr int qs = av + kTile;           // f32 [2 buffers][4][256]: the group's query rows, filled by cp.async
  static constexpr int lens = qs + 2 * kGroup * kE * 4;  // i32 [2 buffers][4]: the group's sentence lengths
  static constexpr int ps = lens + 2 * kGroup * 4;    // f32 [4][8][32]
  static constexpr int pbk = ps + kGroup * kH * kKeys * 4;  // f32 [256]
  static constexpr int pmax = pbk + kE * 4;           // f32 [4 key blocks][8 heads]: per-block score maxima (KB > 1)
  static constexpr int psum = pmax + kGroup * kH * 4;     // f32 [4 key blocks][8 heads]: per-block sums (tolerance mode, KB > 1)
  static constexpr int exp_tab = psum + kGroup * kH * 4;  // u64 [32]
  static constexpr int bars = exp_tab + 32 * 8;
  // w_full ak_full av_full ak_free av_free k_done v_done k_drained v_drained
  static constexpr int n_bars = 9;
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
};

// kFast (tolerance mode): the dequantisation is folded out of the inner loops.  K = um_k * acc_k + pb_k, so
// q . K[key] = um_k * sum_d q[d] * acc_k[key][d] + q . pb_k, and the second term is the same for every key of a (sentence,
// head): it cancels in the softmax and is never formed.  V = um_v * acc_v + pb_v and the probabilities sum to one, so
// sum_key p[key] * V[key][f] = um_v * sum_key p[key] * acc_v[f][key] + pb_v[f].  Per element that leaves one int -> float
// conversion and one FMA; the softmax uses ex2 / rcp and shuffle-tree sums.
template <int KB, bool kFast>  // 32-key blocks per sentence (1: S <= 32, 2: S <= 64)
__global__ void __launch_bounds__(kThreads, 1) cross_attention_rc_kernel(const __grid_constant__ CrossRcArgs a) {
  constexpr int NS = kGroup / KB;  // sentences per group
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* s_wk = smem + Smem::wk;
  uint8_t* s_wv = smem + Smem::wv;
  uint8_t* s_ak = smem + Smem::ak;
  uint8_t* s_av = smem + Smem::av;
  float* s_q_all = reinterpret_cast<float*>(smem + Smem::qs);
  int* s_len_all = reinterpret_cast<int*>(smem + Smem::lens);
  float* s_p = reinterpret_cast<float*>(smem + Smem::ps);
  float* s_pbk = reinterpret_cast<float*>(smem + Smem::pbk);
  float* s_pmax = reinterpret_cast<float*>(smem + Smem::pmax);
  float* s_psum = reinterpret_cast<float*>(smem + Smem::psum);
  uint64_t* exp_tab = reinterpret_cast<uint64_t*>(smem + Smem::exp_tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Smem::bars);
  uint64_t* w_full = bars;
  uint64_t* ak_full = bars + 1;
  uint64_t* av_full = bars + 2;
  uint64_t* ak_free = bars + 3;
  uint64_t* av_free = bars + 4;
  uint64_t* k_done = bars + 5;
  uint64_t* v_done = bars + 6;
  uint64_t* k_drained = bars + 7;
  uint64_t* v_drained = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Smem::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem = rc_prologue(a, bars, tmem_slot, exp_tab, s_pbk, warp, lane, kConsWarps);
  const uint32_t tmem_k = tmem;         // 256 columns: features
  const uint32_t tmem_v = tmem + 256;   // 2 blocks x 128 columns: key rows of the group

  const int n_groups = (a.B + NS - 1) / NS;

  if (warp == 0) {
    // ===== TMA producer
    if (elect_one()) {
      load_weights(a, s_wk, s_wv, w_full);
      uint32_t it = 0;
      for (int g = blockIdx.x; g < n_groups; g += gridDim.x, it++) {
        const uint32_t ph = it & 1;
        const int b0 = g * NS;
        // slot = 32 key rows: sentence slot / KB, its key block slot % KB (rows past the sentence's length -- the next
        // sentence's, or zero fill past the tensor -- are masked by the consumers)
        mbar_wait(ak_free, ph ^ 1);
        mbar_expect_tx(ak_full, kTile);
        for (int kb = 0; kb < 2; kb++)
          for (int slot = 0; slot < kGroup; slot++) {
            const int j = slot / KB;
            const int b = b0 + j < a.B ? b0 + j : b0;  // tail group: repeat a valid sentence, its lanes are ignored
            tma_load_2d(s_ak + kb * 16384 + slot * 4096, &a.map_ak, ak_full, kb * 128, b * a.T + (slot % KB) * kKeys);
          }
        mbar_wait(av_free, ph ^ 1);
        mbar_expect_tx(av_full, kTile);
        for (int kb = 0; kb < 2; kb++)
          for (int slot = 0; slot < kGroup; slot++) {
            const int j = slot / KB;
            const int b = b0 + j < a.B ? b0 + j : b0;
            tma_load_2d(s_av + kb * 16384 + slot * 4096, &a.map_av, av_full, kb * 128, b * a.T + (slot % KB) * kKeys);
          }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer
    if (elect_one()) {
      mbar_wait(w_full, 0);
      uint32_t it = 0;
      for (int g = blockIdx.x; g < n_groups; g += gridDim.x, it++) {
        const uint32_t ph = it & 1;
        mbar_wait(ak_full, ph);
        mbar_wait(k_drained, ph ^ 1);
        tc_fence_after();
        mma_k(tmem_k, s_ak, s_wk);
        umma_commit(k_done);
        umma_commit(ak_free);
        mbar_wait(av_full, ph);
        mbar_wait(v_drained, ph ^ 1);
        tc_fence_after();
        mma_v(tmem_v, s_wv, s_av);
        umma_commit(v_done);
        umma_commit(av_free);
      }
    }
  } else if (warp >= 4) {
    // ===== consumers
    const int cw = warp - 4;
    const int qd = warp & 3;   // TMEM lane quadrant of this warp
    const int sub = cw >> 2;   // 0..3: which share of the quadrant's work
    const int ct = threadIdx.x - 128;
    const uint32_t lane_sel = static_cast<uint32_t>(qd * 32) << 16;
    // V phase: this thread's output feature
    const int v_mb = sub & 1;
    const int v_feat = v_mb * 128 + qd * 32 + lane;
    const int v_head = v_mb * 4 + qd;
    const float pbv = a.pb_v[v_feat];
    // Global inputs of a group (its query rows and sentence lengths) are fetched one group ahead with cp.async straight
    // into the other half of a double-buffered shared block: their latency hides behind the previous group's arithmetic
    // and they occupy no registers meanwhile (held in registers they pushed the kernel over its 96-register budget: the
    // compiler then spilled the freshly loaded values, i.e. waited for the loads it had just issued).
    constexpr int kQPer = NS * kE / kConsThreads;  // query floats per consumer thread: 2 (KB = 1) or 1 (KB = 2)
    static_assert(NS * kE == kQPer * kConsThreads, "query floats per consumer thread");
    const int kj = qd / KB;             // K phase: this warp's sentence of the group ...
    const int kblk = qd % KB;           // ... and which of its key blocks sits in the warp's lane quadrant
    const int key = kblk * kKeys + lane;
    const int vj0 = KB == 1 ? (sub >> 1) * 2 : (sub >> 1);  // V phase: first (KB = 1: of two) sentence of this warp
    // A group's NS query rows are contiguous: float i of the group is a.q[g * NS * kE + i], valid while below B * kE.
    const int q_end = a.B * kE;
    const uint32_t sq_u32 = smem_u32(s_q_all), slen_u32 = smem_u32(s_len_all);
    auto fetch_group = [&](int g, uint32_t buf) {
      const int q0 = g * (NS * kE) + ct;
#pragma unroll
      for (int r = 0; r < kQPer; r++) {
        const int i = q0 + r * kConsThreads;
        cp_async4(sq_u32 + (buf * kGroup * kE + ct + r * kConsThreads) * 4, a.q + (i < q_end ? i : 0), i < q_end);
      }
      if (ct < NS) {
        const int b = g * NS + ct;
        cp_async4(slen_u32 + (buf * kGroup + ct) * 4, a.lengths + (b < a.B ? b : 0), b < a.B);
      }
      cp_async_commit();
    };
    fetch_group(blockIdx.x, 0);
    // Accumulators travel TMEM -> registers one phase ahead of their use: the V accumulators are requested as soon as the
    // scores are formed (the K registers are dead then) and arrive during the softmax; the next group's K accumulators are
    // requested at the end of the V phase and arrive during the loop head.  tmem_ld_wait_dep() is the only point after
    // which the registers may be read.
    uint32_t v0[32], v1[32];
    const int h0 = sub * 2;
    const int c0 = (sub >> 1) * 64;  // V phase: the warp's 64 key columns of the group
    auto request_k = [&](uint32_t ph) {
      mbar_wait(k_done, ph);
      tc_fence_after();
      tmem_ld32_nowait(tmem_k + lane_sel + h0 * 32, v0);
      tmem_ld32_nowait(tmem_k + lane_sel + h0 * 32 + 32, v1);
    };
    auto request_v = [&](uint32_t ph) {
      mbar_wait(v_done, ph);
      tc_fence_after();
      tmem_ld32_nowait(tmem_v + lane_sel + v_mb * 128 + c0, v0);
      tmem_ld32_nowait(tmem_v + lane_sel + v_mb * 128 + c0 + 32, v1);
    };
    if (static_cast<int>(blockIdx.x) < n_groups) request_k(0);
    uint32_t it = 0;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x, it++) {
      const uint32_t ph = it & 1;
      const int b0 = g * NS;
      // this group's rows and lengths were requested a group ago; the other buffer is free (its readers, the previous
      // group's K and V phases, are behind this warp) and takes the next group's
      const float* s_q = s_q_all + (it & 1) * kGroup * kE;
      const int* s_len = s_len_all + (it & 1) * kGroup;
      cp_async_wait_all();
      fetch_group(g + gridDim.x, (it & 1) ^ 1);
      named_bar_sync(1, kConsThreads);

      // ---- K phase: quadrant = 32 keys of a sentence, lane = key, two heads per warp
      {
        const int j = kj;
        const int b = b0 + j;
        const int len_k = min(s_len[kj], a.T);
        const bool valid = key < len_k;
        tmem_ld_wait_dep(v0, v1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(k_drained);
        constexpr int kRow = KB * kKeys;  // probabilities of one (sentence, head)
        float* prow = s_p + (j * kH + h0) * kRow;
        if constexpr (kFast) {
          // scores in the log2 domain, up to a per-(sentence, head) constant (see the kernel comment)
          float sc[2];
          {
            const float* qh = s_q + j * kE + h0 * kDH;
            float acc0 = 0.0f, acc1 = 0.0f;
#pragma unroll
            for (int d = 0; d < kDH; d += 4) {
              const float4 q0 = *reinterpret_cast<const float4*>(qh + d);
              const float4 q1 = *reinterpret_cast<const float4*>(qh + kDH + d);
              acc0 = fmaf(q0.x, __int2float_rn(static_cast<int>(v0[d])), acc0);
              acc1 = fmaf(q1.x, __int2float_rn(static_cast<int>(v1[d])), acc1);
              acc0 = fmaf(q0.y, __int2float_rn(static_cast<int>(v0[d + 1])), acc0);
              acc1 = fmaf(q1.y, __int2float_rn(static_cast<int>(v1[d + 1])), acc1);
              acc0 = fmaf(q0.z, __int2float_rn(static_cast<int>(v0[d + 2])), acc0);
              acc1 = fmaf(q1.z, __int2float_rn(static_cast<int>(v1[d + 2])), acc1);
              acc0 = fmaf(q0.w, __int2float_rn(static_cast<int>(v0[d + 3])), acc0);
              acc1 = fmaf(q1.w, __int2float_rn(static_cast<int>(v1[d + 3])), acc1);
            }
            const float sk = a.dk * a.um_k * 1.4426950408889634f;
            sc[0] = valid ? acc0 * sk : -3.402823466e+38f;
            sc[1] = valid ? acc1 * sk : -3.402823466e+38f;
          }
          request_v(ph);
          float mx[2] = {sc[0], sc[1]};
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int hh = 0; hh < 2; hh++) mx[hh] = fmaxf(mx[hh], __shfl_xor_sync(0xffffffffu, mx[hh], o));
          }
          if constexpr (KB > 1) {
            if (lane < 2) s_pmax[qd * kH + h0 + lane] = mx[lane];
            named_bar_sync(2 + kj * 4 + sub, KB * 32);
#pragma unroll
            for (int hh = 0; hh < 2; hh++)
#pragma unroll
              for (int o = 0; o < KB; o++) mx[hh] = fmaxf(mx[hh], s_pmax[(kj * KB + o) * kH + h0 + hh]);
          }
          float e[2], sum[2];
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            e[hh] = valid ? exp2_fast(sc[hh] - mx[hh]) : 0.0f;
            sum[hh] = warp_sum(e[hh]);
          }
          if constexpr (KB > 1) {
            if (lane < 2) s_psum[qd * kH + h0 + lane] = sum[lane];
            named_bar_sync(2 + kj * 4 + sub, KB * 32);
#pragma unroll
            for (int hh = 0; hh < 2; hh++) {
              float t = 0.0f;
#pragma unroll
              for (int o = 0; o < KB; o++) t += s_psum[(kj * KB + o) * kH + h0 + hh];
              sum[hh] = t;
            }
          }
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            const float p = e[hh] * rcp_fast(sum[hh]);
            prow[hh * kRow + key] = p;
            if (a.attn_head0 != nullptr && h0 + hh == 0 && b < a.B && key < a.T)
              a.attn_head0[static_cast<size_t>(b) * a.T + key] = p;
          }
        } else {
        float sc[2];
        exact_scores2(sc, s_q + j * kE + h0 * kDH, s_pbk, h0, v0, v1, a.um_k, a.dk);
        request_v(ph);
        // softmax over the sentence's keys (slimt/TensorOps.cc:282-315): max, exp, sum in key order, divide.  Both
        // heads advance together: nothing is stored between the two expf evaluations (a store would pin the second
        // one's table load behind it), so their double-precision chains interleave.
        float mx[2], e[2], sum[2];
#pragma unroll
        for (int hh = 0; hh < 2; hh++) mx[hh] = valid ? sc[hh] : -3.402823466e+38f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
          for (int hh = 0; hh < 2; hh++) mx[hh] = fmaxf(mx[hh], __shfl_xor_sync(0xffffffffu, mx[hh], o));
        }
        if constexpr (KB > 1) {
          // the sentence's other key block lives in the neighbouring quadrant's warp with the same head pair: the two
          // block maxima meet in shared memory (the maximum of a set does not depend on the order it is formed in)
          if (lane < 2) s_pmax[qd * kH + h0 + lane] = mx[lane];
          named_bar_sync(2 + kj * 4 + sub, KB * 32);
#pragma unroll
          for (int hh = 0; hh < 2; hh++)
#pragma unroll
            for (int o = 0; o < KB; o++) mx[hh] = fmaxf(mx[hh], s_pmax[(kj * KB + o) * kH + h0 + hh]);
        }
#pragma unroll
        for (int hh = 0; hh < 2; hh++) e[hh] = expf_glibc_nonpos_tab(__fsub_rn(sc[hh], mx[hh]), exp_tab);
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
          e[hh] = valid ? e[hh] : 0.0f;
          prow[hh * kRow + key] = e[hh];
          sum[hh] = 0.0f;
        }
        if constexpr (KB > 1) named_bar_sync(2 + kj * 4 + sub, KB * 32);
        else __syncwarp();
        if constexpr (KB == 1) {
          // one chain per head is enough: the lower half-warp forms head h0's sum, the upper half head h0 + 1's
          const float* pr = prow + (lane >> 4) * kRow;
          float s = 0.0f;
#pragma unroll
          for (int l = 0; l < kRow; l += 4) {
            const float4 t = *reinterpret_cast<const float4*>(pr + l);
            s = __fadd_rn(s, t.x);
            s = __fadd_rn(s, t.y);
            s = __fadd_rn(s, t.z);
            s = __fadd_rn(s, t.w);
          }
          sum[0] = __shfl_sync(0xffffffffu, s, 0);
          sum[1] = __shfl_sync(0xffffffffu, s, 16);
        } else {
#pragma unroll
        for (int l = 0; l < kRow; l += 4) {
#pragma unroll
          for (int hh = 0; hh < 2; hh++) {
            const float4 t = *reinterpret_cast<const float4*>(prow + hh * kRow + l);
            sum[hh] = __fadd_rn(sum[hh], t.x);
            sum[hh] = __fadd_rn(sum[hh], t.y);
            sum[hh] = __fadd_rn(sum[hh], t.z);
            sum[hh] = __fadd_rn(sum[hh], t.w);
          }
        }
        }
        if constexpr (KB > 1) named_bar_sync(2 + kj * 4 + sub, KB * 32);  // every warp of the sentence has read the e's
        else __syncwarp();
#pragma unroll
        for (int hh = 0; hh < 2; hh++) {
          const float p = valid ? __fdiv_rn(e[hh], sum[hh]) : 0.0f;
          prow[hh * kRow + key] = p;
          if (a.attn_head0 != nullptr && h0 + hh == 0 && b < a.B && key < a.T)
            a.attn_head0[static_cast<size_t>(b) * a.T + key] = p;
        }
        }  // exact K phase
      }
      named_bar_sync(1, kConsThreads);

      // ---- V phase: lane = output feature; KB = 1: two sentences per warp, KB = 2: one sentence of up to 64 keys
      {
        tmem_ld_wait_dep(v0, v1);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(v_drained);
        constexpr int kRow = KB * kKeys;
        if constexpr (kFast) {
          // probabilities of keys past a sentence's length are exactly 0, so every chain runs over the whole block
          if constexpr (KB == 1) {
            const int j0 = vj0;
            const float* pr0 = s_p + (j0 * kH + v_head) * kKeys;
            const float* pr1 = pr0 + kH * kKeys;
            float acc0 = 0.0f, acc1 = 0.0f;
#pragma unroll
            for (int l = 0; l < kKeys; l += 4) {
              const float4 p0 = *reinterpret_cast<const float4*>(pr0 + l);
              const float4 p1 = *reinterpret_cast<const float4*>(pr1 + l);
              acc0 = fmaf(p0.x, __int2float_rn(static_cast<int>(v0[l])), acc0);
              acc1 = fmaf(p1.x, __int2float_rn(static_cast<int>(v1[l])), acc1);
              acc0 = fmaf(p0.y, __int2float_rn(static_cast<int>(v0[l + 1])), acc0);
              acc1 = fmaf(p1.y, __int2float_rn(static_cast<int>(v1[l + 1])), acc1);
              acc0 = fmaf(p0.z, __int2float_rn(static_cast<int>(v0[l + 2])), acc0);
              acc1 = fmaf(p1.z, __int2float_rn(static_cast<int>(v1[l + 2])), acc1);
              acc0 = fmaf(p0.w, __int2float_rn(static_cast<int>(v0[l + 3])), acc0);
              acc1 = fmaf(p1.w, __int2float_rn(static_cast<int>(v1[l + 3])), acc1);
            }
            if (b0 + j0 < a.B) emit<kFast>(a, b0 + j0, v_feat, fmaf(a.um_v, acc0, pbv));
            if (b0 + j0 + 1 < a.B) emit<kFast>(a, b0 + j0 + 1, v_feat, fmaf(a.um_v, acc1, pbv));
          } else {
            const int j = vj0;
            const float* pr = s_p + (j * kH + v_head) * kRow;
            float acc0 = 0.0f, acc1 = 0.0f;  // the two key blocks advance together
#pragma unroll
            for (int l = 0; l < kKeys; l += 4) {
              const float4 p0 = *reinterpret_cast<const float4*>(pr + l);
              const float4 p1 = *reinterpret_cast<const float4*>(pr + kKeys + l);
              acc0 = fmaf(p0.x, __int2float_rn(static_cast<int>(v0[l])), acc0);
              acc1 = fmaf(p1.x, __int2float_rn(static_cast<int>(v1[l])), acc1);
              acc0 = fmaf(p0.y, __int2float_rn(static_cast<int>(v0[l + 1])), acc0);
              acc1 = fmaf(p1.y, __int2float_rn(static_cast<int>(v1[l + 1])), acc1);
              acc0 = fmaf(p0.z, __int2float_rn(static_cast<int>(v0[l + 2])), acc0);
              acc1 = fmaf(p1.z, __int2float_rn(static_cast<int>(v1[l + 2])), acc1);
              acc0 = fmaf(p0.w, __int2float_rn(static_cast<int>(v0[l + 3])), acc0);
              acc1 = fmaf(p1.w, __int2float_rn(static_cast<int>(v1[l + 3])), acc1);
            }
            if (b0 + j < a.B) emit<kFast>(a, b0 + j, v_feat, fmaf(a.um_v, acc0 + acc1, pbv));
          }
        } else
        if constexpr (KB == 1) {
          const int j0 = vj0;
          const int len_v[2] = {min(s_len[j0], a.T), min(s_len[j0 + 1], a.T)};
          if (len_v[0] == kKeys && len_v[1] == kKeys && b0 + j0 + 1 < a.B) {
            // both sentences full: their two chains advance together
            const float* pr0 = s_p + (j0 * kH + v_head) * kKeys;
            const float* pr1 = pr0 + kH * kKeys;
            float acc0 = 0.0f, acc1 = 0.0f;
#pragma unroll
            for (int l = 0; l < kKeys; l += 4) {
              const float4 p0 = *reinterpret_cast<const float4*>(pr0 + l);
              const float4 p1 = *reinterpret_cast<const float4*>(pr1 + l);
              acc0 = fmaf(p0.x, dequant1(static_cast<int>(v0[l]), a.um_v, pbv), acc0);
              acc1 = fmaf(p1.x, dequant1(static_cast<int>(v1[l]), a.um_v, pbv), acc1);
              acc0 = fmaf(p0.y, dequant1(static_cast<int>(v0[l + 1]), a.um_v, pbv), acc0);
              acc1 = fmaf(p1.y, dequant1(static_cast<int>(v1[l + 1]), a.um_v, pbv), acc1);
              acc0 = fmaf(p0.z, dequant1(static_cast<int>(v0[l + 2]), a.um_v, pbv), acc0);
              acc1 = fmaf(p1.z, dequant1(static_cast<int>(v1[l + 2]), a.um_v, pbv), acc1);
              acc0 = fmaf(p0.w, dequant1(static_cast<int>(v0[l + 3]), a.um_v, pbv), acc0);
              acc1 = fmaf(p1.w, dequant1(static_cast<int>(v1[l + 3]), a.um_v, pbv), acc1);
            }
            emit<kFast>(a, b0 + j0, v_feat, acc0);
            emit<kFast>(a, b0 + j0 + 1, v_feat, acc1);
          } else {
#pragma unroll
            for (int jj = 0; jj < 2; jj++) {
              const int j = j0 + jj;
              const int b = b0 + j;
              if (b >= a.B) continue;
              // ragged sentence: only its own keys take part (the rows beyond belong to the next sentence)
              const int len = len_v[jj];
              const float* pr = s_p + (j * kH + v_head) * kKeys;
              const uint32_t* vv = jj == 0 ? v0 : v1;
              float acc = 0.0f;
#pragma unroll
              for (int l = 0; l < kKeys; l++) {
                if (l < len) acc = fmaf(pr[l], dequant1(static_cast<int>(vv[l]), a.um_v, pbv), acc);
              }
              emit<kFast>(a, b, v_feat, acc);
            }
          }
        } else {
          // one sentence, one chain over its keys in order: block 0 (v0) then block 1 (v1)
          const int j = vj0;
          const int b = b0 + j;
          if (b < a.B) {
            const int len = min(s_len[j], a.T);
            const float* pr = s_p + (j * kH + v_head) * kRow;
            float acc = 0.0f;
            if (len == kRow) {
              acc = v_chain32(acc, pr, v0, a.um_v, pbv);
              acc = v_chain32(acc, pr + kKeys, v1, a.um_v, pbv);
            } else {
#pragma unroll
              for (int l = 0; l < kKeys; l++) {
                if (l < len) acc = fmaf(pr[l], dequant1(static_cast<int>(v0[l]), a.um_v, pbv), acc);
              }
#pragma unroll
              for (int l = 0; l < kKeys; l++) {
                if (kKeys + l < len) acc = fmaf(pr[kKeys + l], dequant1(static_cast<int>(v1[l]), a.um_v, pbv), acc);
              }
            }
            emit<kFast>(a, b, v_feat, acc);
          }
        }
      }
      if (g + static_cast<int>(gridDim.x) < n_groups) request_k(ph ^ 1);  // the next group's K accumulators, see above
    }
  }
  rc_teardown(tmem, warp);
}

// ================================================ one sentence at a time, 65 .. 256 tokens
//
// The sentence-at-a-time sibling of the kernel above (softmax: slimt/TensorOps.cc:282-315).  The cached kernel
// (cross_attention.cu) streams 2 * len * E * 4 bytes of f32 K / V per sentence, layer and step and sits at 90 % of the
// HBM roofline on the mixed-length workload; this kernel reads the u8 PrepareA bytes instead, like the one above.
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

constexpr int kGKeys = 128;       // key rows per group
constexpr int kMaxS = 256;
constexpr int kMaxGroups = kMaxS / kGKeys;

struct SmemL : SmemHead {
  static constexpr int ring = tiles;
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

__global__ void __launch_bounds__(kThreads, 1) cross_attention_rcl_kernel(const __grid_constant__ CrossRcArgs a) {
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
  // D_v is drained by the eight warps that own output features
  const uint32_t tmem = rc_prologue(a, bars, tmem_slot, exp_tab, s_pbk, warp, lane, kConsWarps / 2);
  const uint32_t tmem_k = tmem;        // 256 columns: features
  const uint32_t tmem_v = tmem + 256;  // 2 blocks x 128 columns: key rows of the group

  auto length_of = [&](int b) { return max(1, min(static_cast<int>(__ldg(a.lengths + b)), a.T)); };

  if (warp == 0) {
    // ===== TMA producer: Wk, Wv once, then every sentence's operand tiles in consumption order
    if (elect_one()) {
      load_weights(a, s_wk, s_wv, w_full);
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
      mbar_wait(w_full, 0);
      uint32_t tile = 0, ck = 0, cv = 0;
      for (int b = blockIdx.x; b < a.B; b += gridDim.x) {
        const int ng = groups_of(length_of(b));
        for (int gi = 0; gi < ng; gi++, tile++, ck++) {
          const uint32_t s = tile & 1, ph = (tile >> 1) & 1;
          mbar_wait(&full[s], ph);
          mbar_wait(k_drained, (ck & 1) ^ 1);
          tc_fence_after();
          mma_k(tmem_k, s_ring + s * kTile, s_wk);
          umma_commit(k_done);
          umma_commit(&empty[s]);
        }
        for (int gi = 0; gi < ng; gi++, tile++, cv++) {
          const uint32_t s = tile & 1, ph = (tile >> 1) & 1;
          mbar_wait(&full[s], ph);
          mbar_wait(v_drained, (cv & 1) ^ 1);
          tc_fence_after();
          mma_v(tmem_v, s_wv, s_ring + s * kTile);
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
          exact_scores2(sc[gi], s_q + h0 * kDH, s_pbk, h0, v0, v1, a.um_k, a.dk);
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
            if (left > 0) acc = v_chain32(acc, pr, v0, a.um_v, pbv);
            if (left > kKeys) acc = v_chain32(acc, pr + kKeys, v1, a.um_v, pbv);
          }
        }
        emit<false>(a, b, v_feat, acc);
      }
    }
  }
  rc_teardown(tmem, warp);
}

}  // namespace

bool cross_attention_rc_supported(int E, int H, int dh, int S) {
  return E == kE && H == kH && dh == kDH && S >= 1 && S <= 2 * kKeys;
}

int launch_cross_attention_rc(const CrossRcArgs& a, int num_sms, bool fast, cudaStream_t stream) {
  if (a.B == 0) return 0;
  const bool two = a.T > kKeys;  // sentences of 33..64 tokens take two key blocks each
  const int per_group = two ? kGroup / 2 : kGroup;
  const int groups = (a.B + per_group - 1) / per_group;
  auto kern = two ? (fast ? cross_attention_rc_kernel<2, true> : cross_attention_rc_kernel<2, false>)
                  : (fast ? cross_attention_rc_kernel<1, true> : cross_attention_rc_kernel<1, false>);
  if (ensure_dyn_smem(kern, Smem::total) != cudaSuccess) return 1;
  return launch_pdl(kern, dim3(groups < num_sms ? groups : num_sms), dim3(kThreads), Smem::total, stream, a) != cudaSuccess;
}

bool cross_attention_rcl_supported(int E, int H, int dh, int S) {
  return E == kE && H == kH && dh == kDH && S >= 1 && S <= kMaxS;
}

int launch_cross_attention_rcl(const CrossRcArgs& a, int num_sms, cudaStream_t stream) {
  if (a.B == 0) return 0;
  auto kern = cross_attention_rcl_kernel;
  if (ensure_dyn_smem(kern, SmemL::total) != cudaSuccess) return 1;
  return launch_pdl(kern, dim3(a.B < num_sms ? a.B : num_sms), dim3(kThreads), SmemL::total, stream, a) != cudaSuccess;
}

}  // namespace sb
