// See fused_rows.cuh.  sm_100a only.
#include "fused_rows.cuh"

#include <stdio.h>

#include "packed_best.cuh"
#include "rows_common.cuh"

namespace sb {

namespace {

using namespace rows;

constexpr int kR = kRowTile;          // rows per CTA tile == UMMA N
constexpr int kOpK = kR * 128;        // one k-block of an activation operand: 32 rows x 128 bytes

// =====================================================================================================
// SSRU cell + query projection
// =====================================================================================================
template <int E>
struct SsruSmem {
  static constexpr int EK = E / 128;
  static constexpr int kStages = 6;
  static constexpr int ring = 0;
  static constexpr int opnd_xf = ring + kStages * kWTile;
  static constexpr int opnd_xw = opnd_xf + EK * kOpK;
  static constexpr int opnd_h = opnd_xw + EK * kOpK;
  static constexpr int xs = opnd_h + EK * kOpK;
  static constexpr int stats = xs + kR * (E + 1) * 4;
  static constexpr int exp_tab = stats + 64 * 4;
  static constexpr int bars = exp_tab + 32 * 8;
  static constexpr int n_bars = 2 * kStages + 4;  // full empty x_full g0_done hq_ready g1_done
  static constexpr int tmem_slot = bars + n_bars * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
};

template <int E, bool kFast, bool kEmbed>
__global__ void __launch_bounds__(kThreads, 1) dec_ssru_kernel(const __grid_constant__ DecSsruArgs a) {
  using L = SsruSmem<E>;
  constexpr int EK = E / 128, EM = E / 128;
  constexpr int XS = E + 1;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* ring = smem + L::ring;
  uint8_t* opnd_xf = smem + L::opnd_xf;
  uint8_t* opnd_xw = smem + L::opnd_xw;
  uint8_t* opnd_h = smem + L::opnd_h;
  float* xs = reinterpret_cast<float*>(smem + L::xs);
  float* stats = reinterpret_cast<float*>(smem + L::stats);
  uint64_t* exp_tab = reinterpret_cast<uint64_t*>(smem + L::exp_tab);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint64_t* full = bars;
  uint64_t* empty = full + L::kStages;
  uint64_t* x_full = empty + L::kStages;
  uint64_t* g0_done = x_full + 1;
  uint64_t* hq_ready = g0_done + 1;
  uint64_t* g1_done = hq_ready + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&a.map_xf);
    tma_prefetch_desc(&a.map_xw);
    tma_prefetch_desc(&a.map_wf);
    tma_prefetch_desc(&a.map_w);
    tma_prefetch_desc(&a.map_wq);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < L::kStages; s++) mbar_init(&full[s], 1), mbar_init(&empty[s], 1);
    mbar_init(x_full, kEmbed ? kEpiWarps : 1);  // kEmbed: the epilogue warps build the x operands themselves
    mbar_init(g0_done, 1);
    mbar_init(hq_ready, kEpiWarps);
    mbar_init(g1_done, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  if (warp == 3) exp_tab[lane] = kExp2fTab[lane];
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  const uint32_t tmem = *tmem_slot;
  const uint32_t tmem_f = tmem;                    // gate pre-activations Wf x
  const uint32_t tmem_w = tmem + EM * kR;          // W x
  const uint32_t tmem_q = tmem + 2 * EM * kR;      // Wq h

  const int n_tiles = (a.M + kR - 1) / kR;
  uint32_t iter = 0;
  RingProducer prod{ring, full, empty, 0, L::kStages};
  RingConsumer<kR> cons{ring, full, empty, 0, L::kStages};

  // One leader lane per warp, elected once (elect.sync also tells the compiler the branch is single-threaded, so
  // descriptors and addresses stay in uniform registers: no per-MMA waterfall loop as with `lane == 0`).  The ring
  // positions live in the leader's registers across tiles, hence a single election.
  const bool leader = elect_one();
  pdl_wait();  // everything above overlapped the previous kernel's tail; its outputs are visible from here on
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, iter++) {
    const int row0 = tile * kR;
    const uint32_t tph = iter & 1;
    if (warp == 0) {
      if (leader) {
        if constexpr (!kEmbed) {
          mbar_expect_tx(x_full, 2 * EK * kOpK);
          for (int kb = 0; kb < EK; kb++) {
            tma_load_2d(opnd_xf + kb * kOpK, &a.map_xf, x_full, kb * 128, row0);
            tma_load_2d(opnd_xw + kb * kOpK, &a.map_xw, x_full, kb * 128, row0);
          }
        }
        // the weight stream of one tile in consumption order
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) prod.load(&a.map_wf, kb, mb);
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) prod.load(&a.map_w, kb, mb);
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) prod.load(&a.map_wq, kb, mb);
      }
    } else if (warp == 1) {
      if (leader) {
        mbar_wait(x_full, tph);
        if constexpr (kEmbed) tc_fence_after();
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) cons.mma(tmem_f + mb * kR, opnd_xf + kb * kOpK, kb == 0);
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) cons.mma(tmem_w + mb * kR, opnd_xw + kb * kOpK, kb == 0);
        umma_commit(g0_done);
        mbar_wait(hq_ready, tph);
        tc_fence_after();
        for (int mb = 0; mb < EM; mb++)
          for (int kb = 0; kb < EK; kb++) cons.mma(tmem_q + mb * kR, opnd_h + kb * kOpK, kb == 0);
        umma_commit(g1_done);
      }
    } else if (warp >= 4) {
      const int ew = warp - 4;
      const int q = warp & 3;
      const int rq = ew >> 2;
      const int et = threadIdx.x - 128;
      const uint32_t lane_sel = static_cast<uint32_t>(q * 32) << 16;
      constexpr int kParts = kEpiThreads / E;
      constexpr int kRowsPer = kR / kParts;
      const int nf = et % E;
      const int nr0 = (et / E) * kRowsPer;

      // ---- highway + relu + residual (slimt/Modules.cc:218-232, TensorOps.cc:662-682) -> xs
      {
        float st[EM][8], xv[EM][8];  // previous cell state and layer input of this thread's (rows, features)
        if constexpr (kEmbed) {
          // the previous step's bookkeeping for the tile's rows (finalize_step_kernel's, thread = row), then the
          // words' embedding rows -> x (registers) and its two quantised operands (shared memory, UMMA layout)
          uint32_t* s_tok = reinterpret_cast<uint32_t*>(stats);  // free until the LayerNorm statistics
          // Only packed best -> shortlist -> token is on the path to the x operands: the row's other inputs are requested
          // alongside the first load, and record() itself (Model.cc:127-137) runs after the operands are handed over.
          uint32_t word = 0, was_done = 1, len_before = 0;
          const int bk = row0 + et;
          if (et < kR) {
            uint32_t tok = 0;
            if (bk < a.M) {
              const unsigned long long packed = a.best[bk];
              was_done = a.done[bk];
              len_before = a.tgt_len[bk];
              const uint32_t forced = a.forced ? a.forced[static_cast<size_t>(a.prev_step) * a.M + bk] : 0u;
              word = best_word(packed, a.shortlist);
              tok = a.forced ? forced : word;
            }
            s_tok[et] = tok;
          }
          named_bar_sync(1, kEpiThreads);
          // swizzled byte offset of (row, f) inside an operand k-block is row * 128 + xo[row & 7] (rows_common.cuh: opnd_off)
          uint32_t xo[8];
          {
            const int kk = q * 32 + lane;
#pragma unroll
            for (int i = 0; i < 8; i++) xo[i] = static_cast<uint32_t>((((kk >> 4) ^ i) << 4) + (kk & 15));
          }
#pragma unroll
          for (int mb = 0; mb < EM; mb++) {
            const int f = mb * 128 + q * 32 + lane;
            const float ps = a.pos0[f];
#pragma unroll
            for (int r = 0; r < 8; r++) {
              const int row = rq * 8 + r;
              const float y = embed1(a.emb_q[static_cast<size_t>(s_tok[row]) * E + f], a.inv_qm, a.sqrt_e, ps);
              xv[mb][r] = y;
              const uint32_t off = static_cast<uint32_t>(mb * kOpK + row * 128) + xo[r];  // row & 7 == r: rq * 8 is a multiple of 8
              opnd_xf[off] = static_cast<uint8_t>(quantize1(y, a.aq_xf));
              opnd_xw[off] = static_cast<uint8_t>(quantize1(y, a.aq_xw));
            }
          }
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(x_full);
          if (et < kR && bk < a.M)
            record_word(word, was_done, len_before, a.eos_id, a.prev_step, a.M, bk, a.step_tokens, a.done, a.tgt_len,
                        a.n_done, a.best);
        }
#pragma unroll
        for (int mb = 0; mb < EM; mb++) {
#pragma unroll
          for (int r = 0; r < 8; r++) {
            const int grow = row0 + rq * 8 + r;
            const size_t o = static_cast<size_t>(grow < a.M ? grow : 0) * E + mb * 128 + q * 32 + lane;
            st[mb][r] = a.state[o];
            if constexpr (!kEmbed) xv[mb][r] = a.x[o];
          }
        }
        mbar_wait(g0_done, tph);
        tc_fence_after();
#pragma unroll
        for (int mb = 0; mb < EM; mb++) {
          uint32_t vf[8], vw[8];
          tmem_ld8_nowait(tmem_f + lane_sel + mb * kR + rq * 8, vf);
          tmem_ld8_nowait(tmem_w + lane_sel + mb * kR + rq * 8, vw);
          const int f = mb * 128 + q * 32 + lane;
          const float pbf = a.pb_f[f], pbw = a.pb_w[f];
          tmem_ld_wait();
#pragma unroll
          for (int r = 0; r < 8; r++) {
            const int grow = row0 + rq * 8 + r;
            float sg, c;
            const float wx = dequant<kFast>(static_cast<int>(vw[r]), a.um_w, pbw);
            if constexpr (kFast) {
              sg = sigmoid_fast(dequant<true>(static_cast<int>(vf[r]), a.um_f, pbf));
              c = fmaf(sg, st[mb][r] - wx, wx);  // sg * c_prev + (1 - sg) * Wx
            } else {
              sg = sigmoid_ref_tab(dequant1(static_cast<int>(vf[r]), a.um_f, pbf), exp_tab);
              c = __fadd_rn(__fmul_rn(sg, st[mb][r]), __fmul_rn(__fsub_rn(1.0f, sg), wx));
            }
            if (grow < a.M) a.state[static_cast<size_t>(grow) * E + f] = c;
            xs[(rq * 8 + r) * XS + f] = __fadd_rn(xv[mb][r], c > 0.0f ? c : 0.0f);
          }
        }
      }
      named_bar_sync(1, kEpiThreads);
      if constexpr (kFast) ln_stats_fast<E, kR>(xs, stats, a.eps, ew, lane);
      else if (et < kR) ln_stats_row<E>(xs + et * XS, &stats[et], &stats[32 + et], a.eps);
      named_bar_sync(1, kEpiThreads);
      {
        const float g = a.ln_scale[nf], b = a.ln_bias[nf];
#pragma unroll 4
        for (int r = nr0; r < nr0 + kRowsPer; r++) {
          const float y = ln_apply_t<kFast>(xs[r * XS + nf], stats[r], stats[32 + r], g, b);
          opnd_h[opnd_off<kR>(r, nf)] = static_cast<uint8_t>(quantize<kFast>(y, a.aq_q));
          const int grow = row0 + r;
          if (grow < a.M) a.h_out[static_cast<size_t>(grow) * E + nf] = y;
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(hq_ready);

      // ---- q = Wq h + bq -> global
      mbar_wait(g1_done, tph);
      tc_fence_after();
#pragma unroll
      for (int mb = 0; mb < EM; mb++) {
        uint32_t v[8];
        tmem_ld8_nowait(tmem_q + lane_sel + mb * kR + rq * 8, v);
        const int f = mb * 128 + q * 32 + lane;
        const float pb = a.pb_q[f];
        tmem_ld_wait();
#pragma unroll
        for (int r = 0; r < 8; r++) {
          const int grow = row0 + rq * 8 + r;
          if (grow < a.M) a.q_out[static_cast<size_t>(grow) * E + f] = dequant<kFast>(static_cast<int>(v[r]), a.um_q, pb);
        }
      }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
  }
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// =====================================================================================================
// SSRU scan of the scoring pass (DecSsruScanArgs)
// =====================================================================================================
// One CTA per sentence, thread = feature: the thread carries its feature's cell state c through the positions in order.
// A tile of kScanRows positions is scanned into shared memory first, so that the LayerNorm statistics -- a sequential
// E-long chain per row -- run one row per thread of the first warp instead of one chain per position.  Padded positions
// (beyond the target's length) are computed and discarded by the caller; the scan is causal, so they affect no valid row.
constexpr int kScanRows = 32;

template <int E>
__global__ void __launch_bounds__(E) dec_ssru_scan_kernel(const DecSsruScanArgs a) {
  constexpr int XS = E + 1;
  extern __shared__ float scan_sm[];
  float* xs = scan_sm;                       // [kScanRows][E + 1]
  float* stats = xs + kScanRows * XS;        // mean [kScanRows], sigma [kScanRows]
  __shared__ uint64_t exp_tab[32];
  const int f = threadIdx.x;
  if (f < 32) exp_tab[f] = kExp2fTab[f];
  __syncthreads();
  const int T = a.T;
  const size_t row0 = static_cast<size_t>(blockIdx.x) * T;
  const float g = a.ln_scale[f], bias = a.ln_bias[f];
  float c = 0.0f;  // Decoder::start_states
  for (int j0 = 0; j0 < T; j0 += kScanRows) {
    const int nr = min(kScanRows, T - j0);
#pragma unroll 4
    for (int r = 0; r < nr; r++) {
      const size_t o = (row0 + j0 + r) * E + f;
      const float sg = sigmoid_ref_tab(a.f[o], exp_tab);
      c = __fadd_rn(__fmul_rn(sg, c), __fmul_rn(__fsub_rn(1.0f, sg), a.wx[o]));
      xs[r * XS + f] = __fadd_rn(a.x[o], c > 0.0f ? c : 0.0f);
    }
    __syncthreads();
    if (f < nr) ln_stats_row<E>(xs + f * XS, &stats[f], &stats[kScanRows + f], a.eps);
    __syncthreads();
    for (int r = 0; r < nr; r++) {
      const size_t o = (row0 + j0 + r) * E + f;
      const float y = ln_apply(xs[r * XS + f], stats[r], stats[kScanRows + r], g, bias);
      a.h_out[o] = y;
      a.hq[o] = static_cast<uint8_t>(quantize1(y, a.aq_q));
    }
    __syncthreads();
  }
}

template <class Kern, class Args>
int launch_rows(Kern kern, const Args& a, size_t smem, cudaStream_t stream) {
  const int tiles = (a.M + kR - 1) / kR;
  if (tiles == 0) return 0;
  ensure_dyn_smem(kern, smem);
  int sms = 148;
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (launch_pdl(kern, dim3(tiles < sms ? tiles : sms), dim3(kThreads), smem, stream, a) != cudaSuccess) return 1;
  return 0;
}

}  // namespace

template <int E>
int launch_ssru_e(const DecSsruArgs& a, bool fast, cudaStream_t stream) {
  constexpr size_t smem = SsruSmem<E>::total;
  if (a.embed)
    return fast ? launch_rows(dec_ssru_kernel<E, true, true>, a, smem, stream) : launch_rows(dec_ssru_kernel<E, false, true>, a, smem, stream);
  return fast ? launch_rows(dec_ssru_kernel<E, true, false>, a, smem, stream) : launch_rows(dec_ssru_kernel<E, false, false>, a, smem, stream);
}

int launch_dec_ssru(const DecSsruArgs& a, int E, bool fast, cudaStream_t stream) {
  if (E == 256) return launch_ssru_e<256>(a, fast, stream);
  if (E == 512) return launch_ssru_e<512>(a, fast, stream);
  return 1;
}

int launch_dec_ssru_scan(const DecSsruScanArgs& a, int E, cudaStream_t stream) {
  if (a.B == 0 || a.T == 0) return 0;
  const size_t smem = (static_cast<size_t>(kScanRows) * (E + 1) + 2 * kScanRows) * sizeof(float);
  auto go = [&](auto kern) {
    if (ensure_dyn_smem(kern, smem) != cudaSuccess) return 1;
    kern<<<a.B, E, smem, stream>>>(a);
    return cudaGetLastError() != cudaSuccess ? 1 : 0;
  };
  if (E == 256) return go(dec_ssru_scan_kernel<256>);
  if (E == 512) return go(dec_ssru_scan_kernel<512>);
  return 1;
}

}  // namespace sb
