// Output projection fused with the greedy choice (reference: Decoder::step's affine /
// affine_with_select on Wemb, slimt/Transformer.cc:176-182, followed by greedy_sample /
// greedy_sample_from_words, :279-339).  [M rows] x [N vocabulary or shortlist columns], K = E.
//
// Persistent warp-specialised tcgen05 kernel: one CTA per SM walks a contiguous range of
// [128 x 256] output tiles in column-major tile order.  The weight tile (B, 256 columns x K) stays
// resident in shared memory for a whole run of row tiles -- it is the larger operand, so this halves
// the L2 -> SM traffic -- while the u8 activation tiles (A, 128 rows x 128-byte k-blocks) stream
// through a TMA/mbarrier ring; accumulators are double-buffered in TMEM (2 x 256 columns) so the MMAs
// of tile i+1 overlap the epilogue of tile i.  Sixteen epilogue warps (TMEM lane quadrant x column
// quarter) reduce their 64 columns to a first-maximum per row and publish (value, lowest index) with a
// filtered 64-bit atomicMax.
//
// Epilogue arithmetic.  The exact logit is y = fl(fl(float(v) * um) + pb[n]) with v the SHIFTED
// accumulator sum_k (qa+127)*B (UnquantizeAndAddBiasAndWrite).  Here A is the SIGNED qa, so TMEM holds
// v' = v - c127[n] (c127 = 127 * colsum(B), exact).  Per 32-column chunk the warp first forms an upper
// bound of every y in the chunk from integer data only:  ub = ru(float(max v') * um + dmax) + eta, where
// dmax = max_n (c127[n] * um + pb[n]) rounded up (precomputed per chunk) and eta covers the float
// roundings of the exact formula.  Only when ub can reach the row's best so far (read back from `best`,
// which other CTAs keep raising) are the 32 exact logits evaluated; a skipped chunk cannot contain the
// maximum, so the result is still the reference's first strict maximum.
#include <limits.h>
#include <stdio.h>

#include "exact_math.cuh"
#include "gemm_i8.cuh"
#include "ptx.cuh"

namespace sb {

namespace {

constexpr int kOutBN = 256;
constexpr int kOutStages = 4;  // a power of two: the ring position is a % and a / in the single-thread issue loops (6: +5 us)
constexpr int kOutThreads = 640;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 idle, warps 4-19 epilogue

__device__ __forceinline__ unsigned long long pack_best_out(float v, uint32_t idx) {
  if (v == 0.0f) v = 0.0f;  // canonicalise -0 so equal values compare equal
  uint32_t b = __float_as_uint(v);
  uint32_t key = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return (static_cast<unsigned long long>(key) << 32) | static_cast<unsigned long long>(0xFFFFFFFFu - idx);
}

// kFast (SLIMT_B200_MATH=fast): the greedy choice is taken on an INTEGER proxy of the logit instead of the float logit.
// y = um * (v' + c127[n]) + pb[n] = um * (v' + t[n]) with t[n] = c127[n] + pb[n] / um, and um > 0, so the argmax of y
// is the argmax of v' + t[n]; t[n] is rounded to an integer once per batch (ipb), which moves a logit by at most half
// a quantum um (~1e-5 of the logit range).  The epilogue is then two integer instructions per element -- x = (v' << 6)
// + ipb6[n] with ipb6[n] = (ipb[n] << 6) + (63 - n % 64) carrying the column's position inside the thread's 64-column
// strip so that ties keep the lowest index, and a running max -- with no divergence and no exact path.
template <int KB, bool kFast>  // K = 128 * KB bytes per row
__global__ void __launch_bounds__(kOutThreads, 1)
    out_argmax_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                      const float* __restrict__ pb, const int32_t* __restrict__ c127, const float* __restrict__ dmax,
                      const int32_t* __restrict__ ipb6, float um, float eta, int M, int N,
                      unsigned long long* __restrict__ best) {
  constexpr int kABytes = kBM * kBK;        // one k-block of A
  constexpr int kBBytes = kOutBN * kBK;     // one k-block of B
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* smem_b = smem;                     // resident weight tile: KB k-blocks
  uint8_t* smem_a = smem + KB * kBBytes;      // ring of activation k-blocks
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_a + kOutStages * kABytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kOutStages;
  uint64_t* b_full = bars + 2 * kOutStages;
  uint64_t* b_empty = b_full + 1;
  uint64_t* tmem_full = b_empty + 1;   // [2]
  uint64_t* tmem_empty = tmem_full + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (N + kOutBN - 1) / kOutBN;
  const int m_tiles = (M + kBM - 1) / kBM;
  const long total = static_cast<long>(n_tiles) * m_tiles;
  const int t_begin = static_cast<int>(total * blockIdx.x / gridDim.x);
  const int t_end = static_cast<int>(total * (blockIdx.x + 1) / gridDim.x);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kOutStages; s++) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(b_full, 1);
    mbar_init(b_empty, 1);
    for (int i = 0; i < 2; i++) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 16);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();  // everything above overlapped the previous kernel's tail; its outputs are visible from here on
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one()) {
      uint32_t kbc = 0;  // running k-block counter (ring position)
      uint32_t run = 0;  // running count of column-tile runs
      int cur_n = -1;
      for (int t = t_begin; t < t_end; t++) {
        const int n = t / m_tiles, m = t % m_tiles;
        if (n != cur_n) {
          mbar_wait(b_empty, (run & 1) ^ 1);
          mbar_expect_tx(b_full, KB * kBBytes);
#pragma unroll
          for (int kb = 0; kb < KB; kb++) tma_load_2d(smem_b + kb * kBBytes, &tma_b, b_full, kb * kBK, n * kOutBN);
          cur_n = n;
          run++;
        }
#pragma unroll
        for (int kb = 0; kb < KB; kb++, kbc++) {
          const uint32_t s = kbc % kOutStages;
          const uint32_t ph = (kbc / kOutStages) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          mbar_expect_tx(&full_bar[s], kABytes);
          tma_load_2d(smem_a + s * kABytes, &tma_a, &full_bar[s], kb * kBK, m * kBM);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (single thread) =====
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_i8(kBM, kOutBN) | (1u << 7);  // A signed: s8 x s8
      uint32_t kbc = 0, run = 0, i = 0;
      int cur_n = -1;
      for (int t = t_begin; t < t_end; t++, i++) {
        const int n = t / m_tiles;
        if (n != cur_n) {
          mbar_wait(b_full, run & 1);
          cur_n = n;
          run++;
        }
        const uint32_t buf = i & 1;
        mbar_wait(&tmem_empty[buf], ((i >> 1) & 1) ^ 1);
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < KB; kb++, kbc++) {
          const uint32_t s = kbc % kOutStages;
          const uint32_t ph = (kbc / kOutStages) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint64_t da = make_kmajor_sw128_desc(smem_u32(smem_a + s * kABytes));
          const uint64_t db = make_kmajor_sw128_desc(smem_u32(smem_b + kb * kBBytes));
#pragma unroll
          for (int k = 0; k < kBK / 32; k++) {
            umma_i8(tmem_base + buf * kOutBN, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          }
          umma_commit(&empty_bar[s]);
        }
        umma_commit(&tmem_full[buf]);
        const bool last_of_run = (t + 1 == t_end) || ((t + 1) / m_tiles != n);
        if (last_of_run) umma_commit(b_empty);
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: thread <-> TMEM lane <-> output row.  Sixteen warps: TMEM lane quadrant (warp % 4)
    // x column quarter (64 columns = two 32-column chunks).  Both chunks are pulled into registers and the
    // TMEM buffer is handed back to the MMA warp at once; bounds and (rarely) exact logits follow. =====
    const int e = warp - 4;
    const int q = warp & 3;
    const int quarter = e >> 2;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + quarter * 64;
    if constexpr (kFast) {
      uint32_t i = 0;
      unsigned long long seen_next = 0ull;
      if (t_begin < t_end) {
        const int row = (t_begin % m_tiles) * kBM + q * 32 + lane;
        seen_next = row < M ? __ldcg(best + row) : ~0ull;
      }
      for (int t = t_begin; t < t_end; t++, i++) {
        const int n = t / m_tiles, m = t % m_tiles;
        const uint32_t buf = i & 1;
        const unsigned long long seen = seen_next;
        if (t + 1 < t_end) {
          const int row = ((t + 1) % m_tiles) * kBM + q * 32 + lane;
          seen_next = row < M ? __ldcg(best + row) : ~0ull;
        }
        const int nb0 = n * kOutBN + quarter * 64;
        const int row = m * kBM + q * 32 + lane;
        // the strip's 64 proxy offsets: the same addresses for every lane and every row tile of this column run (L1)
        const int4* ip = reinterpret_cast<const int4*>(ipb6 + nb0);
        mbar_wait(&tmem_full[buf], (i >> 1) & 1);
        tc_fence_after();
        uint32_t v0[32], v1[32];
        tmem_ld32_nowait(lane_addr + buf * kOutBN, v0);
        tmem_ld32_nowait(lane_addr + buf * kOutBN + 32, v1);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[buf]);  // accumulators are in registers: release the buffer
        int x0 = INT_MIN, x1 = INT_MIN, x2 = INT_MIN, x3 = INT_MIN;  // four independent max chains
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const int4 c = __ldg(ip + (j >> 2));
          x0 = max(x0, (static_cast<int>(v0[j]) << 6) + c.x);
          x1 = max(x1, (static_cast<int>(v0[j + 1]) << 6) + c.y);
          x2 = max(x2, (static_cast<int>(v0[j + 2]) << 6) + c.z);
          x3 = max(x3, (static_cast<int>(v0[j + 3]) << 6) + c.w);
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const int4 c = __ldg(ip + 8 + (j >> 2));
          x0 = max(x0, (static_cast<int>(v1[j]) << 6) + c.x);
          x1 = max(x1, (static_cast<int>(v1[j + 1]) << 6) + c.y);
          x2 = max(x2, (static_cast<int>(v1[j + 2]) << 6) + c.z);
          x3 = max(x3, (static_cast<int>(v1[j + 3]) << 6) + c.w);
        }
        const int x = max(max(x0, x1), max(x2, x3));
        if (row < M) {
          const uint32_t col = static_cast<uint32_t>(nb0 + 63 - (x & 63));
          const uint32_t key = static_cast<uint32_t>(x >> 6) ^ 0x80000000u;  // order-preserving int -> uint
          const unsigned long long packed = (static_cast<unsigned long long>(key) << 32) | (0xFFFFFFFFu - col);
          if (packed > seen) atomicMax(best + row, packed);
        }
      }
    } else {
    const float ninf = -__int_as_float(0x7f800000);
    const int nch = (N + 31) >> 5;
    // prefetched per-tile inputs of the bound filter
    unsigned long long seen_next = 0ull;
    float dm0_next = ninf, dm1_next = ninf;
    auto prefetch = [&](int t) {
      const int n = t / m_tiles, m = t % m_tiles;
      const int row = m * kBM + q * 32 + lane;
      const int ch = (n * kOutBN + quarter * 64) >> 5;
      seen_next = row < M ? __ldcg(best + row) : ~0ull;
      dm0_next = ch < nch ? __ldg(dmax + ch) : ninf;
      dm1_next = ch + 1 < nch ? __ldg(dmax + ch + 1) : ninf;
    };
    // exact logits of one 32-column chunk held in v[]; returns the chunk maximum and its first column
    auto exact_chunk = [&](const uint32_t (&v)[32], int nb, float floor_v, float& mx, int& idx) {
      float y[32];
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        if (nb + j < N) {  // N % 8 == 0: groups of four are entirely inside or outside
          const float4 p4 = __ldg(reinterpret_cast<const float4*>(pb + nb + j));
          const int4 c4 = __ldg(reinterpret_cast<const int4*>(c127 + nb + j));
          y[j] = dequant1(static_cast<int>(v[j]) + c4.x, um, p4.x);
          y[j + 1] = dequant1(static_cast<int>(v[j + 1]) + c4.y, um, p4.y);
          y[j + 2] = dequant1(static_cast<int>(v[j + 2]) + c4.z, um, p4.z);
          y[j + 3] = dequant1(static_cast<int>(v[j + 3]) + c4.w, um, p4.w);
        } else {
          y[j] = y[j + 1] = y[j + 2] = y[j + 3] = ninf;
        }
      }
      float t8[8];
#pragma unroll
      for (int j = 0; j < 8; j++) t8[j] = fmaxf(fmaxf(y[4 * j], y[4 * j + 1]), fmaxf(y[4 * j + 2], y[4 * j + 3]));
      mx = fmaxf(fmaxf(fmaxf(t8[0], t8[1]), fmaxf(t8[2], t8[3])), fmaxf(fmaxf(t8[4], t8[5]), fmaxf(t8[6], t8[7])));
      // first column of the chunk that attains the maximum (greedy_sample keeps the first strict max).  The chunk is
      // evaluated whenever ANY row of the warp passes the bound filter (lane = row: every row has its own best so
      // far, measured ~54 % of warp-chunks), but its maximum only matters for a row it can raise: the 62-instruction
      // search is skipped unless some lane's exact maximum reaches that lane's floor.  A lane whose maximum stays
      // below its floor keeps idx = 31; its candidate then packs to a key below the stored best and is never written.
      idx = 31;
      if (__any_sync(0xffffffffu, mx >= floor_v)) {
#pragma unroll
        for (int j = 30; j >= 0; j--) idx = (y[j] == mx) ? j : idx;
      }
    };
    auto int_max32 = [](const uint32_t (&v)[32]) {
      int vt[8];
#pragma unroll
      for (int j = 0; j < 8; j++)
        vt[j] = max(max(static_cast<int>(v[4 * j]), static_cast<int>(v[4 * j + 1])),
                    max(static_cast<int>(v[4 * j + 2]), static_cast<int>(v[4 * j + 3])));
      return max(max(max(vt[0], vt[1]), max(vt[2], vt[3])), max(max(vt[4], vt[5]), max(vt[6], vt[7])));
    };
    if (t_begin < t_end) prefetch(t_begin);
    uint32_t i = 0;
    for (int t = t_begin; t < t_end; t++, i++) {
      const int n = t / m_tiles, m = t % m_tiles;
      const uint32_t buf = i & 1;
      const unsigned long long seen = seen_next;
      const float dm0 = dm0_next, dm1 = dm1_next;
      if (t + 1 < t_end) prefetch(t + 1);
      const int nb0 = n * kOutBN + quarter * 64;
      const int row = m * kBM + q * 32 + lane;
      mbar_wait(&tmem_full[buf], (i >> 1) & 1);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      tmem_ld32_nowait(lane_addr + buf * kOutBN, v0);
      tmem_ld32_nowait(lane_addr + buf * kOutBN + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);  // accumulators are in registers: release the buffer

      // the row's best so far, from any CTA (monotone: a stale value only weakens the filter)
      float thr = ninf;
      if (seen != 0ull) {
        const uint32_t key = static_cast<uint32_t>(seen >> 32);
        thr = __uint_as_float((key & 0x80000000u) ? (key & 0x7fffffffu) : ~key);
      }
      const float ub0 = nb0 < N ? __fadd_ru(__fmaf_ru(__int2float_rn(int_max32(v0)), um, dm0), eta) : ninf;
      const float ub1 = nb0 + 32 < N ? __fadd_ru(__fmaf_ru(__int2float_rn(int_max32(v1)), um, dm1), eta) : ninf;
      float bv = 0.0f;
      uint32_t bi = 0;
      bool have = false;
      if (__any_sync(0xffffffffu, ub0 >= thr && nb0 < N)) {
        float mx;
        int idx;
        exact_chunk(v0, nb0, thr, mx, idx);
        if (nb0 < N && ub0 >= thr) {
          bv = mx, bi = static_cast<uint32_t>(nb0 + idx), have = true;
          thr = fmaxf(thr, mx);
        }
      }
      if (__any_sync(0xffffffffu, ub1 >= thr && nb0 + 32 < N)) {
        float mx;
        int idx;
        exact_chunk(v1, nb0 + 32, thr, mx, idx);
        if (nb0 + 32 < N && ub1 >= thr && (!have || mx > bv)) {
          bv = mx, bi = static_cast<uint32_t>(nb0 + 32 + idx), have = true;
        }
      }
      if (row < M && have) {
        // `best` only grows: a stale read can only cause a redundant atomic, never a missed one
        const unsigned long long key = pack_best_out(bv, bi);
        if (key > seen) atomicMax(best + row, key);
      }
    }
    }  // exact epilogue
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

size_t out_smem_bytes(int KB) { return static_cast<size_t>(KB) * kOutBN * kBK + kOutStages * kBM * kBK + 256 + 1024; }

}  // namespace

int launch_gemm_out_argmax(const CUtensorMap& tma_a, const CUtensorMap& tma_b, const float* pb, const int32_t* c127,
                           const float* dmax, const int32_t* ipb6, float um, float eta, int M, int N, int K,
                           unsigned long long* best, int num_sms, cudaStream_t stream) {
  const int KB = K / kBK;
  const long tiles = static_cast<long>((M + kBM - 1) / kBM) * ((N + kOutBN - 1) / kOutBN);
  const int grid = static_cast<int>(tiles < num_sms ? tiles : num_sms);
  if (grid == 0) return 0;
  const size_t smem = out_smem_bytes(KB);
  const bool fast = ipb6 != nullptr;
  auto go = [&](auto kern) {
    if (ensure_dyn_smem(kern, smem) != cudaSuccess) return 1;
    return launch_pdl(kern, dim3(grid), dim3(kOutThreads), smem, stream, tma_a, tma_b, pb, c127, dmax, ipb6, um, eta, M, N,
                      best) != cudaSuccess ? 1 : 0;
  };
  if (KB == 2) return fast ? go(out_argmax_kernel<2, true>) : go(out_argmax_kernel<2, false>);
  if (KB == 4) return fast ? go(out_argmax_kernel<4, true>) : go(out_argmax_kernel<4, false>);
  return 1;
}

}  // namespace sb
