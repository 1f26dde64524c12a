// Output projection fused with the greedy choice (reference: Decoder::step's affine / affine_with_select on Wemb,
// slimt/Transformer.cc:176-182, then greedy_sample / greedy_sample_from_words, :279-339).  See out_argmax.cuh.
//
// Persistent warp-specialised tcgen05 kernel: one CTA per SM walks a contiguous range of [128 x 256] output tiles in
// column-major tile order.  The weight tile (256 columns x K) stays resident in shared memory for a whole run of row
// tiles -- it is the larger operand, so this halves the L2 -> SM traffic -- while the s8 activation tiles (128 rows x
// 128-byte k-blocks) stream through a TMA/mbarrier ring; accumulators are double-buffered in TMEM (2 x 256 columns) so
// that the MMAs of tile i+1 overlap the epilogue of tile i.  Sixteen epilogue warps (TMEM lane quadrant x 64-column
// strip) reduce their columns to a candidate per row and publish it with a filtered 64-bit atomicMax into `best`,
// which all CTAs keep raising (a stale read of it only weakens the filter).
//
// The exact logit is y[n] = fl(fl(float(v' + c127[n]) * um) + pb[n]), v' the accumulator of the SIGNED qa held in
// TMEM (UnquantizeAndAddBiasAndWrite's shifted accumulator is v' + c127, c127 = 127 * colsum(B)).
//
// Digits.  y[n] ~ um * (v' + t[n]), t[n] = c127[n] + pb[n] / um.  t[n] is rounded to an integer ipb[n] once per batch
// and written as 32 int8 digits e[n][0..31] with sum_k a_k * e[n][k] = ipb[n] for the constants a = (127 x 31, 1).  One
// extra K = 32 MMA per tile with a constant A block (every row = a) and the digit block of the resident column tile as
// B adds ipb[n] to every accumulator: TMEM then holds the integer PROXY P = v' + ipb[n] of the logit,
// |y / um - P| <= 1.25 (half a unit from the rounding of t[n], the rest from the two float roundings of the exact
// formula; |v' + c127| < 2^23).  A thread reduces its 64 columns to eight group maxima and their maximum m with 3-input
// integer max instructions (36 instead of ~190 instructions per tile) and compares m with the row's best so far; only
// when m can matter does it look at individual columns:
//   tolerance mode  the proxy IS the score: the first column attaining m is the strip's candidate;
//   exact mode      every column with P >= max(m, floor) - 3 is evaluated with the exact formula (a column that loses
//                   by more than 2.5 proxy units provably has the smaller float logit), first strict maximum kept --
//                   the result is bit-identical to the reference's greedy choice, ties included.
//
// Bound filter, for a model whose offsets exceed the digits (|ipb| > 500 093).  Per 32-column chunk the warp first
// forms an upper bound of every y in the chunk from integer data only: ub = ru(float(max v') * um + dmax) + eta, where
// dmax = max_n (c127[n] * um + pb[n]) rounded up (per chunk) and eta covers the float roundings of the exact formula.
// Only when ub can reach the row's best so far are the 32 exact logits evaluated; a skipped chunk cannot contain the
// maximum, so the result is the reference's first strict maximum in either arithmetic mode.
#include "out_argmax.cuh"

#include <limits.h>
#include <stdio.h>

#include "exact_math.cuh"
#include "gemm_i8.cuh"
#include "packed_best.cuh"
#include "ptx.cuh"
#include "score_partial.cuh"

namespace sb {

namespace {

constexpr int kBN = kOutBN;
constexpr int kThreads = 640;  // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warp3 idle, warps 4-19 epilogue
constexpr int kDelta = 3;      // proxy units; 2 * 1.25 rounded up

template <bool kDigits, int KB>
struct Smem {
  static constexpr int kStages = kDigits && KB == 4 ? 2 : 4;      // activation ring (k-blocks of 16 KB); a power of two
  static constexpr int b = 0;                                      // resident weight tile: KB k-blocks x [256 x 128 B]
  static constexpr int b_ext = b + KB * kBN * kBK;                 // digits: the tile's digit block [256 x 128 B], 32 B used per row
  static constexpr int a_ext = b_ext + (kDigits ? kBN * kBK : 0);  // digits: constant A block [128 x 128 B], 32 B used per row
  static constexpr int a = a_ext + (kDigits ? kBM * kBK : 0);      // activation ring
  static constexpr int bars = a + kStages * kBM * kBK;  // full[kStages] empty[kStages] b_full b_empty tmem_full[2] tmem_empty[2]
  static constexpr int tmem_slot = bars + (2 * kStages + 6) * 8;
  static constexpr int total = tmem_slot + 16 + 1024;
  static_assert(total <= 227 * 1024, "shared memory");
};

// ------------------------------------------------------------------ epilogues: one 64-column strip of one row
// Digits: the columns past a ragged N (N % 8 == 0) can never win; eight group maxima (columns 8k .. 8k + 7) and the
// strip maximum.
__device__ __forceinline__ int digit_groups(uint32_t (&v0)[32], uint32_t (&v1)[32], int nb0, int N, int (&g)[8]) {
  if (nb0 + 64 > N) {
#pragma unroll
    for (int j = 0; j < 32; j++) {
      if (nb0 + j >= N) v0[j] = 0x80000000u;
      if (nb0 + 32 + j >= N) v1[j] = 0x80000000u;
    }
  }
#pragma unroll
  for (int k = 0; k < 4; k++) {
    g[k] = max(max(max(static_cast<int>(v0[8 * k]), static_cast<int>(v0[8 * k + 1])),
                   max(static_cast<int>(v0[8 * k + 2]), static_cast<int>(v0[8 * k + 3]))),
               max(max(static_cast<int>(v0[8 * k + 4]), static_cast<int>(v0[8 * k + 5])),
                   max(static_cast<int>(v0[8 * k + 6]), static_cast<int>(v0[8 * k + 7]))));
    g[4 + k] = max(max(max(static_cast<int>(v1[8 * k]), static_cast<int>(v1[8 * k + 1])),
                       max(static_cast<int>(v1[8 * k + 2]), static_cast<int>(v1[8 * k + 3]))),
                   max(max(static_cast<int>(v1[8 * k + 4]), static_cast<int>(v1[8 * k + 5])),
                       max(static_cast<int>(v1[8 * k + 6]), static_cast<int>(v1[8 * k + 7]))));
  }
  return max(max(max(g[0], g[1]), max(g[2], g[3])), max(max(g[4], g[5]), max(g[6], g[7])));
}

// Digits, tolerance mode: the first column attaining the strip's maximum proxy.
__device__ __forceinline__ void digits_tolerance(const uint32_t (&v0)[32], const uint32_t (&v1)[32], const int (&g)[8],
                                                 int mx, unsigned long long seen, int row, int nb0, int M, int N,
                                                 unsigned long long* __restrict__ best) {
  const int seen_p = seen != 0ull ? best_proxy(seen) : INT_MIN;
  const bool trig = row < M && nb0 < N && mx >= seen_p;  // >=: an equal proxy in a lower column still wins
  if (__any_sync(0xffffffffu, trig)) {
    int bi = -1;
    int bvi = INT_MIN;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (__any_sync(0xffffffffu, trig && g[k] >= mx)) {
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
          const int j = 8 * k + jj;
          const int vj = static_cast<int>(j < 32 ? v0[j & 31] : v1[j & 31]);
          if (trig && vj >= mx) {
            if (vj > bvi) bvi = vj, bi = j;
          }
        }
      }
    }
    if (bi >= 0) {
      const unsigned long long packed = pack_best_proxy(bvi, static_cast<uint32_t>(nb0 + bi));
      if (packed > seen) atomicMax(best + row, packed);
    }
  }
}

// Digits, exact mode: the columns within kDelta proxy units of the strip's maximum and of the row's best so far, each
// evaluated with the exact formula; the first strict maximum.
__device__ __forceinline__ void digits_exact(const uint32_t (&v0)[32], const uint32_t (&v1)[32], const int (&g)[8],
                                             int mx, unsigned long long seen, int row, int nb0, int M, int N,
                                             const float* __restrict__ pb, const int32_t* __restrict__ dshift, float um,
                                             float inv_um, unsigned long long* __restrict__ best) {
  int floor_p = INT_MIN + 16;
  // proxy of the best column so far >= its logit / um - 1.25; the product itself is good to half a unit
  if (seen != 0ull) floor_p = __float2int_rd(best_value(seen) * inv_um) - 3;
  const bool trig = row < M && nb0 < N && mx >= floor_p - kDelta;
  const int thr = max(mx, floor_p) - kDelta;
  if (__any_sync(0xffffffffu, trig)) {
    int bi = -1;
    float bvf = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      if (__any_sync(0xffffffffu, trig && g[k] >= thr)) {
#pragma unroll
        for (int jj = 0; jj < 8; jj++) {
          const int j = 8 * k + jj;
          const int vj = static_cast<int>(j < 32 ? v0[j & 31] : v1[j & 31]);
          if (trig && vj >= thr) {
            const int col = nb0 + j;
            const float y = dequant1(vj + __ldg(dshift + col), um, __ldg(pb + col));
            if (bi < 0 || y > bvf) bvf = y, bi = j;
          }
        }
      }
    }
    if (bi >= 0) {
      const unsigned long long packed = pack_best(bvf, static_cast<uint32_t>(nb0 + bi));
      if (packed > seen) atomicMax(best + row, packed);
    }
  }
}

__device__ __forceinline__ int int_max32(const uint32_t (&v)[32]) {
  int vt[8];
#pragma unroll
  for (int j = 0; j < 8; j++)
    vt[j] = max(max(static_cast<int>(v[4 * j]), static_cast<int>(v[4 * j + 1])),
                max(static_cast<int>(v[4 * j + 2]), static_cast<int>(v[4 * j + 3])));
  return max(max(max(vt[0], vt[1]), max(vt[2], vt[3])), max(max(vt[4], vt[5]), max(vt[6], vt[7])));
}

// The exact logits of one 32-column chunk held in v[] (the logits tap's values); columns past N are -inf.
__device__ __forceinline__ void exact_logits32(const uint32_t (&v)[32], int nb, int N, const float* __restrict__ pb,
                                               const int32_t* __restrict__ c127, float um, float (&y)[32]) {
  const float ninf = -__int_as_float(0x7f800000);
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
}

// Bound filter: the exact logits of one 32-column chunk held in v[]; the chunk maximum and its first column.
__device__ __forceinline__ void exact_chunk(const uint32_t (&v)[32], int nb, int N, const float* __restrict__ pb,
                                            const int32_t* __restrict__ c127, float um, float floor_v, float& mx, int& idx) {
  float y[32];
  exact_logits32(v, nb, N, pb, c127, um, y);
  float t8[8];
#pragma unroll
  for (int j = 0; j < 8; j++) t8[j] = fmaxf(fmaxf(y[4 * j], y[4 * j + 1]), fmaxf(y[4 * j + 2], y[4 * j + 3]));
  mx = fmaxf(fmaxf(fmaxf(t8[0], t8[1]), fmaxf(t8[2], t8[3])), fmaxf(fmaxf(t8[4], t8[5]), fmaxf(t8[6], t8[7])));
  // first column of the chunk that attains the maximum (greedy_sample keeps the first strict max).  The chunk is
  // evaluated whenever ANY row of the warp passes the bound filter (lane = row: every row has its own best so far,
  // measured ~54 % of warp-chunks), but its maximum only matters for a row it can raise: the 62-instruction search is
  // skipped unless some lane's exact maximum reaches that lane's floor.  A lane whose maximum stays below its floor
  // keeps idx = 31; its candidate then packs to a key below the stored best and is never written.
  idx = 31;
  if (__any_sync(0xffffffffu, mx >= floor_v)) {
#pragma unroll
    for (int j = 30; j >= 0; j--) idx = (y[j] == mx) ? j : idx;
  }
}

// Bound filter, exact (both arithmetic modes): dm0 / dm1 are the dmax of the strip's two chunks.
__device__ __forceinline__ void bounds_exact(const uint32_t (&v0)[32], const uint32_t (&v1)[32], float dm0, float dm1,
                                             unsigned long long seen, int row, int nb0, int M, int N,
                                             const float* __restrict__ pb, const int32_t* __restrict__ c127, float um,
                                             float eta, unsigned long long* __restrict__ best) {
  const float ninf = -__int_as_float(0x7f800000);
  float thr = seen != 0ull ? best_value(seen) : ninf;
  const float ub0 = nb0 < N ? __fadd_ru(__fmaf_ru(__int2float_rn(int_max32(v0)), um, dm0), eta) : ninf;
  const float ub1 = nb0 + 32 < N ? __fadd_ru(__fmaf_ru(__int2float_rn(int_max32(v1)), um, dm1), eta) : ninf;
  float bv = 0.0f;
  uint32_t bi = 0;
  bool have = false;
  if (__any_sync(0xffffffffu, ub0 >= thr && nb0 < N)) {
    float mx;
    int idx;
    exact_chunk(v0, nb0, N, pb, c127, um, thr, mx, idx);
    if (nb0 < N && ub0 >= thr) {
      bv = mx, bi = static_cast<uint32_t>(nb0 + idx), have = true;
      thr = fmaxf(thr, mx);
    }
  }
  if (__any_sync(0xffffffffu, ub1 >= thr && nb0 + 32 < N)) {
    float mx;
    int idx;
    exact_chunk(v1, nb0 + 32, N, pb, c127, um, thr, mx, idx);
    if (nb0 + 32 < N && ub1 >= thr && (!have || mx > bv)) bv = mx, bi = static_cast<uint32_t>(nb0 + 32 + idx), have = true;
  }
  if (row < M && have) {
    const unsigned long long packed = pack_best(bv, bi);
    if (packed > seen) atomicMax(best + row, packed);
  }
}

// Scores (both arithmetic modes): every column's exact logit.  The strip's partial (m, s) (score_partial.cuh) goes to
// partials[strip][M]; its first maximum is published like the bound filter's, so the choice is the reference's first
// strict maximum.  seen only spares an atomic that cannot raise the word: it decides nothing that is summed.
// kTemper: the same over the tempered logits fl32(y * inv_t) (sampling at a temperature other than 1).
template <bool kTemper>
__device__ __forceinline__ void scores_exact(const uint32_t (&v0)[32], const uint32_t (&v1)[32], unsigned long long seen,
                                             int row, int nb0, int M, int N, const float* __restrict__ pb,
                                             const int32_t* __restrict__ c127, float um,
                                             unsigned long long* __restrict__ best, float2* __restrict__ partials,
                                             float inv_t) {
  if (nb0 >= N) return;  // the whole warp: a strip past the last column has no partial
  float y0[32], y1[32];
  exact_logits32(v0, nb0, N, pb, c127, um, y0);
  exact_logits32(v1, nb0 + 32, N, pb, c127, um, y1);
  if constexpr (kTemper) temper64(y0, y1, inv_t);
  const float2 p = strip_partial(y0, y1);
  if (row >= M) return;
  int idx = 63;
#pragma unroll
  for (int j = 62; j >= 0; j--) idx = ((j < 32 ? y0[j & 31] : y1[j & 31]) == p.x) ? j : idx;
  partials[static_cast<size_t>(nb0 / kScoreStrip) * M + row] = p;
  const unsigned long long packed = pack_best(p.x, static_cast<uint32_t>(nb0 + idx));
  if (packed > seen) atomicMax(best + row, packed);
}

// ------------------------------------------------------------------ the kernel
// kDigits: the encoding; kFast: tolerance mode (digits only); kScores: the scores epilogue (kDigits = false: the weights
// alone, no column table); kTemper: the scores epilogue over the tempered logits (sampling).
// tma_e / dshift / inv_um are read by the digits only, c127 by the bound filter and the scores, dmax / eta by the bound
// filter only, partials by the scores only, inv_t by kTemper only.
template <bool kDigits, int KB, bool kFast, bool kScores = false, bool kTemper = false>  // K = 128 * KB bytes per row
__global__ void __launch_bounds__(kThreads, 1)
    out_argmax_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                      const __grid_constant__ CUtensorMap tma_e, const float* __restrict__ pb,
                      const int32_t* __restrict__ dshift, float um, float inv_um, int M, int N,
                      unsigned long long* __restrict__ best, const int32_t* __restrict__ c127,
                      const float* __restrict__ dmax, float eta, float2* __restrict__ partials, float inv_t) {
  using L = Smem<kDigits, KB>;
  constexpr int kStages = L::kStages;
  constexpr int kABytes = kBM * kBK;
  constexpr int kBBytes = kBN * kBK;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_align1024(smem_raw);
  uint8_t* smem_b = smem + L::b;
  uint8_t* smem_be = smem + L::b_ext;
  uint8_t* smem_ae = smem + L::a_ext;
  uint8_t* smem_a = smem + L::a;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + L::bars);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kStages;
  uint64_t* b_full = bars + 2 * kStages;
  uint64_t* b_empty = b_full + 1;
  uint64_t* tmem_full = b_empty + 1;     // [2]
  uint64_t* tmem_empty = tmem_full + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + L::tmem_slot);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (N + kBN - 1) / kBN;
  const int m_tiles = (M + kBM - 1) / kBM;
  const long total = static_cast<long>(n_tiles) * m_tiles;
  const int t_begin = static_cast<int>(total * blockIdx.x / gridDim.x);
  const int t_end = static_cast<int>(total * (blockIdx.x + 1) / gridDim.x);
  const int n_first = t_begin / m_tiles, m_first = t_begin % m_tiles;  // the only division: tiles then advance by counting

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_b);
    if constexpr (kDigits) tma_prefetch_desc(&tma_e);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; s++) {
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
  if constexpr (kDigits) {
    // the constant A block of the extra k-step, in the K-major 128B-swizzled layout the MMA reads: row r, bytes 0..31
    // = (127 x 31, 1); 16-byte chunk c of a row sits at chunk position c ^ (r & 7)
    for (int i = threadIdx.x; i < kBM * 8; i += kThreads) {
      const int r = i >> 3, pos = i & 7;
      const int c = pos ^ (r & 7);
      uint4 val = make_uint4(0u, 0u, 0u, 0u);
      if (c == 0) val = make_uint4(0x7f7f7f7fu, 0x7f7f7f7fu, 0x7f7f7f7fu, 0x7f7f7f7fu);
      if (c == 1) val = make_uint4(0x7f7f7f7fu, 0x7f7f7f7fu, 0x7f7f7f7fu, 0x017f7f7fu);
      *reinterpret_cast<uint4*>(smem_ae + r * 128 + pos * 16) = val;
    }
    fence_proxy_async();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_launch_dependents();
  pdl_wait();  // everything above overlapped the previous kernel's tail; its outputs are visible from here on
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer =====
    if (elect_one()) {
      uint32_t kbc = 0, run = 0;
      int n = n_first, m = m_first, cur_n = -1;
      for (int t = t_begin; t < t_end; t++) {
        if (n != cur_n) {
          mbar_wait(b_empty, (run & 1) ^ 1);
          mbar_expect_tx(b_full, (KB + (kDigits ? 1 : 0)) * kBBytes);
#pragma unroll
          for (int kb = 0; kb < KB; kb++) tma_load_2d(smem_b + kb * kBBytes, &tma_b, b_full, kb * kBK, n * kBN);
          if constexpr (kDigits) tma_load_2d(smem_be, &tma_e, b_full, 0, n * kBN);
          cur_n = n;
          run++;
        }
#pragma unroll
        for (int kb = 0; kb < KB; kb++, kbc++) {
          const uint32_t s = kbc % kStages;
          const uint32_t ph = (kbc / kStages) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          mbar_expect_tx(&full_bar[s], kABytes);
          tma_load_2d(smem_a + s * kABytes, &tma_a, &full_bar[s], kb * kBK, m * kBM);
        }
        if (++m == m_tiles) m = 0, n++;
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (single thread) =====
    if (elect_one()) {
      constexpr uint32_t idesc = make_idesc_i8(kBM, kBN) | (1u << 7);  // A signed: s8 x s8
      const uint64_t dae = make_kmajor_sw128_desc(smem_u32(smem_ae));
      const uint64_t dbe = make_kmajor_sw128_desc(smem_u32(smem_be));
      uint32_t kbc = 0, run = 0, i = 0;
      int n = n_first, m = m_first, cur_n = -1;
      for (int t = t_begin; t < t_end; t++, i++) {
        if (n != cur_n) {
          mbar_wait(b_full, run & 1);
          cur_n = n;
          run++;
        }
        const uint32_t buf = i & 1;
        const uint32_t tmem_d = tmem_base + buf * kBN;
        mbar_wait(&tmem_empty[buf], ((i >> 1) & 1) ^ 1);
        tc_fence_after();
#pragma unroll
        for (int kb = 0; kb < KB; kb++, kbc++) {
          const uint32_t s = kbc % kStages;
          const uint32_t ph = (kbc / kStages) & 1;
          mbar_wait(&full_bar[s], ph);
          tc_fence_after();
          const uint64_t da = make_kmajor_sw128_desc(smem_u32(smem_a + s * kABytes));
          const uint64_t db = make_kmajor_sw128_desc(smem_u32(smem_b + kb * kBBytes));
#pragma unroll
          for (int k = 0; k < kBK / 32; k++) umma_i8(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          umma_commit(&empty_bar[s]);
        }
        if constexpr (kDigits) umma_i8(tmem_d, dae, dbe, idesc, 1u);  // + ipb[n]: the digit block against the constant block
        umma_commit(&tmem_full[buf]);
        const bool last_of_run = (t + 1 == t_end) || (m + 1 == m_tiles);
        if (last_of_run) umma_commit(b_empty);
        if (++m == m_tiles) m = 0, n++;
      }
    }
  } else if (warp >= 4) {
    // ===== epilogue: thread <-> TMEM lane <-> output row; warp = (lane quadrant, 64-column strip) =====
    const int e = warp - 4;
    const int q = warp & 3;
    const int quarter = e >> 2;
    const uint32_t lane_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + quarter * 64;
    const int row_in_tile = q * 32 + lane;
    const float ninf = -__int_as_float(0x7f800000);
    const int nch = (N + 31) >> 5;
    int n = n_first, m = m_first;
    // the next tile's inputs, requested before this tile's accumulators are waited for
    unsigned long long seen_next = 0ull;
    float dm0_next = ninf, dm1_next = ninf;  // bound filter: the strip's two chunk bounds
    auto prefetch = [&](int n, int m) {
      const int row = m * kBM + row_in_tile;
      seen_next = row < M ? __ldcg(best + row) : ~0ull;
      if constexpr (!kDigits && !kScores) {
        const int ch = (n * kBN + quarter * 64) >> 5;
        dm0_next = ch < nch ? __ldg(dmax + ch) : ninf;
        dm1_next = ch + 1 < nch ? __ldg(dmax + ch + 1) : ninf;
      }
    };
    if (t_begin < t_end) prefetch(n, m);
    uint32_t i = 0;
    for (int t = t_begin; t < t_end; t++, i++) {
      const uint32_t buf = i & 1;
      const unsigned long long seen = seen_next;
      const float dm0 = dm0_next, dm1 = dm1_next;
      const int nb0 = n * kBN + quarter * 64;
      const int row = m * kBM + row_in_tile;
      int m_nx = m + 1, n_nx = n;
      if (m_nx == m_tiles) m_nx = 0, n_nx++;
      if (t + 1 < t_end) prefetch(n_nx, m_nx);
      mbar_wait(&tmem_full[buf], (i >> 1) & 1);
      tc_fence_after();
      uint32_t v0[32], v1[32];
      tmem_ld32_nowait(lane_addr + buf * kBN, v0);
      tmem_ld32_nowait(lane_addr + buf * kBN + 32, v1);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[buf]);  // accumulators are in registers: release the buffer

      if constexpr (kScores) {
        scores_exact<kTemper>(v0, v1, seen, row, nb0, M, N, pb, c127, um, best, partials, inv_t);
      } else if constexpr (kDigits) {
        int g[8];
        const int mx = digit_groups(v0, v1, nb0, N, g);
        if constexpr (kFast)
          digits_tolerance(v0, v1, g, mx, seen, row, nb0, M, N, best);
        else
          digits_exact(v0, v1, g, mx, seen, row, nb0, M, N, pb, dshift, um, inv_um, best);
      } else {
        bounds_exact(v0, v1, dm0, dm1, seen, row, nb0, M, N, pb, c127, um, eta, best);
      }
      m = m_nx, n = n_nx;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) tmem_dealloc<512>(tmem_base);
}

// ------------------------------------------------------------------ per-column tables
// Digits, per output column n: ipb[n] = round(c127[n] + pb[n] / um) in double, written as 32 int8 digits e[n][0..31]
// with sum_k a_k * e[n][k] = ipb[n] for a = (127 x 31, 1), one 128-byte row per column (the layout the weight tile's TMA
// box uses; bytes 32..127 stay zero); dshift[n] = c127[n] - ipb[n] turns a proxy back into the shifted accumulator of
// the exact formula.  Columns N .. n_pad - 1 are zero.  *overflow (when given) is set when some |ipb| exceeds what the
// digits can hold (31 * 127 * 127 + 63).
__global__ void out_ext_kernel(const int32_t* __restrict__ c127, const float* __restrict__ pb, float um, int N, int n_pad,
                               uint8_t* __restrict__ ext, int32_t* __restrict__ dshift, int* __restrict__ overflow) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= n_pad) return;
  uint4* row = reinterpret_cast<uint4*>(ext + static_cast<size_t>(n) * 128);
  uint32_t w[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  int ds = 0;
  if (n < N) {
    double t = rint(static_cast<double>(c127[n]) + static_cast<double>(pb[n]) / static_cast<double>(um));
    if (fabs(t) > 500093.0) {
      if (overflow) atomicOr(overflow, 1);
      t = fmin(fmax(t, -500093.0), 500093.0);
    }
    const int ipb = static_cast<int>(t);
    int Q = static_cast<int>(rint(static_cast<double>(ipb) / 127.0));
    if (Q > 3937) Q = 3937;
    if (Q < -3937) Q = -3937;
    const int r = ipb - 127 * Q;  // |r| <= 63 (<= 126 at the clamped ends, still an int8)
    const int base = Q / 31, rem = Q - 31 * base;
    const int step = rem > 0 ? 1 : -1, cnt = rem > 0 ? rem : -rem;
    for (int k = 0; k < 32; k++) {
      const int d = k < 31 ? base + (k < cnt ? step : 0) : r;
      w[k >> 2] |= static_cast<uint32_t>(d & 0xff) << (8 * (k & 3));
    }
    ds = c127[n] - ipb;
  }
  row[0] = make_uint4(w[0], w[1], w[2], w[3]);
  row[1] = make_uint4(w[4], w[5], w[6], w[7]);
  for (int i = 2; i < 8; i++) row[i] = make_uint4(0u, 0u, 0u, 0u);
  dshift[n] = ds;
}

// Bound filter: dmax[chunk] = max over the chunk's 32 columns of (c127[n] * um + pb[n]), rounded up to float.
__global__ void out_bounds_kernel(const int32_t* __restrict__ c127, const float* __restrict__ pb, float um, int N,
                                  float* __restrict__ dmax) {
  const int chunk = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (chunk * 32 >= N) return;
  const int n = chunk * 32 + lane;
  double d = -1.0e300;
  if (n < N) d = static_cast<double>(c127[n]) * static_cast<double>(um) + static_cast<double>(pb[n]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) d = fmax(d, __shfl_xor_sync(0xffffffffu, d, o));
  if (lane == 0) dmax[chunk] = __double2float_ru(d);
}

}  // namespace

void launch_out_tables(const OutColumns& c, int* overflow, cudaStream_t stream) {
  if (c.digits) {
    const int n_pad = static_cast<int>(OutColumns::pad(c.N));
    if (n_pad == 0) return;
    out_ext_kernel<<<(n_pad + 127) / 128, 128, 0, stream>>>(c.c127, c.pb, c.um, c.N, n_pad, c.ext, c.dshift, overflow);
  } else {
    const int chunks = (c.N + 31) / 32;
    if (chunks == 0) return;
    out_bounds_kernel<<<(chunks + 7) / 8, 256, 0, stream>>>(c.c127, c.pb, c.um, c.N, c.dmax);
  }
}

int launch_out_argmax(const OutColumns& c, const CUtensorMap& tma_a, bool fast, int M, int K, unsigned long long* best,
                      int num_sms, cudaStream_t stream) {
  const int KB = K / kBK, N = c.N;
  const long tiles = static_cast<long>((M + kBM - 1) / kBM) * ((N + kBN - 1) / kBN);
  const int grid = static_cast<int>(tiles < num_sms ? tiles : num_sms);
  if (grid == 0) return 0;
  const float inv_um = 1.0f / c.um;
  auto go = [&](auto kern, size_t smem) {
    if (ensure_dyn_smem(kern, smem) != cudaSuccess) return 1;
    return launch_pdl(kern, dim3(grid), dim3(kThreads), smem, stream, tma_a, c.map_w, c.map_ext, c.pb, c.dshift, c.um,
                      inv_um, M, N, best, c.c127, c.dmax, c.eta, static_cast<float2*>(nullptr), 1.0f) != cudaSuccess ? 1 : 0;
  };
  if (!c.digits) {
    if (KB == 2) return go(out_argmax_kernel<false, 2, false>, Smem<false, 2>::total);
    if (KB == 4) return go(out_argmax_kernel<false, 4, false>, Smem<false, 4>::total);
    return 1;
  }
  if (KB == 2) return fast ? go(out_argmax_kernel<true, 2, true>, Smem<true, 2>::total) : go(out_argmax_kernel<true, 2, false>, Smem<true, 2>::total);
  if (KB == 4) return fast ? go(out_argmax_kernel<true, 4, true>, Smem<true, 4>::total) : go(out_argmax_kernel<true, 4, false>, Smem<true, 4>::total);
  return 1;
}

int launch_out_scores(const OutColumns& c, const CUtensorMap& tma_a, int M, int K, unsigned long long* best,
                      float2* partials, float inv_t, int num_sms, cudaStream_t stream) {
  const int KB = K / kBK, N = c.N;
  const long tiles = static_cast<long>((M + kBM - 1) / kBM) * ((N + kBN - 1) / kBN);
  const int grid = static_cast<int>(tiles < num_sms ? tiles : num_sms);
  if (grid == 0) return 0;
  auto go = [&](auto kern, size_t smem) {
    if (ensure_dyn_smem(kern, smem) != cudaSuccess) return 1;
    return launch_pdl(kern, dim3(grid), dim3(kThreads), smem, stream, tma_a, c.map_w, c.map_w, c.pb,
                      static_cast<const int32_t*>(nullptr), c.um, 0.0f, M, N, best, c.c127,
                      static_cast<const float*>(nullptr), 0.0f, partials, inv_t) != cudaSuccess ? 1 : 0;
  };
  // temperature 1: z = y bit for bit, so the untempered epilogue serves
  const bool temper = inv_t != 1.0f;
  if (KB == 2)
    return temper ? go(out_argmax_kernel<false, 2, false, true, true>, Smem<false, 2>::total)
                  : go(out_argmax_kernel<false, 2, false, true>, Smem<false, 2>::total);
  if (KB == 4)
    return temper ? go(out_argmax_kernel<false, 4, false, true, true>, Smem<false, 4>::total)
                  : go(out_argmax_kernel<false, 4, false, true>, Smem<false, 4>::total);
  return 1;
}

}  // namespace sb
