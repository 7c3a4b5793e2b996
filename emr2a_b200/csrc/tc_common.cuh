// Device helpers shared by the single-CTA (topk_tc.cu) and CTA-pair (topk_tc2.cu) tcgen05 kernels, and the list of
// their instantiations that both launch paths dispatch over.
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace emr2a {

constexpr int T_BM = 128;
constexpr int T_BN = 256;
constexpr int T_BK = 64;
constexpr int T_THREADS = 256;
constexpr uint32_t T_A_BYTES = T_BM * T_BK * 2;   // 16 KB
constexpr uint32_t T_B_BYTES = T_BN * T_BK * 2;   // 32 KB

struct TcParams {
  int64_t Q, N;
  int k_chunks;            // ceil(D / 64)
  int64_t m_tiles, n_tiles;
  int splits;
  int64_t tiles_per_split;
  const uint8_t* q_fold;
  const uint8_t* db_fold;  // padded to n_tiles * 256 bytes
  int fold_sorted;         // both fold vectors are non-decreasing: single-fold tiles of the query's own fold are skipped
  int64_t idx_base;
  int K;
  uint64_t* keys_out;      // [splits][Q][K]
  uint32_t* tau;           // [Q] order-preserving image of a lower bound of the query's global KCAP-th best score
  float* debug_scores;     // optional [Q][N] dump of every score (bring-up / tests)
  // ---- CTA-pair kernel: unit order and database-stream sharing (topk_tc2.cu) ----
  int64_t mg;              // query tiles per group: units are ordered (group, split, tile-in-group); mg >= m_tiles = one group
  int sync_tiles;          // cohort pacing: the pairs that stream the same database split meet every sync_tiles tiles; 0 = off
  int sync_points;         // ceil(tiles_per_split / sync_tiles)
  int sync_budget;         // SM cycles a pair waits at a meeting point at most (pacing only, never required for correctness)
  uint32_t* sync_ctr;      // [cohort slots][sync_points], zeroed per launch
  unsigned long long* unit_clock;  // optional [n_units][2] globaltimer at unit start / end (diagnostics)
  // ---- range epilogue (scan_tile RANGE mode, emr2a_range_search) ----
  float range_t;                   // min_score t; the cut is t - E, rounded down (range_cut)
  int D;
  const float* q_stats;            // K1 stats of both sides: the query side's batch maxima clamp every query
  const float* db_stats;
  ulonglong2* range_out;           // [range_cap] (query, packed key) of every pair with s~ >= cut
  int64_t range_cap;
  unsigned long long* range_count; // pairs found (keeps counting past range_cap)
  // ---- self-join (RANGE mode, emr2a_self_join): one row set, only the pairs i < j of global row numbers ----
  int self_join;                   // 1: tri_skipped tiles are not computed, j <= i is masked on the diagonal tiles
  int64_t q_row0;                  // global row number of query row 0 (added to the query field of every candidate)
  int64_t db_row0;                 // global row number of database row 0
};

// ---- PTX wrappers -------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}\n" : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);          // start address
  d |= static_cast<uint64_t>(0) << 16;                              // leading byte offset (unused for swizzled K-major)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;                      // stride byte offset: 8 rows * 128 B
  d |= static_cast<uint64_t>(1) << 46;                              // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                              // SWIZZLE_128B
  return d;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// instruction descriptor: D=F32, A=B=BF16, both K-major, N=256, M=128
constexpr uint32_t T_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((T_BN >> 3) << 17) | ((T_BM >> 4) << 24);

// ---- register-resident sorted Top-K list ------------------------------------------------
template <int KCAP>
struct RegTopK {
  float s[KCAP];
  uint32_t i[KCAP];
  __device__ __forceinline__ void reset() {
#pragma unroll
    for (int j = 0; j < KCAP; ++j) { s[j] = -INFINITY; i[j] = 0xFFFFFFFFu; }
  }
  __device__ __forceinline__ float threshold() const { return s[KCAP - 1]; }
  // candidates reach a thread in ascending index order, so strict '>' keeps the lower index on ties
  __device__ __forceinline__ void insert(float c, uint32_t ci) {
#pragma unroll
    for (int j = KCAP - 1; j > 0; --j) {
      const bool up = c > s[j - 1];
      const bool here = !up && (c > s[j]);
      s[j] = up ? s[j - 1] : (here ? c : s[j]);
      i[j] = up ? i[j - 1] : (here ? ci : i[j]);
    }
    const bool top = c > s[0];
    s[0] = top ? c : s[0];
    i[0] = top ? ci : i[0];
  }
};

__device__ __forceinline__ float select32(const float (&v)[32], int idx) {
  // 5-level select tree on the bits of idx (keeps v[] in registers)
  float a[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) a[j] = (idx & 1) ? v[2 * j + 1] : v[2 * j];
  float b[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) b[j] = (idx & 2) ? a[2 * j + 1] : a[2 * j];
  float c[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) c[j] = (idx & 4) ? b[2 * j + 1] : b[2 * j];
  const float d0 = (idx & 8) ? c[1] : c[0];
  const float d1 = (idx & 8) ? c[3] : c[2];
  return (idx & 16) ? d1 : d0;
}

// CV rule at tile granularity (fold-sorted inputs): if every query of the tile is in fold f and every
// database row of the tile is in fold f, all 128 x 256 pairs are inadmissible -- no TMA, no MMA, no epilogue.
// The three warp roles evaluate the same predicate from the same global bytes.
__device__ __forceinline__ int unit_fold(const TcParams& p, int64_t mt, int bm = T_BM) {
  if (!p.fold_sorted || p.q_fold == nullptr) return -1;
  const int64_t a = mt * bm, b = (a + bm - 1 < p.Q) ? a + bm - 1 : p.Q - 1;
  const int lo = __ldg(p.q_fold + a), hi = __ldg(p.q_fold + b);
  return lo == hi ? lo : -1;
}
__device__ __forceinline__ bool tile_skipped(const TcParams& p, int ufold, int64_t t) {
  if (ufold < 0) return false;
  const int64_t a = t * T_BN, b = (a + T_BN - 1 < p.N) ? a + T_BN - 1 : p.N - 1;
  return __ldg(p.db_fold + a) == ufold && __ldg(p.db_fold + b) == ufold;
}

// Self-join rule at tile granularity: when the last global row of database tile t is <= the first global row of the
// unit's query tile (bm rows), every pair of the tile has j <= i -- no TMA, no MMA, no epilogue.  Evaluated by the three
// warp roles like tile_skipped; always false outside the range epilogue.
template <bool RANGE>
__device__ __forceinline__ bool tri_skipped(const TcParams& p, int64_t mt, int bm, int64_t t) {
  if constexpr (!RANGE) {
    return false;
  } else {
    if (!p.self_join) return false;
    const int64_t last = (t * T_BN + T_BN - 1 < p.N) ? t * T_BN + T_BN - 1 : p.N - 1;
    return p.db_row0 + last <= p.q_row0 + mt * bm;
  }
}

// Cut of the range epilogue: every pair with exact score s >= t has s~ >= s - E >= t - E, so emitting s~ >= cut with
// cut <= t - E (subtraction rounded down) misses none of them.  E is error_bound with the query side's batch maxima.
// The cut is clamped to -FLT_MAX: t - E rounds to -inf for t near -FLT_MAX (or an infinite E), and -inf is what the
// epilogue writes for the columns past N and for fold-masked pairs -- those must never pass the inclusive compare.
// -FLT_MAX is still a lower bound of every finite score.
__device__ __forceinline__ float range_cut(const TcParams& p) {
  return fmaxf(__fsub_rd(p.range_t, error_bound(__ldg(p.q_stats), __ldg(p.q_stats + 1), p.db_stats, p.D)), -3.402823466e38f);
}

// Range epilogue of one 32-column chunk: the thread emits every score of its query row with s~ >= cut.  One atomicAdd
// per warp and chunk, only when the chunk has candidates; a lane's slots follow from the warp prefix sum of the
// per-lane counts.  Past range_cap the counter keeps counting and nothing is written.
__device__ __forceinline__ void range_emit(const TcParams& p, const float (&v)[32], const float cut, const int64_t c0,
                                           const int64_t q) {
  uint32_t mask = 0u;
  if (q < p.Q) {
#pragma unroll
    for (int c = 0; c < 32; ++c) mask |= (v[c] >= cut) ? (1u << c) : 0u;
  }
  if (!__any_sync(0xffffffffu, mask != 0u)) return;
  const int lane = threadIdx.x & 31;
  const int n = __popc(mask);
  int incl = n;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int total = __shfl_sync(0xffffffffu, incl, 31);
  unsigned long long base = 0ull;
  if (lane == 0) base = atomicAdd(p.range_count, static_cast<unsigned long long>(total));
  base = __shfl_sync(0xffffffffu, base, 0);
  unsigned long long pos = base + static_cast<unsigned long long>(incl - n);
  while (mask) {
    const int c = __ffs(mask) - 1;
    mask &= mask - 1u;
    if (pos < static_cast<unsigned long long>(p.range_cap))
      p.range_out[pos] = make_ulonglong2(static_cast<unsigned long long>(q + p.q_row0),
                                         pack_key(select32(v, c), static_cast<uint32_t>(c0 + c + p.idx_base)));
    ++pos;
  }
}

// Epilogue of one 128 x 256 accumulator tile for the thread's own query row: compare-mostly scan of
// the 256 scores in 8 chunks of 32 TMEM columns, rare sorted insertion into the register list.
// RANGE: no list; thr is the fixed cut of range_cut and every score >= thr is emitted (range_emit); in a self-join the
// scores with j <= i are set to -inf first.
//   taddr = TMEM address of (this warp's lane quarter, first column of the accumulator)
template <int KCAP, bool HAS_FOLD, bool RANGE = false>
__device__ __forceinline__ void scan_tile(const TcParams& p, RegTopK<KCAP>& top, float& thr, const float thr0,
                                          const uint32_t taddr, const int64_t n0, const uint32_t my_fold,
                                          const int64_t q) {
  const bool edge = (n0 + T_BN > p.N);
  // Fold-sorted rows: a tile whose first and last row share a fold holds that fold only.  Then the
  // per-element mask is unnecessary: either every row of the tile is inadmissible for this thread's
  // query (nothing to scan, but the warp still runs the collective TMEM loads) or none is.
  bool mask_rows = HAS_FOLD, all_masked = false;
  if (HAS_FOLD && p.fold_sorted) {
    const int64_t last = (n0 + T_BN - 1 < p.N) ? n0 + T_BN - 1 : p.N - 1;
    const uint32_t f_lo = __ldg(p.db_fold + n0), f_hi = __ldg(p.db_fold + last);
    if (f_lo == f_hi) { mask_rows = false; all_masked = (f_lo == my_fold); }
  }
#pragma unroll 1
  for (int ch = 0; ch < T_BN / 32; ++ch) {
    float v[32];
    tmem_ld32(taddr + static_cast<uint32_t>(ch * 32), v);
    const int64_t c0 = n0 + ch * 32;
    if (p.debug_scores && q < p.Q) {
#pragma unroll
      for (int c = 0; c < 32; ++c) if (c0 + c < p.N) p.debug_scores[q * p.N + c0 + c] = v[c];
    }
    if (edge) {                                   // columns past the last database row
#pragma unroll
      for (int c = 0; c < 32; ++c) if (c0 + c >= p.N) v[c] = -INFINITY;
    }
    if (HAS_FOLD && all_masked) {
#pragma unroll
      for (int c = 0; c < 32; ++c) v[c] = -INFINITY;
    }
    if (HAS_FOLD && mask_rows) {                  // CV rule: rows of the query's own fold are inadmissible
      const uint4* fp = reinterpret_cast<const uint4*>(p.db_fold + c0);
      const uint4 f0 = __ldg(fp), f1 = __ldg(fp + 1);
      const uint32_t w[8] = {f0.x, f0.y, f0.z, f0.w, f1.x, f1.y, f1.z, f1.w};
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const uint32_t f = (w[c >> 2] >> (8 * (c & 3))) & 0xFFu;
        v[c] = (f == my_fold) ? -INFINITY : v[c];
      }
    }
    if constexpr (RANGE) {
      if (p.self_join) {                          // diagonal tiles: a row is never paired with itself or an earlier row
        const int64_t lim = p.q_row0 + q - p.db_row0 - c0;      // columns c <= lim of this chunk hold j <= i
        if (lim >= 0) {
#pragma unroll
          for (int c = 0; c < 32; ++c) v[c] = (c <= lim) ? -INFINITY : v[c];
        }
      }
      range_emit(p, v, thr, c0, q);
    } else {
      float mx = v[0];
#pragma unroll
      for (int c = 1; c < 32; ++c) mx = fmaxf(mx, v[c]);
      if (mx > thr) {                             // rare: at least one score beats the current threshold
        uint32_t mask = 0u;
#pragma unroll
        for (int c = 0; c < 32; ++c) mask |= (v[c] > thr) ? (1u << c) : 0u;
        while (mask) {
          const int c = __ffs(mask) - 1;
          mask &= mask - 1u;
          const float val = select32(v, c);
          if (val > thr) {
            top.insert(val, static_cast<uint32_t>(c0 + c + p.idx_base));
            thr = fmaxf(top.threshold(), thr0);
          }
        }
      }
    }
    __syncwarp();                                 // tcgen05.ld is warp-collective: reconverge before the next chunk
  }
}

// ---- unit order of the CTA-pair kernel ----------------------------------------------------
// A work unit is (query tile mt, database split).  Units are numbered group by group: a group is p.mg consecutive
// query tiles; inside a group the split is the slow index, so the mg units of one (group, split) -- a COHORT: they
// stream the same database tiles -- carry consecutive numbers and run concurrently on consecutive pairs.
//   * mg bounds the query-plane working set of the concurrent pairs (mg tiles x 256 rows x ld x 2 B) so that it
//     stays in L2 next to the database stream (D = 5120: a 10k-query plane is 102 MB -- ncu r2: 651 GB of DRAM reads
//     per launch for a 20 GB plane before grouping);
//   * cohort members pace each other (cohort_sync) so the stream is fetched from HBM once per cohort, not once per pair.
__device__ __forceinline__ void unit_coords(const TcParams& p, int64_t u, int64_t& split, int64_t& mt) {
  const int64_t per_group = p.mg * p.splits;
  const int64_t g = u / per_group;
  const int64_t r = u - g * per_group;
  const int64_t left = p.m_tiles - g * p.mg;
  const int64_t mg_eff = left < p.mg ? left : p.mg;
  split = r / mg_eff;
  mt = g * p.mg + (r - split * mg_eff);
}
// Cohort part of unit u among the units [step * n_workers, (step + 1) * n_workers) that run concurrently:
// slot = unique id of (cohort, step), size = members of the cohort inside this step.
__device__ __forceinline__ void unit_cohort(const TcParams& p, int64_t u, int64_t n_workers, int64_t n_units,
                                            int64_t& slot, int& size) {
  const int64_t per_group = p.mg * p.splits;
  const int64_t g = u / per_group;
  const int64_t r = u - g * per_group;
  const int64_t left = p.m_tiles - g * p.mg;
  const int64_t mg_eff = left < p.mg ? left : p.mg;
  const int64_t split = r / mg_eff;
  int64_t c0 = g * per_group + split * mg_eff, c1 = c0 + mg_eff;          // the cohort's units [c0, c1)
  const int64_t step = u / n_workers;
  const int64_t s0 = step * n_workers, s1 = (s0 + n_workers < n_units) ? s0 + n_workers : n_units;
  c0 = c0 > s0 ? c0 : s0;
  c1 = c1 < s1 ? c1 : s1;
  size = static_cast<int>(c1 - c0);
  slot = g * p.splits + split + step;                                     // strictly increasing over the parts
}
// Meeting point of a cohort (called by ONE thread of the pair).  Pure pacing: a pair that arrives early waits --
// at most p.sync_budget cycles -- until the others have arrived, so that all members request a database tile
// while it is in L2.  Nothing depends on the wait being complete.
__device__ __forceinline__ void cohort_sync(const TcParams& p, int64_t slot, int point, int size) {
  uint32_t* ctr = p.sync_ctr + slot * p.sync_points + point;
  const uint32_t seen = atomicAdd(ctr, 1u) + 1u;
  if (seen >= static_cast<uint32_t>(size)) return;
  const long long t0 = clock64();
  while (__ldcg(ctr) < static_cast<uint32_t>(size)) {
    if (clock64() - t0 > p.sync_budget) break;
    __nanosleep(40);
  }
}

// Start threshold of a work unit from the shared per-query bound tau[q]: units of the same query tile that
// finished earlier published their KCAP-th best score; the global KCAP-th best is at least that, so rows
// strictly below it can be skipped without changing the merged list (">= bound" is kept, hence one ulp down).
__device__ __forceinline__ float unit_start_threshold(const TcParams& p, int64_t q) {
  if (p.tau == nullptr || q >= p.Q) return -INFINITY;
  const uint32_t t = __ldcg(p.tau + q);
  if (t == 0u) return -INFINITY;
  const float b = unorder_f32(t);
  const uint32_t bits = __float_as_uint(b);
  if (b > 0.f) return __uint_as_float(bits - 1u);
  if (b < 0.f) return __uint_as_float(bits + 1u);
  return -1e-45f;                                 // just below zero
}

// ---- host: the instantiations of both kernels ------------------------------------------------------------------------
// Every instantiation of tc_topk_kernel and tc2_topk_kernel has this type.
typedef void (*TcKernel)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, TcParams);

// The instantiations that exist, the same for both kernels: Top-K with passes {1, 3} x register list {8, 16, 32}, and
// the range epilogue with 1 pass (its register list is unused: KCAP 8); each with and without folds.
// K<PASSES, KCAP, RANGE>::get(fold) names one of them.  Any other combination gets null.
template <template <int, int, bool> class K>
static TcKernel tc_pick(int passes, int kcap, bool fold, bool range) {
  if (range) return passes == 1 && kcap == 8 ? K<1, 8, true>::get(fold) : nullptr;
  if (passes == 1)
    return kcap == 8 ? K<1, 8, false>::get(fold) : kcap == 16 ? K<1, 16, false>::get(fold) : kcap == 32 ? K<1, 32, false>::get(fold) : nullptr;
  if (passes == 3)
    return kcap == 8 ? K<3, 8, false>::get(fold) : kcap == 16 ? K<3, 16, false>::get(fold) : kcap == 32 ? K<3, 32, false>::get(fold) : nullptr;
  return nullptr;
}

}  // namespace emr2a
