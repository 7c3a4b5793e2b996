// EMR2A_PREC_BF16_RESCORE: exact re-scoring of the candidates the 1-pass tensor-core filter kept,
// verified selection, and an exact re-scan for the (rare) queries the bound cannot verify.
//
// Filter:   s~(q,d) = <bf16(q), bf16(d)> accumulated in fp32 on the tensor cores; per query the KP = 32
//           rows with the largest s~ are kept (K <= 10: the slack below the K-th best must hold ~2E of scores).
// Rescore:  s(q,d) = fp32 dot product of the fp32 rows K1 wrote (the same values the fp32 arm uses).
// Bound:    |s~ - s| <= E = r_q * n_d + (n_q + r_q) * r_d + (1.02 D + 8) * 2^-23 * (n_q + r_q) * (n_d + r_d)
//           for every pair, where n_d, r_d = max row norm and max ||row - bf16(row)|| over the database rows (K1
//           `stats`), n_q, r_q = the same two norms of THIS query (computed here, clamped by the batch maxima of K1
//           `stats`).  The first two terms are Cauchy-Schwarz on the two quantisation residuals (bf16 keeps 8
//           significant bits, so r ~ 1.7e-3 for a unit row and E ~ 4e-3).  The last term covers the arithmetic:
//             * tensor core: the D products of bf16 values are exact; they are summed in groups of 16 (UMMA_K) and
//               added to the fp32 accumulator in TMEM.  Model: every one of the D additions loses at most one unit
//               in the last place of a 24-bit significand aligned to the largest magnitude involved (truncation,
//               no guard bits -- the worst any fp32-accumulating tensor pipe documents), and all partial sums are
//               bounded by sum |x_i y_i| <= ||bf16(q)|| ||bf16(d)|| <= (n_q + r_q)(n_d + r_d):  D * 2^-23 * that;
//             * the fp32 re-scoring the comparison is made against: D/32 round-to-nearest FMAs per lane plus the
//               shuffle tree, <= (D/32 + 6) * 2^-24 * n_q n_d  (inside the 0.02 D + 8).
//           D = 1024: 1.3e-4, D = 5120: 6.2e-4 per unit norms -- 3 % / 15 % on top of the quantisation terms.
//           Measured tensor-core error on bf16-exact operands (tests/test_gpu_rescore_bound.py, D = 5120): up to
//           1.4e-5 * n_q n_d when all products have one sign (the accumulator truncates) -- above the constant
//           1e-5 the first version of this bound used, 45x below this term.
// Verify:   every row outside the candidate list has s~ <= tau (the KP-th approximate score), hence
//           s <= tau + E.  If the exact K-th best candidate score exceeds tau + E strictly, no
//           outside row can enter the Top-K and the selection is exact.  Otherwise the query is
//           appended to a flag list and re-searched exactly against the whole database
//           (exact_rescan_kernel, cost proportional to the number of flagged queries).
// Roofline: HBM-bound gather: Q * KP * D * 4 bytes (C2: 1.3 GB, ~0.3 ms).
#include <stdlib.h>
#include "row_math.cuh"

namespace emr2a {

struct RescoreParams {
  const uint64_t* approx;   // [Q][KP] approximate keys, best first (KP = 32 or 64)
  int KP;
  const uint32_t* tau;      // [Q] bound (order-preserving image) on the filter score of rows outside the per-split lists; may be null
  const float* q; int64_t ldq;
  const float* db; int64_t lddb;
  int64_t Q, N;
  int D;
  int64_t idx_base;
  int K;
  const float* q_stats;
  const float* db_stats;
  uint64_t* out;            // [Q][K]
  int* status;              // [0] = #unverified queries, [1] = flag list overflow
  int* flag_list;
  int cap;
  uint8_t* qflags;          // optional [Q]: 1 = selection not verified by the bound (valid even when the list overflows)
  // cooperative shards (emr2a_rescore_select): the verification is made by the caller on the merged lists
  const float* kth_floor;   // optional [Q]: lower bound of the GLOBAL K-th best filter score (max over the shards' local K-th)
  float* bound_out;         // optional [Q]: upper bound of the exact score of every row of THIS shard that was not re-scored
                            //               because it is not a candidate (tau + E); -inf if there is no such row
  // exact re-scan
  const uint8_t* q_fold;
  const uint8_t* db_fold;
  uint64_t* fb_parts;       // [blocks][cap][K]
  LazyRows lazy;            // SRC != 0: the database rows are re-created from the raw rows (row_math.cuh), db is unused
  int n_fixed;              // >= 0: the flag list holds exactly this many queries (emr2a_exact_rescan); < 0: status[0]
  int compact;              // != 0: the re-scan writes list i of the flag list to out[i][K] instead of out[flag_list[i]][K]
  // filtered re-scan (filtered_rescan_kernel): stream the bf16 plane, score exactly only what can reach the Top-K
  const uint16_t* db_hi;    // [N][lddb_hi] bf16 plane of the database (K1), zero padded; null = unfiltered re-scan
  int64_t lddb_hi;
  const uint64_t* seed;     // optional exact keys whose K-th best seeds the cut: [Q][K] (by query) or [n_flagged][K] (seed_compact)
  int seed_compact;
};

__device__ __forceinline__ int flagged_count(const RescoreParams& p) {
  int n = p.n_fixed >= 0 ? p.n_fixed : p.status[0];
  return n > p.cap ? p.cap : n;
}

// SRC: where the fp32 database rows come from.  0 = the fp32 matrix K1 wrote; 1 / 2 = re-created from the raw fp32 /
// bf16 rows with the divisors K1 recorded (deferred fp32 rows: same values bit for bit, no fp32 copy of the database).
template <int SRC> struct RawOf { typedef float T; };
template <> struct RawOf<2> { typedef __nv_bfloat16 T; };

// The query side of the bound is taken per query: ||q|| and ||q - bf16(q)|| of THIS query's fp32 row (the hi plane
// the filter used is bf16_rn of exactly these values), clamped by the batch maxima K1 wrote.  Batches whose query
// norms differ (late fusion with per-query z-score / min-max scaling, emr2a_b200/late.py) get a bound as tight as a
// homogeneous batch would.
template <bool VEC>
__device__ __forceinline__ void query_norms(const float* __restrict__ qrow, int D, int lane, const float* qs,
                                            float& nq, float& rq) {
  float n2 = 0.f, r2 = 0.f;
  if (VEC) {                                 // 128-bit loads, four of them in flight: the pass is pure load latency
#pragma unroll 4
    for (int e = lane * 4; e < D; e += 128) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(qrow + e));
      const float v[4] = {x.x, x.y, x.z, x.w};
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float r = v[c] - __bfloat162float(__float2bfloat16_rn(v[c]));
        n2 = fmaf(v[c], v[c], n2);
        r2 = fmaf(r, r, r2);
      }
    }
  } else {
#pragma unroll 4
    for (int e = lane; e < D; e += 32) {
      const float x = __ldg(qrow + e);
      const float r = x - __bfloat162float(__float2bfloat16_rn(x));
      n2 = fmaf(x, x, n2);
      r2 = fmaf(r, r, r2);
    }
  }
  n2 = warp_sum(n2);
  r2 = warp_sum(r2);
  nq = fminf(sqrtf(n2) * 1.000002f, qs[0]);          // rounded up: the bound must stay an upper bound
  rq = fminf(sqrtf(r2) * 1.000002f, qs[1]);
}

// WPQ = warps per query.  1: a warp owns a query (throughput layout, 8 queries per block).  8: a BLOCK owns a query
// and its 8 warps re-score 8 of the 64 candidates each -- for small batches (serving), where a single warp walking
// 16 groups of dependent row gathers is pure latency (~90 us at D = 1024); selection and verification are then done
// by warp 0 from the exact keys the warps exchanged through shared memory.
template <bool VEC, int WPQ, int SRC = 0>
__global__ void __launch_bounds__(256, WPQ == 1 ? (SRC == 0 ? 4 : 2) : 1) rescore_select_kernel(const RescoreParams p) {
  static_assert(SRC == 0 || VEC, "deferred fp32 rows need the 128-bit path");
  __shared__ uint64_t xkeys[WPQ == 1 ? 1 : 64];
  const int lane = threadIdx.x & 31;
  const int wq = WPQ == 1 ? 0 : (threadIdx.x >> 5);                      // this warp's share of the candidate groups
  const int64_t q = WPQ == 1 ? (static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5
                             : static_cast<int64_t>(blockIdx.x);
  if (q >= p.Q) return;
  if (WPQ > 1) {
    if (threadIdx.x < 64) xkeys[threadIdx.x] = 0ull;
    __syncthreads();
  }
  // lane holds candidates lane and lane + 32
  uint64_t akey[2], ekey[2] = {0ull, 0ull};
  akey[0] = lane < p.KP ? p.approx[q * p.KP + lane] : 0ull;
  akey[1] = lane + 32 < p.KP ? p.approx[q * p.KP + lane + 32] : 0ull;
  const uint64_t last = __shfl_sync(0xffffffffu, p.KP > 32 ? akey[1] : akey[0], (p.KP - 1) & 31);
  const float* qrow = p.q + q * p.ldq;
  // A candidate c with s~(c) + E < s~(K-th candidate) - E cannot be among the exact K best (the K best
  // filter scores all have exact scores >= s~_K - E), so it is not re-scored: typically ~20 of 64 are.
  float nq, rq;
  query_norms<VEC>(qrow, p.D, lane, p.q_stats, nq, rq);
  const float E = error_bound(nq, rq, p.db_stats, p.D);
  const uint64_t kth_approx = __shfl_sync(0xffffffffu, akey[0], p.K - 1);
  float kth_lb = kth_approx != 0ull ? key_score(kth_approx) : -INFINITY;
  if (p.kth_floor != nullptr) kth_lb = fmaxf(kth_lb, __ldg(p.kth_floor + q));      // another shard already holds K better rows
  float cut = kth_lb - 2.0f * E;
  bool done = false, tightened = false;
  // deferred fp32 rows: every lane fetches the recorded divisors of ITS candidates now (all gathers in flight at once);
  // the groups below pick them up with shuffles instead of paying a dependent 16-byte gather per group
  float4 rdiv[SRC == 0 ? 1 : 2];
  if (SRC != 0) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      rdiv[SRC == 0 ? 0 : h] = make_float4(1.f, 1.f, 1.f, 0.f);
      if (akey[h] != 0ull && key_score(akey[h]) >= cut)
        rdiv[SRC == 0 ? 0 : h] = __ldg(reinterpret_cast<const float4*>(p.lazy.row_div) +
                                       (static_cast<int64_t>(key_index(akey[h])) - p.idx_base));
    }
  }
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    for (int g = 0; g < 32 && !done && h * 32 + g < p.KP; g += 4) {
      uint64_t kk[4];
      float acc[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        kk[c] = __shfl_sync(0xffffffffu, akey[h], g + c);
        if (kk[c] != 0ull && key_score(kk[c]) < cut) kk[c] = 0ull;      // sorted by s~: everything after is below too
        acc[c] = 0.f;
      }
      if (kk[0] == 0ull) { done = true; break; }      // lists are packed: nothing valid beyond the first empty slot
      if (WPQ > 1 && (((h * 32 + g) >> 2) % WPQ) != wq) continue;      // another warp of the block takes this group
      if (VEC) {
        LazyRowCtx ctx[SRC == 0 ? 1 : 4];
        if (SRC != 0) {
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            float4 d;
            d.x = __shfl_sync(0xffffffffu, rdiv[SRC == 0 ? 0 : h].x, g + c);
            d.y = __shfl_sync(0xffffffffu, rdiv[SRC == 0 ? 0 : h].y, g + c);
            d.z = __shfl_sync(0xffffffffu, rdiv[SRC == 0 ? 0 : h].z, g + c);
            d.w = __shfl_sync(0xffffffffu, rdiv[SRC == 0 ? 0 : h].w, g + c);
            ctx[SRC == 0 ? 0 : c] = lazy_ctx_from(p.lazy, d);
          }
        }
#pragma unroll 2
        for (int e = lane * 4; e < p.D; e += 128) {
          const float4 x = __ldg(reinterpret_cast<const float4*>(qrow + e));
          typedef typename RawChunk<typename RawOf<SRC>::T>::T Raw;
          Raw raw[SRC == 0 ? 1 : 4];
          if (SRC != 0) {                      // all four gathers first, then the arithmetic
#pragma unroll
            for (int c = 0; c < 4; ++c)
              if (kk[c] != 0ull)
                raw[SRC == 0 ? 0 : c] = lazy_raw4<typename RawOf<SRC>::T>(p.lazy, static_cast<int64_t>(key_index(kk[c])) - p.idx_base, e);
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            if (kk[c] != 0ull) {
              const int64_t row = static_cast<int64_t>(key_index(kk[c])) - p.idx_base;
              const float4 y = SRC == 0 ? __ldg(reinterpret_cast<const float4*>(p.db + row * p.lddb + e))
                                        : lazy_apply4<typename RawOf<SRC>::T>(p.lazy, ctx[SRC == 0 ? 0 : c], raw[SRC == 0 ? 0 : c], e);
              acc[c] = fmaf(x.x, y.x, acc[c]); acc[c] = fmaf(x.y, y.y, acc[c]);
              acc[c] = fmaf(x.z, y.z, acc[c]); acc[c] = fmaf(x.w, y.w, acc[c]);
            }
          }
        }
      } else {
        for (int e = lane; e < p.D; e += 32) {
          const float x = __ldg(qrow + e);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            if (kk[c] != 0ull) {
              const int64_t row = static_cast<int64_t>(key_index(kk[c])) - p.idx_base;
              acc[c] = fmaf(x, __ldg(p.db + row * p.lddb + e), acc[c]);
            }
          }
        }
      }
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float s = warp_sum(acc[c]);
        if (lane == g + c && kk[c] != 0ull) ekey[h] = pack_key(s, key_index(kk[c]));
      }
      // Once the K + 2 .. K + 5 best filter candidates have their exact scores, the K-th best of THOSE (<= the final
      // exact K-th best) tightens the cut: a candidate with s~ + E below it has s <= s~ + E < that K-th best and cannot
      // enter the Top-K.  This replaces the a-priori margin 2E by E for the rest of the list -- about a third fewer
      // row gathers (the scores within 2E of the K-th best are as many again as the Top-K itself).
      if (WPQ == 1 && h == 0 && !tightened && g + 4 >= p.K + 2) {
        float v = ekey[0] != 0ull ? key_score(ekey[0]) : -INFINITY;
#pragma unroll
        for (int k2 = 2; k2 <= 32; k2 <<= 1) {                 // bitonic sort across the warp, descending
#pragma unroll
          for (int j = k2 >> 1; j > 0; j >>= 1) {
            const float o = __shfl_xor_sync(0xffffffffu, v, j);
            const bool take_max = ((lane & j) == 0) == ((lane & k2) == 0);
            v = take_max ? fmaxf(v, o) : fminf(v, o);
          }
        }
        const float kth_exact = __shfl_sync(0xffffffffu, v, p.K - 1);
        cut = fmaxf(cut, kth_exact - E);
        tightened = true;
      }
    }
  }
  if (WPQ > 1) {                                     // gather the block's exact keys in warp 0
    if (ekey[0] != 0ull) xkeys[lane] = ekey[0];
    if (ekey[1] != 0ull) xkeys[32 + lane] = ekey[1];
    __syncthreads();
    if (wq != 0) return;
    ekey[0] = xkeys[lane];
    ekey[1] = xkeys[32 + lane];
  }
  // exact Top-K of the candidates
  uint64_t mine = 0ull;
  for (int r = 0; r < p.K; ++r) {
    const uint64_t loc = ekey[0] > ekey[1] ? ekey[0] : ekey[1];
    const uint64_t best = warp_max_u64(loc);
    if (best != 0ull) {
      if (ekey[0] == best) ekey[0] = 0ull;
      if (ekey[1] == best) ekey[1] = 0ull;
    }
    if (lane == r) mine = best;
  }
  if (lane < p.K) p.out[q * p.K + lane] = mine;
  // Verification.  Rows that are not candidates have a filter score <= tau:
  //   - rows a split kept but the merge dropped:            <= the last merged candidate's score
  //   - rows a split did not keep (its list was full, or the shared threshold pruned them):
  //                                                          <= p.tau[q] = max over the full lists of their last score
  float tau = -INFINITY;
  bool bounded = false;
  if (last != 0ull) { tau = key_score(last); bounded = true; }
  if (p.tau != nullptr) {
    const uint32_t t = __ldcg(p.tau + q);
    if (t != 0u) { tau = fmaxf(tau, unorder_f32(t)); bounded = true; }
  }
  if (p.bound_out != nullptr) {               // cooperative shards: publish the bound, the caller verifies globally
    if (lane == 0) p.bound_out[q] = bounded ? tau + E : -INFINITY;
    return;
  }
  bool ok = true;
  if (bounded) {
    const uint64_t kth = __shfl_sync(0xffffffffu, mine, p.K - 1);
    ok = kth != 0ull && key_score(kth) > tau + E;
    if (!ok && lane == 0) {
      const int i = atomicAdd(&p.status[0], 1);
      if (i < p.cap) p.flag_list[i] = static_cast<int>(q); else p.status[1] = 1;
    }
  }
  if (p.qflags != nullptr && lane == 0) p.qflags[q] = ok ? 0 : 1;
}

// Exact re-search of the flagged queries against every database row (fp32, CUDA cores).  A block
// owns a contiguous row range and walks the flagged queries in groups held in shared memory; each
// warp keeps one sorted list per query of the group.
constexpr int FB_WARPS = 8;      // warps per block; wide rows (the query group would not fit beside a second block) take 16
constexpr int FB_GMAX = 8;
constexpr int FB_ROWS = 4;     // database rows a warp scores per pass over the query group

// NW = warps per block.  8 (two blocks per SM) while a group of 8 queries fits in 96 KB of shared memory; wider rows
// (D = 5120: 20 KB per query) run ONE block of 16 warps per SM with up to 200 KB, so that a pass over the database still
// serves 8 queries -- the passes, not the queries, are what the re-scan costs.
template <bool VEC, int SRC = 0, int NW = FB_WARPS>
__global__ void __launch_bounds__(NW * 32, NW == FB_WARPS ? 2 : 1) exact_rescan_kernel(const RescoreParams p, int G) {
  static_assert(SRC == 0 || VEC, "deferred fp32 rows need the 128-bit path");
  extern __shared__ __align__(16) unsigned char fb_smem[];
  const int n = flagged_count(p);
  if (n <= 0) return;
  float* qbuf = reinterpret_cast<float*>(fb_smem);                                   // [G][Dp]
  const int Dp = (p.D + 3) & ~3;
  uint64_t* lists = reinterpret_cast<uint64_t*>(fb_smem + sizeof(float) * G * Dp);   // [NW][G][K]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K = p.K;
  const int64_t per = (p.N + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * per;
  const int64_t r1 = (r0 + per < p.N) ? r0 + per : p.N;

  for (int g0 = 0; g0 < n; g0 += G) {
    const int gc = (n - g0 < G) ? (n - g0) : G;
    __syncthreads();
    for (int e = threadIdx.x; e < gc * Dp; e += blockDim.x) {
      const int g = e / Dp, c = e - g * Dp;
      qbuf[e] = c < p.D ? p.q[static_cast<int64_t>(p.flag_list[g0 + g]) * p.ldq + c] : 0.f;
    }
    for (int e = threadIdx.x; e < NW * G * K; e += blockDim.x) lists[e] = 0ull;
    __syncthreads();
    uint64_t kth = 0ull;                             // lane g: K-th best of (this warp, query g)
    const int my_fold = (p.q_fold && lane < gc) ? p.q_fold[p.flag_list[g0 + lane]] : -1;
    // A warp walks FB_ROWS rows at a time.  Every row element is fetched (or re-created) ONCE and every query chunk read
    // from shared memory serves FB_ROWS rows: with one row per warp the kernel was bound by shared-memory bandwidth
    // (G query reads per row chunk: 0.9-1.4 TB/s of database stream), not by HBM.  Per (row, query) the fused
    // multiply-adds run in the order the re-scoring stage uses, so the scores of the two stages are equal bit for bit.
    for (int64_t rb = r0 + static_cast<int64_t>(warp) * FB_ROWS; rb < r1; rb += NW * FB_ROWS) {
      const int nr = (r1 - rb < FB_ROWS) ? static_cast<int>(r1 - rb) : FB_ROWS;
      float acc[FB_ROWS][FB_GMAX];
#pragma unroll
      for (int r = 0; r < FB_ROWS; ++r)
#pragma unroll
        for (int g = 0; g < FB_GMAX; ++g) acc[r][g] = 0.f;
      if (VEC) {
        typedef typename RawChunk<typename RawOf<SRC>::T>::T Raw;
        LazyRowCtx ctx[SRC == 0 ? 1 : FB_ROWS];
        if (SRC != 0) {
#pragma unroll
          for (int r = 0; r < FB_ROWS; ++r)
            if (r < nr) ctx[SRC == 0 ? 0 : r] = lazy_row_ctx(p.lazy, rb + r);
        }
#pragma unroll 2
        for (int c = lane * 4; c < p.D; c += 128) {
          Raw raw[FB_ROWS];
#pragma unroll
          for (int r = 0; r < FB_ROWS; ++r) {            // FB_ROWS independent 128-bit (fp32) / 64-bit (bf16) loads in flight
            if (r < nr) {
              if (SRC == 0) *reinterpret_cast<float4*>(&raw[r]) = __ldg(reinterpret_cast<const float4*>(p.db + (rb + r) * p.lddb + c));
              else raw[r] = lazy_raw4<typename RawOf<SRC>::T>(p.lazy, rb + r, c);
            }
          }
          float4 y[FB_ROWS];
#pragma unroll
          for (int r = 0; r < FB_ROWS; ++r) {
            if (r < nr) y[r] = SRC == 0 ? *reinterpret_cast<const float4*>(&raw[r])
                                        : lazy_apply4<typename RawOf<SRC>::T>(p.lazy, ctx[SRC == 0 ? 0 : r], raw[r], c);
            else y[r] = make_float4(0.f, 0.f, 0.f, 0.f);
          }
#pragma unroll
          for (int g = 0; g < FB_GMAX; ++g) {
            if (g < gc) {
              const float4 x = *reinterpret_cast<const float4*>(qbuf + g * Dp + c);
#pragma unroll
              for (int r = 0; r < FB_ROWS; ++r) {
                acc[r][g] = fmaf(x.x, y[r].x, acc[r][g]); acc[r][g] = fmaf(x.y, y[r].y, acc[r][g]);
                acc[r][g] = fmaf(x.z, y[r].z, acc[r][g]); acc[r][g] = fmaf(x.w, y[r].w, acc[r][g]);
              }
            }
          }
        }
      } else {
        for (int c = lane; c < p.D; c += 32) {
#pragma unroll
          for (int r = 0; r < FB_ROWS; ++r) {
            if (r < nr) {
              const float y = __ldg(p.db + (rb + r) * p.lddb + c);
#pragma unroll
              for (int g = 0; g < FB_GMAX; ++g)
                if (g < gc) acc[r][g] = fmaf(qbuf[g * Dp + c], y, acc[r][g]);
            }
          }
        }
      }
#pragma unroll
      for (int r = 0; r < FB_ROWS; ++r) {
        if (r >= nr) break;
        const int dfold = p.db_fold ? p.db_fold[rb + r] : -2;
#pragma unroll
        for (int g = 0; g < FB_GMAX; ++g) {
          if (g >= gc) break;
          const float s = warp_sum(acc[r][g]);
          if (lane == g && dfold != my_fold) {
            const uint64_t key = pack_key(s, static_cast<uint32_t>(rb + r + p.idx_base));
            if (key > kth) {
              uint64_t* mine = lists + (warp * G + g) * K;
              int pos = K - 1;
              while (pos > 0 && mine[pos - 1] < key) { mine[pos] = mine[pos - 1]; --pos; }
              mine[pos] = key;
              kth = mine[K - 1];
            }
          }
        }
      }
    }
    __syncthreads();
    // merge the NW lists of each query: warp w serves queries w, w + NW, ...
    for (int g = warp; g < gc; g += NW) {
      uint64_t bound = ~0ull;
      for (int rnk = 0; rnk < K; ++rnk) {
        uint64_t best = 0ull;
        for (int t = lane; t < NW * K; t += 32) {
          const int w = t / K, j = t - w * K;
          const uint64_t key = lists[(w * G + g) * K + j];
          if (key < bound && key > best) best = key;
        }
        best = warp_max_u64(best);
        bound = best;
        if (lane == 0) p.fb_parts[(static_cast<int64_t>(blockIdx.x) * p.cap + g0 + g) * K + rnk] = best;
        if (best == 0ull) {
          for (int r2 = rnk + 1 + lane; r2 < K; r2 += 32)
            p.fb_parts[(static_cast<int64_t>(blockIdx.x) * p.cap + g0 + g) * K + r2] = 0ull;
          break;
        }
      }
    }
  }
}

// Filtered exact re-scan.  The exact re-scan above reads the fp32 rows of the WHOLE database (or re-creates them) to
// find a handful of rows.  This one streams the bf16 plane instead -- half the bytes, no re-creation -- and computes
// the filter score s~' = <bf16(q), bf16(d)> on the CUDA cores (exact products, fp32 accumulation: within the same
// bound E of the exact score s as the tensor-core filter, error_bound()).  A row is scored exactly -- by the warp, in
// the arithmetic of the re-scoring stage, from the fp32 rows or the deferred rows -- only if s~' >= cut, where
// cut = (running K-th best EXACT score of this warp's list, or of the seed list) - E.  Any row that belongs to the
// final Top-K has s >= final K-th best >= running K-th best, hence s~' >= s - E >= cut: it is scored, so the lists
// are the exact Top-K.  After a short warm-up almost no row passes and the pass is an HBM stream of the plane.
constexpr int FR_ROWS = 4;

template <int SRC>
__global__ void __launch_bounds__(FB_WARPS * 32, 2) filtered_rescan_kernel(const RescoreParams p, int G) {
  extern __shared__ __align__(16) unsigned char fb_smem[];
  const int n = flagged_count(p);
  if (n <= 0) return;
  const int Dh = (p.D + 7) & ~7;                                                    // bf16 columns walked (plane is zero padded)
  uint16_t* qh = reinterpret_cast<uint16_t*>(fb_smem);                              // [G][Dh] bf16(q)
  uint64_t* lists = reinterpret_cast<uint64_t*>(fb_smem + ((sizeof(uint16_t) * G * Dh + 15) & ~static_cast<size_t>(15)));   // [FB_WARPS][G][K]
  __shared__ float e_of[FB_GMAX], seed_of[FB_GMAX];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int K = p.K;
  const int64_t per = (p.N + gridDim.x - 1) / gridDim.x;
  const int64_t r0 = static_cast<int64_t>(blockIdx.x) * per;
  const int64_t r1 = (r0 + per < p.N) ? r0 + per : p.N;

  for (int g0 = 0; g0 < n; g0 += G) {
    const int gc = (n - g0 < G) ? (n - g0) : G;
    __syncthreads();
    for (int e = threadIdx.x; e < gc * Dh; e += blockDim.x) {
      const int g = e / Dh, c = e - g * Dh;
      const float x = c < p.D ? p.q[static_cast<int64_t>(p.flag_list[g0 + g]) * p.ldq + c] : 0.f;
      qh[e] = __bfloat16_as_ushort(__float2bfloat16_rn(x));
    }
    for (int e = threadIdx.x; e < FB_WARPS * G * K; e += blockDim.x) lists[e] = 0ull;
    for (int g = warp; g < gc; g += FB_WARPS) {          // per query: the error bound and the seed of the cut
      const int64_t qd = p.flag_list[g0 + g];
      float nq, rq;
      query_norms<false>(p.q + qd * p.ldq, p.D, lane, p.q_stats, nq, rq);
      if (lane == 0) {
        e_of[g] = error_bound(nq, rq, p.db_stats, p.D);
        float sd = -INFINITY;
        if (p.seed != nullptr) {
          const uint64_t k = p.seed[(p.seed_compact ? static_cast<int64_t>(g0 + g) : qd) * K + K - 1];
          if (k != 0ull) sd = key_score(k);
        }
        seed_of[g] = sd;
      }
    }
    __syncthreads();
    uint64_t kth = 0ull;                                 // lane g: K-th best exact key of (this warp, query g)
    const int my_fold = (p.q_fold && lane < gc) ? p.q_fold[p.flag_list[g0 + lane]] : -1;
    const float my_e = lane < gc ? e_of[lane] : 0.f;
    float my_cut = lane < gc ? seed_of[lane] - my_e : INFINITY;        // lane g: rows of query g below this are skipped
    for (int64_t rb = r0 + static_cast<int64_t>(warp) * FR_ROWS; rb < r1; rb += FB_WARPS * FR_ROWS) {
      const int nr = (r1 - rb < FR_ROWS) ? static_cast<int>(r1 - rb) : FR_ROWS;
      float acc[FR_ROWS][FB_GMAX];
#pragma unroll
      for (int r = 0; r < FR_ROWS; ++r)
#pragma unroll
        for (int g = 0; g < FB_GMAX; ++g) acc[r][g] = 0.f;
      for (int c = lane * 8; c < Dh; c += 256) {
        float y[FR_ROWS][8];
#pragma unroll
        for (int r = 0; r < FR_ROWS; ++r) {
          uint4 raw = make_uint4(0u, 0u, 0u, 0u);
          if (r < nr) raw = __ldg(reinterpret_cast<const uint4*>(p.db_hi + (rb + r) * p.lddb_hi + c));
          const uint32_t w[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            y[r][2 * j] = __uint_as_float(w[j] << 16);
            y[r][2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
          }
        }
#pragma unroll
        for (int g = 0; g < FB_GMAX; ++g) {
          if (g < gc) {
            const uint4 qr = *reinterpret_cast<const uint4*>(qh + g * Dh + c);
            const uint32_t w[4] = {qr.x, qr.y, qr.z, qr.w};
            float x[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              x[2 * j] = __uint_as_float(w[j] << 16);
              x[2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
            }
#pragma unroll
            for (int r = 0; r < FR_ROWS; ++r)
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[r][g] = fmaf(x[j], y[r][j], acc[r][g]);
          }
        }
      }
#pragma unroll
      for (int r = 0; r < FR_ROWS; ++r) {
        if (r >= nr) break;
        const int64_t row = rb + r;
        const int dfold = p.db_fold ? p.db_fold[row] : -2;
#pragma unroll
        for (int g = 0; g < FB_GMAX; ++g) {
          if (g >= gc) break;
          const float approx = warp_sum(acc[r][g]);
          const float cut = __shfl_sync(0xffffffffu, my_cut, g);
          const int qfold = __shfl_sync(0xffffffffu, my_fold, g);
          if (approx < cut || dfold == qfold) continue;            // warp-uniform: cannot reach the Top-K / inadmissible
          // exact score, in the order of the re-scoring stage (128-bit chunks, four fused multiply-adds each, warp sum)
          const float* qrow = p.q + static_cast<int64_t>(p.flag_list[g0 + g]) * p.ldq;
          float ex = 0.f;
          LazyRowCtx ctx;
          if (SRC != 0) ctx = lazy_row_ctx(p.lazy, row);
          for (int e = lane * 4; e < p.D; e += 128) {
            const float4 x = __ldg(reinterpret_cast<const float4*>(qrow + e));
            const float4 v = SRC == 0 ? __ldg(reinterpret_cast<const float4*>(p.db + row * p.lddb + e))
                                      : lazy_load4<typename RawOf<SRC>::T>(p.lazy, ctx, row, e);
            ex = fmaf(x.x, v.x, ex); ex = fmaf(x.y, v.y, ex); ex = fmaf(x.z, v.z, ex); ex = fmaf(x.w, v.w, ex);
          }
          ex = warp_sum(ex);
          if (lane == g) {
            const uint64_t key = pack_key(ex, static_cast<uint32_t>(row + p.idx_base));
            if (key > kth) {
              uint64_t* mine = lists + (warp * G + g) * K;
              int pos = K - 1;
              while (pos > 0 && mine[pos - 1] < key) { mine[pos] = mine[pos - 1]; --pos; }
              mine[pos] = key;
              kth = mine[K - 1];
              if (kth != 0ull) my_cut = fmaxf(my_cut, key_score(kth) - my_e);
            }
          }
        }
      }
    }
    __syncthreads();
    // merge the warps' lists of each query: warp w serves queries w, w + FB_WARPS, ...
    for (int g = warp; g < gc; g += FB_WARPS) {
      uint64_t bound = ~0ull;
      for (int rnk = 0; rnk < K; ++rnk) {
        uint64_t best = 0ull;
        for (int t = lane; t < FB_WARPS * K; t += 32) {
          const int w = t / K, j = t - w * K;
          const uint64_t key = lists[(w * G + g) * K + j];
          if (key < bound && key > best) best = key;
        }
        best = warp_max_u64(best);
        bound = best;
        if (lane == 0) p.fb_parts[(static_cast<int64_t>(blockIdx.x) * p.cap + g0 + g) * K + rnk] = best;
        if (best == 0ull) {
          for (int r2 = rnk + 1 + lane; r2 < K; r2 += 32)
            p.fb_parts[(static_cast<int64_t>(blockIdx.x) * p.cap + g0 + g) * K + r2] = 0ull;
          break;
        }
      }
    }
  }
}

__global__ void __launch_bounds__(256) rescan_merge_kernel(const RescoreParams p, int blocks) {
  const int n = flagged_count(p);
  const int lane = threadIdx.x & 31;
  const int i = static_cast<int>((static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5);
  if (i >= n) return;
  const int K = p.K;
  const int64_t qd = p.compact ? i : p.flag_list[i];
  uint64_t bound = ~0ull;
  for (int rnk = 0; rnk < K; ++rnk) {
    uint64_t best = 0ull;
    if (bound != 0ull) {
      for (int t = lane; t < blocks * K; t += 32) {
        const int b = t / K, j = t - b * K;
        const uint64_t key = p.fb_parts[(static_cast<int64_t>(b) * p.cap + i) * K + j];
        if (key < bound && key > best) best = key;
      }
      best = warp_max_u64(best);
    }
    bound = best;
    if (lane == 0) p.out[qd * K + rnk] = best;
  }
}

// [Q] local K-th best filter score (-inf if the list is shorter) -- what the shards exchange (max) before re-scoring
__global__ void __launch_bounds__(256) kth_score_kernel(const uint64_t* __restrict__ approx, int KP, int K, int64_t Q,
                                                        float* __restrict__ kth) {
  const int64_t q = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  const uint64_t k = K <= KP ? approx[q * KP + K - 1] : 0ull;
  kth[q] = k != 0ull ? key_score(k) : -INFINITY;
}

// merged lists of all shards + every shard's bound: flag the queries whose exact K-th best does not clear every bound
__global__ void __launch_bounds__(256) verify_merged_kernel(const uint64_t* __restrict__ keys, int K, int64_t Q,
                                                            const float* __restrict__ bounds, int parts,
                                                            int64_t bounds_stride, uint8_t* __restrict__ flags,
                                                            int* __restrict__ count) {
  const int64_t q = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (q >= Q) return;
  float b = -INFINITY;
  for (int p = 0; p < parts; ++p) b = fmaxf(b, bounds[static_cast<int64_t>(p) * bounds_stride + q]);
  const uint64_t kth = keys[q * K + K - 1];
  const bool ok = (b == -INFINITY) || (kth != 0ull && key_score(kth) > b);
  flags[q] = ok ? 0 : 1;
  if (!ok) { atomicAdd(count, 1); count[1] = 1; }      // [1]: the merged selection needs the exact re-scan
}

int rescore_kth_scores(const uint64_t* approx, int KP, int K, int64_t Q, float* kth, cudaStream_t st) {
  kth_score_kernel<<<static_cast<unsigned>((Q + 255) / 256), 256, 0, st>>>(approx, KP, K, Q, kth);
  EMR2A_LAUNCH_CHECK("kth_score_kernel");
  return EMR2A_OK;
}

// src of the fp32 database rows: 0 = matrix, 1 / 2 = deferred (raw fp32 / bf16 rows + K1's divisors)
static int rows_src(const emr2a_lazy_rows* lz) { return lz == nullptr ? 0 : (lz->dtype == EMR2A_BF16 ? 2 : 1); }

static int lazy_fill(RescoreParams& p, const emr2a_lazy_rows* lz, int D) {
  if (lz == nullptr) return EMR2A_OK;
  const size_t al = lz->dtype == EMR2A_BF16 ? 8 : 16;
  auto ok = [&](const void* x) { return x != nullptr && (reinterpret_cast<uintptr_t>(x) % al) == 0; };
  if ((lz->dtype != EMR2A_F32 && lz->dtype != EMR2A_BF16) || lz->d0 <= 0 || lz->d1 < 0 || lz->d0 + lz->d1 != D ||
      (lz->d0 % 4) || (lz->d1 % 4) || (lz->ld0 % 4) || (lz->d1 > 0 && (lz->ld1 % 4)) || !ok(lz->seg0) ||
      (lz->d1 > 0 && !ok(lz->seg1)) || lz->row_div == nullptr || (reinterpret_cast<uintptr_t>(lz->row_div) & 15) ||
      (lz->flags & EMR2A_NF_STANDARDIZE))
    return fail(EMR2A_ERR_UNSUPPORTED, "deferred fp32 rows need 4-element-aligned segments, aligned pointers, row_div and no fused standardisation");
  p.lazy.seg0 = lz->seg0; p.lazy.seg1 = lz->seg1; p.lazy.d0 = lz->d0; p.lazy.d1 = lz->d1; p.lazy.ld0 = lz->ld0;
  p.lazy.ld1 = lz->d1 > 0 ? lz->ld1 : 0; p.lazy.w0 = lz->w0; p.lazy.w1 = lz->w1; p.lazy.flags = lz->flags;
  p.lazy.row_div = lz->row_div;
  return EMR2A_OK;
}

template <int SRC>
static void launch_select_src(const RescoreParams& p, bool vec, cudaStream_t st) {
  if (p.Q <= 4 * static_cast<int64_t>(sm_count())) {        // small batch: a block per query (latency layout)
    if (vec) rescore_select_kernel<true, 8, SRC><<<static_cast<unsigned>(p.Q), 256, 0, st>>>(p);
    else if constexpr (SRC == 0) rescore_select_kernel<false, 8, 0><<<static_cast<unsigned>(p.Q), 256, 0, st>>>(p);
  } else {
    const unsigned blocks = static_cast<unsigned>((p.Q * 32 + 255) / 256);
    if (vec) rescore_select_kernel<true, 1, SRC><<<blocks, 256, 0, st>>>(p);
    else if constexpr (SRC == 0) rescore_select_kernel<false, 1, 0><<<blocks, 256, 0, st>>>(p);
  }
}

static bool rows_vec(const RescoreParams& p, int src) {
  auto al16 = [](const void* x) { return (reinterpret_cast<uintptr_t>(x) & 15) == 0; };
  const bool qv = (p.D % 4 == 0) && (p.ldq % 4 == 0) && al16(p.q);
  return src != 0 ? qv : (qv && (p.lddb % 4 == 0) && al16(p.db));
}

static int launch_select(const RescoreParams& p, int src, cudaStream_t st) {
  const bool vec = rows_vec(p, src);
  if (src != 0 && !vec) return fail(EMR2A_ERR_UNSUPPORTED, "deferred fp32 rows need 16-byte aligned fp32 query rows with D %% 4 == 0");
  if (src == 0) launch_select_src<0>(p, vec, st);
  else if (src == 1) launch_select_src<1>(p, vec, st);
  else launch_select_src<2>(p, vec, st);
  EMR2A_LAUNCH_CHECK("rescore_select_kernel");
  return EMR2A_OK;
}

// re-score only (no local verification, no re-scan): exact keys of the candidates that clear the (global) cut + bound_out
int rescore_select_only(const uint64_t* approx, int KP, const uint32_t* tau, const float* kth_floor, const float* q,
                        int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int64_t Q, int64_t N, int D,
                        int64_t idx_base, int K, const float* q_stats, const float* db_stats, uint64_t* out_keys,
                        float* bound_out, cudaStream_t st) {
  RescoreParams p{};
  p.approx = approx; p.KP = KP; p.tau = tau; p.q = q; p.ldq = ldq; p.db = db; p.lddb = lddb; p.Q = Q; p.N = N; p.D = D;
  p.idx_base = idx_base; p.K = K; p.q_stats = q_stats; p.db_stats = db_stats; p.out = out_keys;
  p.kth_floor = kth_floor; p.bound_out = bound_out;
  const int rc = lazy_fill(p, db_lazy, D);
  if (rc != EMR2A_OK) return rc;
  return launch_select(p, rows_src(db_lazy), st);
}

int rescore_verify_merged(const uint64_t* keys, int K, int64_t Q, const float* bounds, int parts, int64_t bounds_stride,
                          uint8_t* flags, int* count, cudaStream_t st) {
  verify_merged_kernel<<<static_cast<unsigned>((Q + 255) / 256), 256, 0, st>>>(keys, K, Q, bounds, parts, bounds_stride, flags, count);
  EMR2A_LAUNCH_CHECK("verify_merged_kernel");
  return EMR2A_OK;
}

int rescore_fallback_blocks() { return 2 * sm_count(); }
// Capacity of the exact re-scan list.  A re-scan group (8 queries) streams the whole fp32 database once
// (HBM-bound), the 3-pass tensor-core search of ALL queries costs about 0.04 * Q such groups, so beyond
// ~4 % unverifiable queries handing the batch to BF16X3 (status[1]) is cheaper than re-scanning.
int rescore_cap(int64_t Q) {
  int64_t cap = Q / 25;
  if (cap < 64) cap = 64;
  if (cap > 1024) cap = 1024;
  return static_cast<int>(cap < Q ? cap : Q);
}

size_t rescore_workspace_bytes(int64_t Q, int K) {
  const int cap = rescore_cap(Q);
  return sizeof(int) * static_cast<size_t>(cap) + 256 +
         sizeof(uint64_t) * static_cast<size_t>(rescore_fallback_blocks()) * cap * K + 256;
}

template <int SRC, int NW>
static int launch_rescan_src(const RescoreParams& p, bool vec, int G, size_t smem, int fb_blocks, cudaStream_t st) {
  if (vec) {
    EMR2A_CUDA_TRY(cudaFuncSetAttribute(exact_rescan_kernel<true, SRC, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024));
    exact_rescan_kernel<true, SRC, NW><<<fb_blocks, NW * 32, smem, st>>>(p, G);
  } else if constexpr (SRC == 0) {
    EMR2A_CUDA_TRY(cudaFuncSetAttribute(exact_rescan_kernel<false, 0, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, 208 * 1024));
    exact_rescan_kernel<false, 0, NW><<<fb_blocks, NW * 32, smem, st>>>(p, G);
  }
  EMR2A_LAUNCH_CHECK("exact_rescan_kernel");
  return EMR2A_OK;
}

static bool rescan_filter_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("EMR2A_RESCAN_FILTER");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v != 0;
}

template <int SRC>
static int launch_filtered_src(const RescoreParams& p, int G, size_t smem, int blocks, cudaStream_t st) {
  EMR2A_CUDA_TRY(cudaFuncSetAttribute(filtered_rescan_kernel<SRC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  filtered_rescan_kernel<SRC><<<blocks, FB_WARPS * 32, smem, st>>>(p, G);
  EMR2A_LAUNCH_CHECK("filtered_rescan_kernel");
  return EMR2A_OK;
}

static int launch_rescan(const RescoreParams& p, int src, cudaStream_t st) {
  const int D = p.D, K = p.K;
  // filtered re-scan: needs the bf16 plane, K1's statistics (the bound) and the 128-bit path of the exact scoring
  // and a seed for the cut (without one every warp would score rows exactly until its OWN list is full of good rows)
  if (rescan_filter_enabled() && p.seed != nullptr && p.db_hi != nullptr && p.q_stats != nullptr && p.db_stats != nullptr && rows_vec(p, src) &&
      (p.lddb_hi % 8) == 0 && p.lddb_hi >= ((D + 7) & ~7) && (reinterpret_cast<uintptr_t>(p.db_hi) & 15) == 0) {
    const int Dh = (D + 7) & ~7;
    const size_t list_bytes = sizeof(uint64_t) * FB_WARPS * FB_GMAX * K;
    int G = static_cast<int>((96 * 1024 - list_bytes) / (sizeof(uint16_t) * Dh));
    if (G > FB_GMAX) G = FB_GMAX;
    if (G >= 1) {
      const size_t smem = ((sizeof(uint16_t) * G * Dh + 15) & ~static_cast<size_t>(15)) + sizeof(uint64_t) * FB_WARPS * G * K;
      const int blocks = rescore_fallback_blocks();
      const int rc = src == 0 ? launch_filtered_src<0>(p, G, smem, blocks, st)
                   : src == 1 ? launch_filtered_src<1>(p, G, smem, blocks, st)
                              : launch_filtered_src<2>(p, G, smem, blocks, st);
      if (rc != EMR2A_OK) return rc;
      rescan_merge_kernel<<<static_cast<unsigned>((static_cast<int64_t>(p.cap) * 32 + 255) / 256), 256, 0, st>>>(p, blocks);
      EMR2A_LAUNCH_CHECK("rescan_merge_kernel");
      return EMR2A_OK;
    }
  }
  const int Dp = (D + 3) & ~3;
  int G = static_cast<int>((96 * 1024) / (sizeof(float) * Dp));
  const bool wide = G < FB_GMAX;            // the query group does not fit beside a second block: one 16-warp block per SM
  if (wide) G = static_cast<int>((200 * 1024 - sizeof(uint64_t) * 16 * FB_GMAX * K) / (sizeof(float) * Dp));
  if (G > FB_GMAX) G = FB_GMAX;
  if (G < 1) return fail(EMR2A_ERR_UNSUPPORTED, "topk_search(rescore): D=%d too large for the exact re-scan", D);
  const int nw = wide ? 16 : FB_WARPS;
  const size_t smem = sizeof(float) * G * Dp + sizeof(uint64_t) * nw * G * K;
  const int fb_blocks = wide ? sm_count() : rescore_fallback_blocks();      // resident blocks: one / two per SM (the workspace holds two)
  const bool vec = rows_vec(p, src);
  if (src != 0 && !vec) return fail(EMR2A_ERR_UNSUPPORTED, "deferred fp32 rows need 16-byte aligned fp32 query rows with D %% 4 == 0");
  int rc;
  if (wide) rc = src == 0 ? launch_rescan_src<0, 16>(p, vec, G, smem, fb_blocks, st)
               : src == 1 ? launch_rescan_src<1, 16>(p, vec, G, smem, fb_blocks, st)
                          : launch_rescan_src<2, 16>(p, vec, G, smem, fb_blocks, st);
  else rc = src == 0 ? launch_rescan_src<0, FB_WARPS>(p, vec, G, smem, fb_blocks, st)
          : src == 1 ? launch_rescan_src<1, FB_WARPS>(p, vec, G, smem, fb_blocks, st)
                     : launch_rescan_src<2, FB_WARPS>(p, vec, G, smem, fb_blocks, st);
  if (rc != EMR2A_OK) return rc;
  rescan_merge_kernel<<<static_cast<unsigned>((static_cast<int64_t>(p.cap) * 32 + 255) / 256), 256, 0, st>>>(p, fb_blocks);
  EMR2A_LAUNCH_CHECK("rescan_merge_kernel");
  return EMR2A_OK;
}

// approx: merged approximate keys [Q][KP]; writes exact keys [Q][K]; status[0..1] must be zeroed by the caller.
int rescore_pipeline(const uint64_t* approx, int KP, const uint32_t* tau, const float* q, int64_t ldq, const float* db,
                     int64_t lddb, const emr2a_lazy_rows* db_lazy, const uint16_t* db_hi, int64_t lddb_hi, int64_t Q, int64_t N,
                     int D, int64_t idx_base, int K,
                     const float* q_stats, const float* db_stats, const uint8_t* q_fold, const uint8_t* db_fold,
                     uint64_t* out_keys, int* status, uint8_t* qflags, void* workspace, size_t ws_bytes, cudaStream_t st) {
  if (!q_stats || !db_stats) return fail(EMR2A_ERR_INVALID, "topk_search(rescore): q_stats/db_stats (K1 stats) required");
  if (!status) return fail(EMR2A_ERR_INVALID, "topk_search(rescore): status_out required");
  if (rescore_workspace_bytes(Q, K) > ws_bytes) return fail(EMR2A_ERR_WORKSPACE, "topk_search(rescore): workspace too small");
  RescoreParams p{};
  p.approx = approx; p.KP = KP; p.tau = tau; p.q = q; p.ldq = ldq; p.db = db; p.lddb = lddb; p.Q = Q; p.N = N; p.D = D;
  p.idx_base = idx_base; p.K = K; p.q_stats = q_stats; p.db_stats = db_stats; p.out = out_keys; p.status = status;
  p.cap = rescore_cap(Q);
  p.n_fixed = -1;
  p.qflags = qflags;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  p.flag_list = reinterpret_cast<int*>(ws);
  const size_t off = (sizeof(int) * static_cast<size_t>(p.cap) + 255) & ~static_cast<size_t>(255);
  p.fb_parts = reinterpret_cast<uint64_t*>(ws + off);
  p.q_fold = q_fold; p.db_fold = db_fold;
  p.db_hi = db_hi; p.lddb_hi = lddb_hi;
  p.seed = out_keys; p.seed_compact = 0;        // the exact Top-K of the candidates seeds the cut of the filtered re-scan
  int rc = lazy_fill(p, db_lazy, D);
  if (rc != EMR2A_OK) return rc;
  const int src = rows_src(db_lazy);
  if ((rc = launch_select(p, src, st)) != EMR2A_OK) return rc;
  // exact re-scan of unverified queries; both kernels return at once when status[0] == 0
  return launch_rescan(p, src, st);
}

// The exact re-scan alone, for a flag list the caller holds (cooperative shards: the queries the MERGED lists could not
// verify are re-searched exactly on every shard, the compact lists [n_flagged][K] are merged by the caller).
size_t exact_rescan_workspace_bytes(int n_flagged, int K) {
  return sizeof(uint64_t) * static_cast<size_t>(rescore_fallback_blocks()) * static_cast<size_t>(n_flagged > 0 ? n_flagged : 1) * K + 256;
}

int rescore_exact_rescan(const float* q, int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int64_t N,
                         int D, int64_t idx_base, int K, const uint8_t* q_fold, const uint8_t* db_fold, const int* flag_list,
                         int n_flagged, uint64_t* out_compact, void* workspace, size_t ws_bytes, const uint16_t* db_hi,
                         int64_t lddb_hi, const float* q_stats, const float* db_stats, const uint64_t* seed_keys,
                         cudaStream_t st) {
  if (n_flagged <= 0) return EMR2A_OK;
  if (!workspace || exact_rescan_workspace_bytes(n_flagged, K) > ws_bytes) return fail(EMR2A_ERR_WORKSPACE, "exact_rescan: workspace too small");
  RescoreParams p{};
  p.q = q; p.ldq = ldq; p.db = db; p.lddb = lddb; p.N = N; p.D = D; p.idx_base = idx_base; p.K = K; p.out = out_compact;
  p.flag_list = const_cast<int*>(flag_list); p.cap = n_flagged; p.n_fixed = n_flagged; p.compact = 1;
  p.q_fold = q_fold; p.db_fold = db_fold;
  p.fb_parts = reinterpret_cast<uint64_t*>(workspace);
  p.db_hi = db_hi; p.lddb_hi = lddb_hi; p.q_stats = q_stats; p.db_stats = db_stats;
  p.seed = seed_keys; p.seed_compact = 1;
  const int rc = lazy_fill(p, db_lazy, D);
  if (rc != EMR2A_OK) return rc;
  return launch_rescan(p, rows_src(db_lazy), st);
}

// ---- range search, refine stage (emr2a_range_search) ----------------------------------------------------------------
// The filter emitted every admissible pair with s~ >= t - E; the exact score s of each is computed here and the pair is
// kept iff s >= t.  A warp per candidate, in the arithmetic and reduction order of rescore_select_kernel (128-bit
// chunks, four fused multiply-adds each, then warp_sum; 32-bit chunks without the 128-bit path), so the scores are
// bit-identical to the ones the Top-K of the rescore arm reports for the same pair.
struct RangeRefineParams {
  const ulonglong2* cand;                  // [min(counts[0], cand_cap)] (query, approximate key)
  int64_t cand_cap;
  unsigned long long* counts;              // [0] candidates (filter), [1] results (here)
  ulonglong2* out;                         // [out_cap] (query, exact key)
  int64_t out_cap;
  const float* q; int64_t ldq;
  const float* db; int64_t lddb;
  LazyRows lazy;
  int D;
  int64_t idx_base;
  float t;
};

template <bool VEC, int SRC>
__global__ void __launch_bounds__(256) range_refine_kernel(const RangeRefineParams p) {
  static_assert(SRC == 0 || VEC, "deferred fp32 rows need the 128-bit path");
  const unsigned long long n = p.counts[0];
  if (n > static_cast<unsigned long long>(p.cand_cap)) return;      // incomplete candidate list: the caller retries
  const int lane = threadIdx.x & 31;
  const unsigned long long warps = static_cast<unsigned long long>(gridDim.x) * (blockDim.x >> 5);
  for (unsigned long long i = (static_cast<unsigned long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
    const ulonglong2 c = p.cand[i];
    const uint32_t gidx = key_index(c.y);
    const int64_t row = static_cast<int64_t>(gidx) - p.idx_base;
    const float* qrow = p.q + static_cast<int64_t>(c.x) * p.ldq;
    float acc = 0.f;
    if (VEC) {
      LazyRowCtx ctx;
      if (SRC != 0) ctx = lazy_row_ctx(p.lazy, row);
      for (int e = lane * 4; e < p.D; e += 128) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(qrow + e));
        const float4 y = SRC == 0 ? __ldg(reinterpret_cast<const float4*>(p.db + row * p.lddb + e))
                                  : lazy_load4<typename RawOf<SRC>::T>(p.lazy, ctx, row, e);
        acc = fmaf(x.x, y.x, acc); acc = fmaf(x.y, y.y, acc);
        acc = fmaf(x.z, y.z, acc); acc = fmaf(x.w, y.w, acc);
      }
    } else {
      for (int e = lane; e < p.D; e += 32) acc = fmaf(__ldg(qrow + e), __ldg(p.db + row * p.lddb + e), acc);
    }
    const float s = warp_sum(acc);
    if (lane == 0 && s >= p.t) {
      const unsigned long long pos = atomicAdd(p.counts + 1, 1ull);
      if (pos < static_cast<unsigned long long>(p.out_cap)) p.out[pos] = make_ulonglong2(c.x, pack_key(s, gidx));
    }
  }
}

template <int SRC>
static void launch_refine_src(const RangeRefineParams& p, bool vec, unsigned blocks, cudaStream_t st) {
  if (vec) range_refine_kernel<true, SRC><<<blocks, 256, 0, st>>>(p);
  else if constexpr (SRC == 0) range_refine_kernel<false, 0><<<blocks, 256, 0, st>>>(p);
}

// Operand rules of the refine stage (deferred rows, 128-bit path): fills rp, launches nothing.
static int range_refine_operands(RescoreParams& rp, const float* q, int64_t ldq, const float* db, int64_t lddb,
                                 const emr2a_lazy_rows* db_lazy, int D) {
  rp.q = q; rp.ldq = ldq; rp.db = db; rp.lddb = lddb; rp.D = D;
  const int rc = lazy_fill(rp, db_lazy, D);
  if (rc != EMR2A_OK) return rc;
  if (rows_src(db_lazy) != 0 && !rows_vec(rp, rows_src(db_lazy)))
    return fail(EMR2A_ERR_UNSUPPORTED, "deferred fp32 rows need 16-byte aligned fp32 query rows with D %% 4 == 0");
  return EMR2A_OK;
}

int range_refine_check(const float* q, int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int D) {
  RescoreParams rp{};
  return range_refine_operands(rp, q, ldq, db, lddb, db_lazy, D);
}

int range_refine(const uint64_t* cand, int64_t cand_cap, unsigned long long* counts, uint64_t* out, int64_t out_cap,
                 const float* q, int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int D,
                 int64_t idx_base, float min_score, cudaStream_t st) {
  RescoreParams rp{};
  const int rc = range_refine_operands(rp, q, ldq, db, lddb, db_lazy, D);
  if (rc != EMR2A_OK) return rc;
  const int src = rows_src(db_lazy);
  const bool vec = rows_vec(rp, src);
  RangeRefineParams p{};
  p.cand = reinterpret_cast<const ulonglong2*>(cand); p.cand_cap = cand_cap; p.counts = counts;
  p.out = reinterpret_cast<ulonglong2*>(out); p.out_cap = out_cap;
  p.q = q; p.ldq = ldq; p.db = db; p.lddb = lddb; p.lazy = rp.lazy; p.D = D; p.idx_base = idx_base; p.t = min_score;
  const unsigned blocks = static_cast<unsigned>(8 * sm_count());      // grid-stride: the candidate count is on the device
  if (src == 0) launch_refine_src<0>(p, vec, blocks, st);
  else if (src == 1) launch_refine_src<1>(p, vec, blocks, st);
  else launch_refine_src<2>(p, vec, blocks, st);
  EMR2A_LAUNCH_CHECK("range_refine_kernel");
  return EMR2A_OK;
}

}  // namespace emr2a
