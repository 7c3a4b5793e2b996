// K2 (tensor-core arm): query x database similarity as a tcgen05/TMEM GEMM fed by TMA, with the
// Top-K selection fused into the epilogue -- the score matrix never reaches HBM.
//
// Mapping (sm_100a, one CTA per SM, 256 threads, warp-specialised):
//   M (TMEM lanes)   = 128 queries      -> each epilogue thread owns ONE query row
//   N (TMEM columns) = 256 database rows per tile, two accumulators (2 x 256 = all 512 columns)
//   K                = 64 bf16 per stage (one 128-byte swizzle row), UMMA_K = 16
//   warp 0  TMA producer   : cp.async.bulk.tensor.2d -> 128B-swizzled smem ring, mbarrier complete_tx
//   warp 1  MMA issuer     : tcgen05.mma.cta_group::1.kind::f16 (bf16 x bf16 -> fp32 in TMEM)
//                            BF16X3: per k-step hi*hi + hi*lo + lo*hi into the same accumulator
//   warp 2  TMEM allocator
//   warps 4-7 epilogue     : tcgen05.ld 32x32b.x32 -> 32 scores of the thread's own query per chunk,
//                            running max against the thread's K-th best (compare-mostly), rare sorted
//                            insertion into a register-resident Top-K list; the epilogue of tile t
//                            overlaps the MMAs of tile t+1 through the second accumulator.
// A CTA walks work units (query tile, database split) statically; each unit ends with the thread
// writing its list as packed keys to the partial-list workspace, merged afterwards by K3.
//
// Roofline: tensor pipe.  Algorithmic FLOPs = 2 * D * Q * N_admissible; BF16X3 issues 3x that.
#include <stdlib.h>
#include "tc_common.cuh"

namespace emr2a {

template <int PASSES, int KCAP, bool HAS_FOLD, bool RANGE = false>
__global__ void __launch_bounds__(T_THREADS, 1)
tc_topk_kernel(const __grid_constant__ CUtensorMap tm_q_hi, const __grid_constant__ CUtensorMap tm_q_lo,
               const __grid_constant__ CUtensorMap tm_db_hi, const __grid_constant__ CUtensorMap tm_db_lo,
               const TcParams p) {
  constexpr int PLANES = PASSES == 3 ? 2 : 1;
  constexpr uint32_t STAGE_BYTES = PLANES * (T_A_BYTES + T_B_BYTES);
  constexpr int STAGES = PASSES == 3 ? 2 : 4;

  extern __shared__ uint8_t smem_dyn[];
  __shared__ __align__(8) uint64_t bar_full[STAGES];
  __shared__ __align__(8) uint64_t bar_empty[STAGES];
  __shared__ __align__(8) uint64_t bar_tfull[2];
  __shared__ __align__(8) uint64_t bar_tempty[2];
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t tiles_base = (smem_u32(smem_dyn) + 1023u) & ~1023u;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tm_q_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tm_db_hi)) : "memory");
    if (PASSES == 3) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tm_q_lo)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tm_db_lo)) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&bar_tfull[a]), 1); mbar_init(smem_u32(&bar_tempty[a]), 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "n"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  const int64_t n_units = p.m_tiles * p.splits;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int64_t split = u / p.m_tiles, mt = u - split * p.m_tiles;
        const int m0 = static_cast<int>(mt * T_BM);
        const int64_t t0 = split * p.tiles_per_split;
        const int64_t t1 = (t0 + p.tiles_per_split < p.n_tiles) ? t0 + p.tiles_per_split : p.n_tiles;
        const int ufold = HAS_FOLD ? unit_fold(p, mt) : -1;
        for (int64_t t = t0; t < t1; ++t) {
          if ((HAS_FOLD && tile_skipped(p, ufold, t)) || tri_skipped<RANGE>(p, mt, T_BM, t)) continue;
          const int n0 = static_cast<int>(t * T_BN);
          for (int kc = 0; kc < p.k_chunks; ++kc) {
            mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
            const uint32_t full = smem_u32(&bar_full[stage]);
            mbar_arrive_expect_tx(full, STAGE_BYTES);
            const uint32_t sb = tiles_base + stage * STAGE_BYTES;
            tma_load_2d(sb, &tm_q_hi, full, kc * T_BK, m0);
            tma_load_2d(sb + PLANES * T_A_BYTES, &tm_db_hi, full, kc * T_BK, n0);
            if (PASSES == 3) {
              tma_load_2d(sb + T_A_BYTES, &tm_q_lo, full, kc * T_BK, m0);
              tma_load_2d(sb + PLANES * T_A_BYTES + T_B_BYTES, &tm_db_lo, full, kc * T_BK, n0);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
        const int64_t split = u / p.m_tiles;
        const int64_t t0 = split * p.tiles_per_split;
        const int64_t t1 = (t0 + p.tiles_per_split < p.n_tiles) ? t0 + p.tiles_per_split : p.n_tiles;
        const int64_t mt = u - split * p.m_tiles;
        const int ufold = HAS_FOLD ? unit_fold(p, mt) : -1;
        for (int64_t t = t0; t < t1; ++t) {
          if ((HAS_FOLD && tile_skipped(p, ufold, t)) || tri_skipped<RANGE>(p, mt, T_BM, t)) continue;
          mbar_wait(smem_u32(&bar_tempty[acc]), acc_phase ^ 1u);
          tcgen05_fence_after();
          const uint32_t d_tmem = tmem_base + static_cast<uint32_t>(acc * T_BN);
          for (int kc = 0; kc < p.k_chunks; ++kc) {
            mbar_wait(smem_u32(&bar_full[stage]), phase);
            tcgen05_fence_after();
            const uint32_t sb = tiles_base + stage * STAGE_BYTES;
            const uint64_t a_hi = make_smem_desc(sb);
            const uint64_t b_hi = make_smem_desc(sb + PLANES * T_A_BYTES);
            const uint64_t a_lo = make_smem_desc(sb + T_A_BYTES);
            const uint64_t b_lo = make_smem_desc(sb + PLANES * T_A_BYTES + T_B_BYTES);
#pragma unroll
            for (int k = 0; k < T_BK / 16; ++k) {
              const uint64_t koff = static_cast<uint64_t>((k * 32) >> 4);     // 16 bf16 = 32 bytes along the swizzled row
              if (PASSES == 3) {
                // small cross terms first, dominant term last
                umma_bf16(d_tmem, a_hi + koff, b_lo + koff, T_IDESC, (kc | k) != 0 ? 1u : 0u);
                umma_bf16(d_tmem, a_lo + koff, b_hi + koff, T_IDESC, 1u);
                umma_bf16(d_tmem, a_hi + koff, b_hi + koff, T_IDESC, 1u);
              } else {
                umma_bf16(d_tmem, a_hi + koff, b_hi + koff, T_IDESC, (kc | k) != 0 ? 1u : 0u);
              }
            }
            umma_commit(smem_u32(&bar_empty[stage]));       // smem slot free once these MMAs retire
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
          umma_commit(smem_u32(&bar_tfull[acc]));           // accumulator complete -> epilogue
          if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue: fused Top-K =====================
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    RegTopK<KCAP> top;
    float cut = 0.f;
    if constexpr (RANGE) cut = range_cut(p);
    for (int64_t u = blockIdx.x; u < n_units; u += gridDim.x) {
      const int64_t split = u / p.m_tiles, mt = u - split * p.m_tiles;
      const int64_t q = mt * T_BM + row;
      const int64_t t0 = split * p.tiles_per_split;
      const int64_t t1 = (t0 + p.tiles_per_split < p.n_tiles) ? t0 + p.tiles_per_split : p.n_tiles;
      const uint32_t my_fold = (HAS_FOLD && q < p.Q) ? p.q_fold[q] : 0xFFFFu;
      if constexpr (!RANGE) top.reset();
      const float thr0 = RANGE ? cut : unit_start_threshold(p, q);
      float thr = thr0;
      const int ufold = HAS_FOLD ? unit_fold(p, mt) : -1;
      for (int64_t t = t0; t < t1; ++t) {
        if ((HAS_FOLD && tile_skipped(p, ufold, t)) || tri_skipped<RANGE>(p, mt, T_BM, t)) continue;
        const int64_t n0 = t * T_BN;
        mbar_wait(smem_u32(&bar_tfull[acc]), acc_phase);
        tcgen05_fence_after();
        scan_tile<KCAP, HAS_FOLD, RANGE>(p, top, thr, thr0,
                                         tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(acc * T_BN),
                                         n0, my_fold, q);
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&bar_tempty[acc]));
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      if (!RANGE && q < p.Q) {
        if (p.tau != nullptr && top.i[KCAP - 1] != 0xFFFFFFFFu) atomicMax(p.tau + q, order_f32(top.s[KCAP - 1]));
        uint64_t* dst = p.keys_out + (split * p.Q + q) * p.K;
#pragma unroll
        for (int j = 0; j < KCAP; ++j)
          if (j < p.K) dst[j] = (top.i[j] == 0xFFFFFFFFu) ? 0ull : pack_key(top.s[j], top.i[j]);
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512));
  }
}

// ---- host side ------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(sym);
  }
  return fn;
}

static int make_plane_map(CUtensorMap* map, const uint16_t* base, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  PFN_encodeTiled enc = get_encode();
  if (!enc) return fail(EMR2A_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  cuuint64_t gstride[1] = {static_cast<cuuint64_t>(ld) * 2};
  cuuint32_t box[2] = {static_cast<cuuint32_t>(T_BK), static_cast<cuuint32_t>(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(EMR2A_ERR_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d): rows=%lld cols=%lld ld=%lld", (int)r, (long long)rows, (long long)cols, (long long)ld);
  return EMR2A_OK;
}

// When the caller asks for it, the per-split lists are left unmerged and described here.
struct TcPartials {
  const uint64_t* parts;   // [splits][Q][K]
  int splits;
  const uint32_t* tau;     // [Q] max over splits of the split's K-th (last kept) score, 0 = no list was full; null if splits == 1
};

struct TcPlan {
  int64_t m_tiles, n_tiles, tiles_per_split;
  int splits;
  int grid;
  size_t keys_bytes, fold_bytes, tau_bytes;
  // CTA pairs: unit grouping and cohort pacing (tc_common.cuh: unit_coords / cohort_sync)
  int64_t mg;
  int sync_tiles, sync_points, sync_budget;
  size_t sync_bytes;
};

static int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return (e && *e) ? atoi(e) : dflt;
}

// diagnostics (emr2a_debug_unit_clocks): globaltimer at the start / end of every work unit of the last pair-kernel launch
constexpr int64_t UNIT_CLOCK_MAX = 1 << 16;
__device__ unsigned long long g_unit_clock[2 * UNIT_CLOCK_MAX];
static int64_t g_last_plan[8];

// CTA-pair kernel (topk_tc2.cu)
int tc2_dispatch(int passes, int kcap, bool has_fold, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c,
                 const CUtensorMap& d, const TcParams& p, int grid, cudaStream_t st);

// CTA pairs (M = 256 per tile, cta_group::2) or single CTAs (M = 128).  Pairs win whenever the tensor pipe is the
// bound (one third less L2->SM traffic per FLOP).  A batch of up to 128 queries is HBM-bound -- the database plane is
// streamed once whatever the batch size -- and the pair kernel would still compute a full M = 256 tile (tensor pipe
// 77 % busy at Q = 64): there 148 single CTAs stream the plane faster (1M x 1024, Q = 64: 0.34 ms = 6.0 TB/s against
// 0.40 ms).  EMR2A_TC2 = 0 / 1 forces the single-CTA / pair kernel.
static bool use_cta_pairs(int64_t Q) {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("EMR2A_TC2");
    v = !e ? 2 : (e[0] == '0' ? 0 : 1);
  }
  return v == 2 ? Q > T_BM : v == 1;
}

static TcPlan tc_plan(int64_t Q, int64_t N, int K, bool has_fold, bool pairs, int min_splits = 1, int64_t ld = 1024,
                      int planes = 1) {
  TcPlan pl{};
  const int bm = pairs ? 2 * T_BM : T_BM;
  pl.m_tiles = (Q + bm - 1) / bm;
  pl.n_tiles = (N + T_BN - 1) / T_BN;
  const int sms = pairs ? sm_count() / 2 : sm_count();      // concurrent workers: CTAs or CTA pairs
  // pick the split count whose unit count fills whole waves of CTAs best
  int best_s = 1; double best_eff = -1.0;
  // at most 64 splits -- except for small query batches: with fewer query tiles than 64 splits can spread over
  // the workers, the cap rises to one unit per worker (148 CTAs / 74 pairs), so that a single-tile batch (serving,
  // Q <= 256) streams the database with every SM instead of 64 of them
  int64_t cap = 64;
  if (pl.m_tiles * cap < sms) {
    const int kcap = K <= 8 ? 8 : (K <= 16 ? 16 : 32);
    cap = sms < 2048 / kcap ? sms : 2048 / kcap;       // the register merge (K3) takes up to 2048 keys per query
    if (cap < 64) cap = 64;
  }
  const int64_t max_s = pl.n_tiles < cap ? pl.n_tiles : cap;
  int64_t first_s = min_splits < max_s ? min_splits : max_s;
  if (first_s < 1) first_s = 1;
  best_s = static_cast<int>(first_s);
  for (int64_t s = first_s; s <= max_s; ++s) {
    const int64_t tps = (pl.n_tiles + s - 1) / s;
    const int64_t s_eff = (pl.n_tiles + tps - 1) / tps;       // splits that actually get tiles
    if (s_eff != s) continue;
    const int64_t units = pl.m_tiles * s;
    const int64_t waves = (units + sms - 1) / sms;
    // per-CTA time ~ waves * tps tiles (+ ~2 tiles of list warm-up per unit)
    const double cost = static_cast<double>(waves) * (static_cast<double>(tps) + 2.0);
    const double ideal = static_cast<double>(pl.m_tiles) * pl.n_tiles / sms;
    const double eff = ideal / cost;
    if (eff > best_eff + 1e-9) { best_eff = eff; best_s = static_cast<int>(s); }
  }
  pl.splits = best_s;
  pl.tiles_per_split = (pl.n_tiles + pl.splits - 1) / pl.splits;
  const int64_t units = pl.m_tiles * pl.splits;
  pl.grid = static_cast<int>(units < sms ? units : sms) * (pairs ? 2 : 1);
  pl.keys_bytes = sizeof(uint64_t) * static_cast<size_t>(pl.splits) * Q * K;
  pl.fold_bytes = has_fold ? static_cast<size_t>(pl.n_tiles) * T_BN : 0;
  pl.tau_bytes = (sizeof(uint32_t) * static_cast<size_t>(Q) + 255) & ~static_cast<size_t>(255);
  pl.mg = pl.m_tiles;
  if (pairs) {
    // Query tiles per group: the query planes of the concurrently running pairs (mg tiles of 256 rows) are re-read
    // from L2 for every database tile and must stay there next to the database stream.  EMR2A_TC_A_MB = budget.
    const double a_tile = 2.0 * T_BM * static_cast<double>(ld) * 2.0 * planes;
    int64_t mg = static_cast<int64_t>(env_int("EMR2A_TC_A_MB", 40) * 1048576.0 / a_tile);
    if (mg < 1) mg = 1;
    if (mg < pl.m_tiles) {
      const int64_t j = (sms + mg - 1) / mg;       // whole cohorts per wave of pairs where possible
      mg = sms / j;
      if (mg < 1) mg = 1;
      pl.mg = mg;
    }
    // Cohort pacing: meeting points every ~2 MB of database stream (per cohort), budget in SM cycles.
    const double b_tile = static_cast<double>(T_BN) * static_cast<double>(ld) * 2.0 * planes;
    int st = static_cast<int>(2097152.0 / b_tile + 0.5);
    st = st < 1 ? 1 : (st > 16 ? 16 : st);
    st = env_int("EMR2A_TC_SYNC", st);
    const int64_t cohort_max = pl.mg < pl.m_tiles ? pl.mg : pl.m_tiles;
    if (st > 0 && cohort_max > 1 && units > 1) {
      pl.sync_tiles = st;
      pl.sync_points = static_cast<int>((pl.tiles_per_split + st - 1) / st);
      pl.sync_budget = env_int("EMR2A_TC_SYNC_BUDGET", 12000);
      const int64_t groups = (pl.m_tiles + pl.mg - 1) / pl.mg;
      const int64_t slots = groups * pl.splits + (units + sms - 1) / sms + 2;
      pl.sync_bytes = (sizeof(uint32_t) * static_cast<size_t>(slots) * pl.sync_points + 255) & ~static_cast<size_t>(255);
    }
  }
  return pl;
}

// number of database splits the search will use (the rescore arm sizes its candidate lists by it)
int tc_planned_splits(int64_t Q, int64_t N, int min_splits) {
  return tc_plan(Q, N, 1, false, use_cta_pairs(Q), min_splits).splits;
}

size_t tc_topk_workspace_bytes(int64_t Q, int64_t N, int K, int D) {
  size_t need = 0;
  const int64_t ld = (static_cast<int64_t>(D) + T_BK - 1) / T_BK * T_BK;
  for (int v = 0; v < 8; ++v) {
    TcPlan pl = tc_plan(Q, N, K, true, (v & 1) != 0, (v & 2) ? 2 : 1, ld, (v & 4) ? 2 : 1);
    const size_t b = ((pl.keys_bytes + 255) & ~static_cast<size_t>(255)) + pl.fold_bytes + pl.tau_bytes + pl.sync_bytes + 1024;
    need = b > need ? b : need;
  }
  return need;
}

// diagnostics: plan and unit clocks of the last pair-kernel launch made with EMR2A_TC_UNIT_CLOCK=1
int tc_debug_unit_clocks(unsigned long long* host_out, int64_t cap_units, int64_t* plan_out) {
  for (int i = 0; i < 8; ++i) plan_out[i] = g_last_plan[i];
  int64_t n = g_last_plan[7];
  if (n > cap_units) n = cap_units;
  if (n > UNIT_CLOCK_MAX) n = UNIT_CLOCK_MAX;
  if (n > 0) EMR2A_CUDA_TRY(cudaMemcpyFromSymbol(host_out, g_unit_clock, sizeof(unsigned long long) * 2 * n));
  return EMR2A_OK;
}

// Diagnostics (emr2a_debug_tc_timing / emr2a_debug_tc_elapsed): CUDA events on the launching stream right before and
// right after the Top-K kernel of every search, so that bench.py can report the duration of the DOMINANT KERNEL ALONE
// (the C-ABI call also launches memsets, the merge of the partial lists and the re-scoring stage) without a profiler.
constexpr int TC_EV_RING = 1024;
static cudaEvent_t g_tc_ev[TC_EV_RING][2];
static bool g_tc_ev_made[TC_EV_RING];
static long long g_tc_ev_count = 0;
static int g_tc_ev_on = 0;

static void tc_ev_record(int which, cudaStream_t st) {
  if (!g_tc_ev_on) return;
  const int slot = static_cast<int>(g_tc_ev_count % TC_EV_RING);
  if (!g_tc_ev_made[slot]) {
    if (cudaEventCreate(&g_tc_ev[slot][0]) != cudaSuccess || cudaEventCreate(&g_tc_ev[slot][1]) != cudaSuccess) { g_tc_ev_on = 0; return; }
    g_tc_ev_made[slot] = true;
  }
  cudaEventRecord(g_tc_ev[slot][which], st);
  if (which == 1) ++g_tc_ev_count;
}
int tc_timing_enable(int on) {
  g_tc_ev_on = on ? 1 : 0;
  g_tc_ev_count = 0;
  return EMR2A_OK;
}
// elapsed milliseconds of the last (up to cap) timed launches, oldest first; waits for them to finish
int tc_timing_read(float* ms_out, int cap, int* n_out) {
  long long n = g_tc_ev_count < TC_EV_RING ? g_tc_ev_count : TC_EV_RING;
  if (n > cap) n = cap;
  for (long long i = 0; i < n; ++i) {
    const int slot = static_cast<int>((g_tc_ev_count - n + i) % TC_EV_RING);
    EMR2A_CUDA_TRY(cudaEventSynchronize(g_tc_ev[slot][1]));
    EMR2A_CUDA_TRY(cudaEventElapsedTime(ms_out + i, g_tc_ev[slot][0], g_tc_ev[slot][1]));
  }
  *n_out = static_cast<int>(n);
  return EMR2A_OK;
}

template <int PASSES, int KCAP, bool HAS_FOLD, bool RANGE = false>
static int tc_launch(const CUtensorMap& mq_hi, const CUtensorMap& mq_lo, const CUtensorMap& md_hi, const CUtensorMap& md_lo,
                     const TcParams& p, int grid, cudaStream_t st) {
  constexpr int PLANES = PASSES == 3 ? 2 : 1;
  constexpr int STAGES = PASSES == 3 ? 2 : 4;
  const size_t smem = static_cast<size_t>(STAGES) * PLANES * (T_A_BYTES + T_B_BYTES) + 1024;
  auto kern = tc_topk_kernel<PASSES, KCAP, HAS_FOLD, RANGE>;
  EMR2A_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  kern<<<grid, T_THREADS, smem, st>>>(mq_hi, mq_lo, md_hi, md_lo, p);
  EMR2A_LAUNCH_CHECK("tc_topk_kernel");
  return EMR2A_OK;
}

template <int PASSES, int KCAP>
static int tc_launch_fold(bool has_fold, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c, const CUtensorMap& d,
                          const TcParams& p, int grid, cudaStream_t st) {
  return has_fold ? tc_launch<PASSES, KCAP, true>(a, b, c, d, p, grid, st)
                  : tc_launch<PASSES, KCAP, false>(a, b, c, d, p, grid, st);
}

// Shape rules of the bf16 planes (K1 layout) shared by the Top-K and the range filter.
static int check_planes(const char* who, const uint16_t* q_hi, const uint16_t* q_lo, const uint16_t* db_hi,
                        const uint16_t* db_lo, int64_t Q, int64_t N, int D, int64_t ldq, int64_t lddb, int64_t idx_base,
                        int passes) {
  const int64_t Dp = (static_cast<int64_t>(D) + T_BK - 1) / T_BK * T_BK;
  if (ldq < Dp || lddb < Dp || (ldq % 8) || (lddb % 8))
    return fail(EMR2A_ERR_UNSUPPORTED, "%s: planes need ld >= round_up(D,64) and ld %% 8 == 0 (ldq=%lld lddb=%lld D=%d)", who, (long long)ldq, (long long)lddb, D);
  if (!q_hi || !db_hi || (passes == 3 && (!q_lo || !db_lo))) return fail(EMR2A_ERR_INVALID, "%s: missing operand plane", who);
  auto mis = [](const void* ptr) { return (reinterpret_cast<uintptr_t>(ptr) & 15) != 0; };
  if (mis(q_hi) || mis(db_hi) || (passes == 3 && (mis(q_lo) || mis(db_lo))))
    return fail(EMR2A_ERR_UNSUPPORTED, "%s: operand planes must be 16-byte aligned", who);
  if (Q >= (1LL << 31) || N >= (1LL << 31) - T_BN) return fail(EMR2A_ERR_UNSUPPORTED, "%s: Q/N too large for one call", who);
  if (N + idx_base >= 0xFFFFFFFFLL) return fail(EMR2A_ERR_UNSUPPORTED, "%s: global index exceeds 32 bits", who);
  return EMR2A_OK;
}

int tc_topk_search(const uint16_t* q_hi, const uint16_t* q_lo, const uint16_t* db_hi, const uint16_t* db_lo,
                   int64_t Q, int64_t N, int D, int64_t ldq, int64_t lddb,
                   const uint8_t* q_fold, const uint8_t* db_fold, int64_t idx_base, int K, int passes,
                   uint64_t* out_keys, void* workspace, size_t ws_bytes, float* debug_scores, cudaStream_t st,
                   TcPartials* partials, int fold_sorted, int min_splits) {
  if (K > 32) return fail(EMR2A_ERR_UNSUPPORTED, "topk_search(bf16): K=%d > 32 (use EMR2A_PREC_FP32)", K);
  const int64_t Dp = (static_cast<int64_t>(D) + T_BK - 1) / T_BK * T_BK;
  {
    const int rc = check_planes("topk_search(bf16)", q_hi, q_lo, db_hi, db_lo, Q, N, D, ldq, lddb, idx_base, passes);
    if (rc != EMR2A_OK) return rc;
  }
  const bool has_fold = q_fold != nullptr;
  const bool pairs = use_cta_pairs(Q);
  TcPlan pl = tc_plan(Q, N, K, has_fold, pairs, min_splits, lddb > ldq ? lddb : ldq, passes == 3 ? 2 : 1);
  const size_t keys_off = 0;
  const size_t fold_off = (pl.keys_bytes + 255) & ~static_cast<size_t>(255);
  const size_t tau_off = (fold_off + pl.fold_bytes + 255) & ~static_cast<size_t>(255);
  const size_t sync_off = tau_off + pl.tau_bytes;
  const size_t need = sync_off + pl.sync_bytes;
  if (!workspace || ws_bytes < need) return fail(EMR2A_ERR_WORKSPACE, "topk_search(bf16): workspace %zu < %zu", ws_bytes, need);
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  if ((reinterpret_cast<uintptr_t>(ws) & 255) != 0) return fail(EMR2A_ERR_INVALID, "topk_search(bf16): workspace must be 256-byte aligned");

  CUtensorMap mq_hi, mq_lo, md_hi, md_lo;
  int rc;
  if ((rc = make_plane_map(&mq_hi, q_hi, Q, Dp, ldq, T_BM)) != EMR2A_OK) return rc;
  const int db_box = pairs ? T_BN / 2 : T_BN;           // a CTA of a pair loads half of the database tile
  if ((rc = make_plane_map(&md_hi, db_hi, N, Dp, lddb, db_box)) != EMR2A_OK) return rc;
  if (passes == 3) {
    if ((rc = make_plane_map(&mq_lo, q_lo, Q, Dp, ldq, T_BM)) != EMR2A_OK) return rc;
    if ((rc = make_plane_map(&md_lo, db_lo, N, Dp, lddb, db_box)) != EMR2A_OK) return rc;
  } else {
    mq_lo = mq_hi; md_lo = md_hi;
  }
  TcParams p{};
  p.Q = Q; p.N = N; p.k_chunks = static_cast<int>(Dp / T_BK);
  p.m_tiles = pl.m_tiles; p.n_tiles = pl.n_tiles; p.splits = pl.splits; p.tiles_per_split = pl.tiles_per_split;
  p.idx_base = idx_base; p.K = K; p.debug_scores = debug_scores;
  p.keys_out = (pl.splits > 1 || partials) ? reinterpret_cast<uint64_t*>(ws + keys_off) : out_keys;
  if (pl.splits > 1) {     // sharing only pays (and is only needed) when a query tile is searched by several units
    p.tau = reinterpret_cast<uint32_t*>(ws + tau_off);
    EMR2A_CUDA_TRY(cudaMemsetAsync(p.tau, 0, sizeof(uint32_t) * static_cast<size_t>(Q), st));
  }
  p.mg = pl.mg;
  if (pairs && pl.sync_bytes) {
    p.sync_tiles = pl.sync_tiles; p.sync_points = pl.sync_points; p.sync_budget = pl.sync_budget;
    p.sync_ctr = reinterpret_cast<uint32_t*>(ws + sync_off);
    EMR2A_CUDA_TRY(cudaMemsetAsync(p.sync_ctr, 0, pl.sync_bytes, st));
  }
  if (pairs && env_int("EMR2A_TC_UNIT_CLOCK", 0) && pl.m_tiles * pl.splits <= UNIT_CLOCK_MAX) {
    void* sym = nullptr;
    EMR2A_CUDA_TRY(cudaGetSymbolAddress(&sym, g_unit_clock));
    p.unit_clock = static_cast<unsigned long long*>(sym);
    const int64_t plan[8] = {pl.m_tiles, pl.n_tiles, pl.splits, pl.tiles_per_split, pl.mg, pl.sync_tiles, pl.grid,
                             pl.m_tiles * pl.splits};
    for (int i = 0; i < 8; ++i) g_last_plan[i] = plan[i];
  }
  if (has_fold) {
    uint8_t* fpad = ws + fold_off;
    EMR2A_CUDA_TRY(cudaMemsetAsync(fpad, 0xFF, pl.fold_bytes, st));
    EMR2A_CUDA_TRY(cudaMemcpyAsync(fpad, db_fold, static_cast<size_t>(N), cudaMemcpyDeviceToDevice, st));
    p.q_fold = q_fold; p.db_fold = fpad; p.fold_sorted = fold_sorted;
  }
  const int kcap = K <= 8 ? 8 : (K <= 16 ? 16 : 32);
  tc_ev_record(0, st);
  if (pairs) {
    rc = tc2_dispatch(passes, kcap, has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
  } else if (passes == 3) {
    if (kcap == 8) rc = tc_launch_fold<3, 8>(has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
    else if (kcap == 16) rc = tc_launch_fold<3, 16>(has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
    else rc = tc_launch_fold<3, 32>(has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
  } else {
    if (kcap == 8) rc = tc_launch_fold<1, 8>(has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
    else if (kcap == 16) rc = tc_launch_fold<1, 16>(has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
    else rc = tc_launch_fold<1, 32>(has_fold, mq_hi, mq_lo, md_hi, md_lo, p, pl.grid, st);
  }
  tc_ev_record(1, st);
  if (rc != EMR2A_OK) return rc;
  if (partials) {
    partials->parts = p.keys_out;
    partials->splits = pl.splits;
    partials->tau = p.tau;
    return EMR2A_OK;
  }
  if (pl.splits > 1)
    return emr2a_topk_merge(reinterpret_cast<const uint64_t*>(ws + keys_off), pl.splits, Q, K, Q * K, K, K, out_keys, st);
  return EMR2A_OK;
}

void tc_timing_record(int which, cudaStream_t st) { tc_ev_record(which, st); }

int tc2_range_dispatch(bool has_fold, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c,
                       const CUtensorMap& d, const TcParams& p, int grid, cudaStream_t st);

// Filter of emr2a_range_search: the 1-pass (hi plane) tensor-core GEMM of tc_topk_search with the range epilogue --
// every admissible pair with s~ >= t - E goes to cand [cand_cap] as (query, key); *count (zeroed by the caller) counts
// them all.  Workspace: tc_topk_workspace_bytes(Q, N, 1, D) (fold padding and cohort counters of the same plan).
// tri (emr2a_self_join): query and database rows are the rows [q_row0, ...) and [idx_base, ...) of ONE row set, only
// pairs of global rows i < j are computed, and the query field of a candidate is the global row i.  The cohort pacing
// of a self-join band runs when the workspace holds its counters (emr2a_self_join_workspace_bytes sizes them for the
// whole cohort as one band; pacing never changes a result).
int tc_range_filter(const uint16_t* q_hi, const uint16_t* db_hi, int64_t Q, int64_t N, int D, int64_t ldq, int64_t lddb,
                    const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted, int64_t idx_base, float min_score,
                    const float* q_stats, const float* db_stats, uint64_t* cand, int64_t cand_cap,
                    unsigned long long* count, void* workspace, size_t ws_bytes, cudaStream_t st, bool tri,
                    int64_t q_row0) {
  const char* who = tri ? "self_join" : "range_search";
  int rc = check_planes(who, q_hi, nullptr, db_hi, nullptr, Q, N, D, ldq, lddb, idx_base, 1);
  if (rc != EMR2A_OK) return rc;
  const int64_t Dp = (static_cast<int64_t>(D) + T_BK - 1) / T_BK * T_BK;
  const bool has_fold = q_fold != nullptr;
  const bool pairs = use_cta_pairs(Q);
  const TcPlan pl = tc_plan(Q, N, 1, has_fold, pairs, 1, lddb > ldq ? lddb : ldq, 1);
  const size_t sync_off = (pl.fold_bytes + 255) & ~static_cast<size_t>(255);
  const size_t need = tri ? sync_off : sync_off + pl.sync_bytes;
  if (!workspace || ws_bytes < need) return fail(EMR2A_ERR_WORKSPACE, "%s: workspace %zu < %zu", who, ws_bytes, need);
  const bool paced = pairs && pl.sync_bytes && ws_bytes >= sync_off + pl.sync_bytes;
  uint8_t* ws = static_cast<uint8_t*>(workspace);
  CUtensorMap mq, md;
  if ((rc = make_plane_map(&mq, q_hi, Q, Dp, ldq, T_BM)) != EMR2A_OK) return rc;
  if ((rc = make_plane_map(&md, db_hi, N, Dp, lddb, pairs ? T_BN / 2 : T_BN)) != EMR2A_OK) return rc;
  TcParams p{};
  p.Q = Q; p.N = N; p.k_chunks = static_cast<int>(Dp / T_BK);
  p.m_tiles = pl.m_tiles; p.n_tiles = pl.n_tiles; p.splits = pl.splits; p.tiles_per_split = pl.tiles_per_split;
  p.idx_base = idx_base; p.K = 1;
  p.mg = pl.mg;
  if (paced) {
    p.sync_tiles = pl.sync_tiles; p.sync_points = pl.sync_points; p.sync_budget = pl.sync_budget;
    p.sync_ctr = reinterpret_cast<uint32_t*>(ws + sync_off);
    EMR2A_CUDA_TRY(cudaMemsetAsync(p.sync_ctr, 0, pl.sync_bytes, st));
  }
  if (pairs && env_int("EMR2A_TC_UNIT_CLOCK", 0) && pl.m_tiles * pl.splits <= UNIT_CLOCK_MAX) {
    void* sym = nullptr;
    EMR2A_CUDA_TRY(cudaGetSymbolAddress(&sym, g_unit_clock));
    p.unit_clock = static_cast<unsigned long long*>(sym);
    const int64_t plan[8] = {pl.m_tiles, pl.n_tiles, pl.splits, pl.tiles_per_split, pl.mg, p.sync_tiles, pl.grid,
                             pl.m_tiles * pl.splits};
    for (int i = 0; i < 8; ++i) g_last_plan[i] = plan[i];
  }
  if (has_fold) {
    EMR2A_CUDA_TRY(cudaMemsetAsync(ws, 0xFF, pl.fold_bytes, st));
    EMR2A_CUDA_TRY(cudaMemcpyAsync(ws, db_fold, static_cast<size_t>(N), cudaMemcpyDeviceToDevice, st));
    p.q_fold = q_fold; p.db_fold = ws; p.fold_sorted = fold_sorted;
  }
  p.range_t = min_score; p.D = D; p.q_stats = q_stats; p.db_stats = db_stats;
  p.range_out = reinterpret_cast<ulonglong2*>(cand); p.range_cap = cand_cap; p.range_count = count;
  if (tri) { p.self_join = 1; p.q_row0 = q_row0; p.db_row0 = idx_base; }
  tc_ev_record(0, st);
  if (pairs) rc = tc2_range_dispatch(has_fold, mq, mq, md, md, p, pl.grid, st);
  else rc = has_fold ? tc_launch<1, 8, true, true>(mq, mq, md, md, p, pl.grid, st)
                     : tc_launch<1, 8, false, true>(mq, mq, md, md, p, pl.grid, st);
  tc_ev_record(1, st);
  return rc;
}

}  // namespace emr2a
