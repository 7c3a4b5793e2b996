// K2, CTA-pair variant: the same fused similarity + Top-K kernel with tcgen05.mma.cta_group::2.
//
// Two CTAs of one cluster (one TPC) work on one 256-query x 256-row tile:
//   CTA r holds queries [128 r, 128 r + 128) (its 128 TMEM lanes) and HALF of the database tile
//   (rows [128 r, 128 r + 128)) in shared memory; the pair's tensor cores exchange the B halves,
//   so each SM fills 16 KB (A) + 16 KB (B half) per 64-wide k-chunk instead of 16 + 32 KB: one third
//   less L2->SM traffic and shared-memory bandwidth per FLOP, and room for a 6-deep smem ring.
//   Only the leader CTA (rank 0) issues MMAs; both CTAs issue their own TMA loads, which complete
//   on the LEADER's full barrier; tcgen05.commit multicasts the "slot free" and "accumulator ready"
//   arrivals to both CTAs; the peer's epilogue warps release the accumulator with a remote arrive.
// Each epilogue thread still owns one query row and sees all 256 scores of the tile, so the
// register-resident Top-K epilogue (scan_tile) is unchanged.
#include "tc_common.cuh"

namespace emr2a {

constexpr int T2_BM = 256;                       // queries per CTA pair
constexpr uint32_t T2_BH_BYTES = 128 * T_BK * 2;  // half database tile: 16 KB
// instruction descriptor: D=F32, A=B=BF16, K-major, N=256, M=256 (2 x 128)
constexpr uint32_t T2_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | ((T_BN >> 3) << 17) | ((T2_BM >> 4) << 24);

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint32_t bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t"
      "}\n" ::"r"(bar), "r"(cta) : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar_leader, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(map)), "r"(bar_leader), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(bar), "h"(static_cast<uint16_t>(3)) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}

template <int PASSES, int KCAP, bool HAS_FOLD, bool RANGE = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(T_THREADS, 1)
tc2_topk_kernel(const __grid_constant__ CUtensorMap tm_q_hi, const __grid_constant__ CUtensorMap tm_q_lo,
                const __grid_constant__ CUtensorMap tm_db_hi, const __grid_constant__ CUtensorMap tm_db_lo,
                const TcParams p) {
  constexpr int PLANES = PASSES == 3 ? 2 : 1;
  constexpr uint32_t STAGE_BYTES = PLANES * (T_A_BYTES + T2_BH_BYTES);      // per CTA
  constexpr int STAGES = PASSES == 3 ? 3 : 6;

  extern __shared__ uint8_t smem_dyn[];
  __shared__ __align__(8) uint64_t bar_full[STAGES];     // used in the leader CTA only
  __shared__ __align__(8) uint64_t bar_empty[STAGES];
  __shared__ __align__(8) uint64_t bar_tfull[2];
  __shared__ __align__(8) uint64_t bar_tempty[2];        // used in the leader CTA only (8 arrivals)
  __shared__ uint32_t tmem_base_smem;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  const uint32_t tiles_base = (smem_u32(smem_dyn) + 1023u) & ~1023u;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tm_q_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&tm_db_hi)) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) { mbar_init(smem_u32(&bar_full[s]), 1); mbar_init(smem_u32(&bar_empty[s]), 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(smem_u32(&bar_tfull[a]), 1); mbar_init(smem_u32(&bar_tempty[a]), 8); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;");
  }
  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();                      // barriers of both CTAs initialised before any remote arrive / multicast
  tcgen05_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  const int64_t n_units = p.m_tiles * p.splits;        // m_tiles counts 256-query pair tiles here
  const int64_t pair = blockIdx.x >> 1;
  const int64_t n_pairs = gridDim.x >> 1;

  if (warp == 0) {
    // ===================== TMA producer (both CTAs: own queries + own half of the database tile) =====================
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int64_t u = pair; u < n_units; u += n_pairs) {
        int64_t split, mt;
        unit_coords(p, u, split, mt);
        const int m0 = static_cast<int>(mt * T2_BM + rank * T_BM);
        const int64_t t0 = split * p.tiles_per_split;
        const int64_t t1 = (t0 + p.tiles_per_split < p.n_tiles) ? t0 + p.tiles_per_split : p.n_tiles;
        const int ufold = HAS_FOLD ? unit_fold(p, mt, T2_BM) : -1;
        int64_t slot = 0; int cohort = 1;
        if (leader && p.sync_tiles > 0) unit_cohort(p, u, n_pairs, n_units, slot, cohort);
        for (int64_t t = t0; t < t1; ++t) {
          // the leader's producer paces the pair (the peer's producer follows through the slot barriers); meeting
          // points are counted in absolute tiles so that members that skip own-fold or triangle tiles still show up
          if (leader && cohort > 1 && (t - t0) % p.sync_tiles == 0)
            cohort_sync(p, slot, static_cast<int>((t - t0) / p.sync_tiles), cohort);
          if (leader && p.unit_clock != nullptr && t == t0) {
            unsigned long long now;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
            p.unit_clock[2 * u] = now;
          }
          if ((HAS_FOLD && tile_skipped(p, ufold, t)) || tri_skipped<RANGE>(p, mt, T2_BM, t)) continue;
          const int n0 = static_cast<int>(t * T_BN + rank * 128);
          for (int kc = 0; kc < p.k_chunks; ++kc) {
            mbar_wait(smem_u32(&bar_empty[stage]), phase ^ 1u);
            const uint32_t full_leader = smem_u32(&bar_full[stage]) & 0xFEFFFFFFu;     // peer bit cleared: CTA 0's barrier
            if (leader) mbar_arrive_expect_tx(smem_u32(&bar_full[stage]), 2u * STAGE_BYTES);
            const uint32_t sb = tiles_base + stage * STAGE_BYTES;
            tma_load_2d_2sm(sb, &tm_q_hi, full_leader, kc * T_BK, m0);
            tma_load_2d_2sm(sb + PLANES * T_A_BYTES, &tm_db_hi, full_leader, kc * T_BK, n0);
            if (PASSES == 3) {
              tma_load_2d_2sm(sb + T_A_BYTES, &tm_q_lo, full_leader, kc * T_BK, m0);
              tma_load_2d_2sm(sb + PLANES * T_A_BYTES + T2_BH_BYTES, &tm_db_lo, full_leader, kc * T_BK, n0);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader && lane == 0) {
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int64_t u = pair; u < n_units; u += n_pairs) {
        int64_t split, mt;
        unit_coords(p, u, split, mt);
        const int64_t t0 = split * p.tiles_per_split;
        const int64_t t1 = (t0 + p.tiles_per_split < p.n_tiles) ? t0 + p.tiles_per_split : p.n_tiles;
        const int ufold = HAS_FOLD ? unit_fold(p, mt, T2_BM) : -1;
        for (int64_t t = t0; t < t1; ++t) {
          if ((HAS_FOLD && tile_skipped(p, ufold, t)) || tri_skipped<RANGE>(p, mt, T2_BM, t)) continue;
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
            const uint64_t b_lo = make_smem_desc(sb + PLANES * T_A_BYTES + T2_BH_BYTES);
#pragma unroll
            for (int k = 0; k < T_BK / 16; ++k) {
              const uint64_t koff = static_cast<uint64_t>((k * 32) >> 4);
              if (PASSES == 3) {
                umma_bf16_2sm(d_tmem, a_hi + koff, b_lo + koff, T2_IDESC, (kc | k) != 0 ? 1u : 0u);
                umma_bf16_2sm(d_tmem, a_lo + koff, b_hi + koff, T2_IDESC, 1u);
                umma_bf16_2sm(d_tmem, a_hi + koff, b_hi + koff, T2_IDESC, 1u);
              } else {
                umma_bf16_2sm(d_tmem, a_hi + koff, b_hi + koff, T2_IDESC, (kc | k) != 0 ? 1u : 0u);
              }
            }
            umma_commit_2sm(smem_u32(&bar_empty[stage]));      // frees the slot in BOTH CTAs
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
          }
          umma_commit_2sm(smem_u32(&bar_tfull[acc]));          // accumulator ready in BOTH CTAs
          if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
      }
    }
  } else if (warp >= 4) {
    // ===================== epilogue (both CTAs, own 128 query rows) =====================
    const int quarter = warp & 3;
    const int row = quarter * 32 + lane;
    int acc = 0; uint32_t acc_phase = 0;
    RegTopK<KCAP> top;
    float cut = 0.f;
    if constexpr (RANGE) cut = range_cut(p);
    for (int64_t u = pair; u < n_units; u += n_pairs) {
      int64_t split, mt;
      unit_coords(p, u, split, mt);
      const int64_t q = mt * T2_BM + rank * T_BM + row;
      const int64_t t0 = split * p.tiles_per_split;
      const int64_t t1 = (t0 + p.tiles_per_split < p.n_tiles) ? t0 + p.tiles_per_split : p.n_tiles;
      const uint32_t my_fold = (HAS_FOLD && q < p.Q) ? p.q_fold[q] : 0xFFFFu;
      if constexpr (!RANGE) top.reset();
      const float thr0 = RANGE ? cut : unit_start_threshold(p, q);
      float thr = thr0;
      const int ufold = HAS_FOLD ? unit_fold(p, mt, T2_BM) : -1;
      for (int64_t t = t0; t < t1; ++t) {
        if ((HAS_FOLD && tile_skipped(p, ufold, t)) || tri_skipped<RANGE>(p, mt, T2_BM, t)) continue;
        const int64_t n0 = t * T_BN;
        mbar_wait(smem_u32(&bar_tfull[acc]), acc_phase);
        tcgen05_fence_after();
        scan_tile<KCAP, HAS_FOLD, RANGE>(p, top, thr, thr0,
                                         tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + static_cast<uint32_t>(acc * T_BN),
                                         n0, my_fold, q);
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (leader) mbar_arrive(smem_u32(&bar_tempty[acc]));
          else mbar_arrive_remote(smem_u32(&bar_tempty[acc]), 0);
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      if (!RANGE && q < p.Q) {
        if (p.tau != nullptr && top.i[KCAP - 1] != 0xFFFFFFFFu) atomicMax(p.tau + q, order_f32(top.s[KCAP - 1]));
        uint64_t* dst = p.keys_out + (split * p.Q + q) * p.K;
#pragma unroll
        for (int j = 0; j < KCAP; ++j)
          if (j < p.K) dst[j] = (top.i[j] == 0xFFFFFFFFu) ? 0ull : pack_key(top.s[j], top.i[j]);
      }
      if (leader && p.unit_clock != nullptr && threadIdx.x == 128) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
        p.unit_clock[2 * u + 1] = now;
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  cluster_sync_all();                      // no CTA leaves (or frees TMEM) while its peer may still touch it
  if (warp == 2) {
    tcgen05_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

template <int PASSES, int KCAP, bool HAS_FOLD, bool RANGE = false>
static int tc2_launch(const CUtensorMap& mq_hi, const CUtensorMap& mq_lo, const CUtensorMap& md_hi, const CUtensorMap& md_lo,
                      const TcParams& p, int grid, cudaStream_t st) {
  constexpr int PLANES = PASSES == 3 ? 2 : 1;
  constexpr int STAGES = PASSES == 3 ? 3 : 6;
  const size_t smem = static_cast<size_t>(STAGES) * PLANES * (T_A_BYTES + T2_BH_BYTES) + 1024;
  auto kern = tc2_topk_kernel<PASSES, KCAP, HAS_FOLD, RANGE>;
  EMR2A_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem)));
  kern<<<grid, T_THREADS, smem, st>>>(mq_hi, mq_lo, md_hi, md_lo, p);
  EMR2A_LAUNCH_CHECK("tc2_topk_kernel");
  return EMR2A_OK;
}

// dispatch over (passes, kcap, fold)
int tc2_dispatch(int passes, int kcap, bool has_fold, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c,
                 const CUtensorMap& d, const TcParams& p, int grid, cudaStream_t st) {
#define EMR2A_TC2_CASE(P, KC)                                                                  \
  if (passes == P && kcap == KC)                                                              \
    return has_fold ? tc2_launch<P, KC, true>(a, b, c, d, p, grid, st) : tc2_launch<P, KC, false>(a, b, c, d, p, grid, st);
  EMR2A_TC2_CASE(1, 8) EMR2A_TC2_CASE(1, 16) EMR2A_TC2_CASE(1, 32)
  EMR2A_TC2_CASE(3, 8) EMR2A_TC2_CASE(3, 16) EMR2A_TC2_CASE(3, 32)
#undef EMR2A_TC2_CASE
  return fail(EMR2A_ERR_INVALID, "tc2_dispatch: unsupported (passes=%d, kcap=%d)", passes, kcap);
}

// range epilogue (emr2a_range_search): the 1-pass filter, no register list
int tc2_range_dispatch(bool has_fold, const CUtensorMap& a, const CUtensorMap& b, const CUtensorMap& c,
                       const CUtensorMap& d, const TcParams& p, int grid, cudaStream_t st) {
  return has_fold ? tc2_launch<1, 8, true, true>(a, b, c, d, p, grid, st) : tc2_launch<1, 8, false, true>(a, b, c, d, p, grid, st);
}

}  // namespace emr2a
