// C-ABI glue: error text, device check, emr2a_topk_search dispatch.
#include "common.cuh"

#include <math.h>
#include <stdlib.h>
#include <string.h>

namespace emr2a {

static thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
int cuda_fail(cudaError_t e, const char* where) {
  snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) at %s", static_cast<int>(e), cudaGetErrorString(e), where);
  cudaGetLastError();
  return EMR2A_ERR_CUDA;
}
int sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
  return n;
}

// implemented in simt_paths.cu / topk_tc.cu
size_t simt_topk_workspace_bytes(int64_t Q, int64_t N, int K);
int simt_topk_search(const float* q, const float* db, int64_t Q, int64_t N, int D, int64_t ldq, int64_t lddb,
                     const uint8_t* q_fold, const uint8_t* db_fold, int64_t idx_base, int K, uint64_t* out_keys,
                     void* workspace, size_t ws_bytes, cudaStream_t st);
size_t tc_topk_workspace_bytes(int64_t Q, int64_t N, int K, int D);
int tc_debug_unit_clocks(unsigned long long* host_out, int64_t cap_units, int64_t* plan_out);
struct TcPartials {
  const uint64_t* parts;
  int splits;
  const uint32_t* tau;
};
int tc_topk_search(const uint16_t* q_hi, const uint16_t* q_lo, const uint16_t* db_hi, const uint16_t* db_lo,
                   int64_t Q, int64_t N, int D, int64_t ldq, int64_t lddb, const uint8_t* q_fold,
                   const uint8_t* db_fold, int64_t idx_base, int K, int passes, uint64_t* out_keys,
                   void* workspace, size_t ws_bytes, float* debug_scores, cudaStream_t st, TcPartials* partials,
                   int fold_sorted, int min_splits);
int tc_planned_splits(int64_t Q, int64_t N, int min_splits);
int tc_timing_enable(int on);
int tc_timing_read(float* ms_out, int cap, int* n_out);
void tc_timing_record(int which, cudaStream_t st);
int tc_range_filter(const uint16_t* q_hi, const uint16_t* db_hi, int64_t Q, int64_t N, int D, int64_t ldq, int64_t lddb,
                    const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted, int64_t idx_base, float min_score,
                    const float* q_stats, const float* db_stats, uint64_t* cand, int64_t cand_cap,
                    unsigned long long* count, void* workspace, size_t ws_bytes, cudaStream_t st, bool tri,
                    int64_t q_row0);

size_t rescore_workspace_bytes(int64_t Q, int K);
int rescore_pipeline(const uint64_t* approx, int KP, const uint32_t* tau, const float* q, int64_t ldq, const float* db,
                     int64_t lddb, const emr2a_lazy_rows* db_lazy, const uint16_t* db_hi, int64_t lddb_hi, int64_t Q, int64_t N,
                     int D, int64_t idx_base, int K,
                     const float* q_stats, const float* db_stats, const uint8_t* q_fold, const uint8_t* db_fold,
                     uint64_t* out_keys, int* status, uint8_t* qflags, void* workspace, size_t ws_bytes, cudaStream_t st);

int rescore_kth_scores(const uint64_t* approx, int KP, int K, int64_t Q, float* kth, cudaStream_t st);
int rescore_select_only(const uint64_t* approx, int KP, const uint32_t* tau, const float* kth_floor, const float* q,
                        int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int64_t Q, int64_t N, int D,
                        int64_t idx_base, int K, const float* q_stats, const float* db_stats, uint64_t* out_keys,
                        float* bound_out, cudaStream_t st);
int rescore_verify_merged(const uint64_t* keys, int K, int64_t Q, const float* bounds, int parts, int64_t bounds_stride,
                          uint8_t* flags, int* count, cudaStream_t st);
size_t exact_rescan_workspace_bytes(int n_flagged, int K);
int rescore_exact_rescan(const float* q, int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int64_t N,
                         int D, int64_t idx_base, int K, const uint8_t* q_fold, const uint8_t* db_fold, const int* flag_list,
                         int n_flagged, uint64_t* out_compact, void* workspace, size_t ws_bytes, const uint16_t* db_hi,
                         int64_t lddb_hi, const float* q_stats, const float* db_stats, const uint64_t* seed_keys,
                         cudaStream_t st);

int range_refine_check(const float* q, int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int D);
int range_refine(const uint64_t* cand, int64_t cand_cap, unsigned long long* counts, uint64_t* out, int64_t out_cap,
                 const float* q, int64_t ldq, const float* db, int64_t lddb, const emr2a_lazy_rows* db_lazy, int D,
                 int64_t idx_base, float min_score, cudaStream_t st);

constexpr int RESCORE_KP = 32;    // candidates kept per (query, database split) by the filter; 16 leaves too little slack (measured)
constexpr int RESCORE_KPM = 64;   // candidates per query re-scored after merging the splits
static inline size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

__global__ void zero_keys_kernel(uint64_t* k, int64_t n) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) k[i] = 0ull;
}

// the key lists of an empty database: n empty keys
static int zero_keys(uint64_t* k, int64_t n, cudaStream_t st) {
  zero_keys_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, st>>>(k, n);
  EMR2A_LAUNCH_CHECK("zero_keys_kernel");
  return EMR2A_OK;
}

}  // namespace emr2a

using namespace emr2a;

extern "C" int emr2a_abi_version(void) { return EMR2A_ABI_VERSION; }
extern "C" const char* emr2a_last_error(void) { return g_err; }

extern "C" int emr2a_device_check(int* sms, int* cc_major, int* cc_minor) {
  int dev = 0;
  EMR2A_CUDA_TRY(cudaGetDevice(&dev));
  int major = 0, minor = 0, n = 0;
  EMR2A_CUDA_TRY(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  EMR2A_CUDA_TRY(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  EMR2A_CUDA_TRY(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  if (sms) *sms = n;
  if (cc_major) *cc_major = major;
  if (cc_minor) *cc_minor = minor;
  if (major != 10) return fail(EMR2A_ERR_UNSUPPORTED, "libemr2a is built for sm_100a only; device is sm_%d%d", major, minor);
  return EMR2A_OK;
}

extern "C" size_t emr2a_topk_search_workspace_bytes(int64_t Q, int64_t N, int D, int K, int precision) {
  if (Q <= 0 || N <= 0 || K <= 0) return 256;
  if (precision == EMR2A_PREC_FP32) return simt_topk_workspace_bytes(Q, N, K) + 256;
  if (precision == EMR2A_PREC_BF16_RESCORE) {
    return align256(sizeof(uint64_t) * static_cast<size_t>(Q) * RESCORE_KPM) +
           align256(tc_topk_workspace_bytes(Q, N, RESCORE_KP, D)) + align256(rescore_workspace_bytes(Q, K));
  }
  return tc_topk_workspace_bytes(Q, N, K, D);
}

// Filter stage of the RESCORE arm: 1-pass tensor-core search keeping kp candidates per (query, database split), merged
// to the RESCORE_KPM best per query.  *cand -> [Q][*kpm] approximate keys (in `approx` or in the workspace), *tau -> [Q]
// bound on the filter score of the rows no split kept (may be null: a single split whose list is all there is).
static int rescore_filter_stage(const uint16_t* q_hi, int64_t ldq_bf16, const uint16_t* db_hi, int64_t lddb_bf16, int64_t Q,
                                int64_t N, int D, const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted,
                                int64_t idx_base, int K, uint64_t* approx, void* tc_ws, size_t tc_ws_bytes,
                                float* debug_scores, cudaStream_t st, const uint64_t** cand, int* kpm,
                                const uint32_t** tau) {
  TcPartials parts{};
  // At least two splits so that the merged candidates of several lists back the verification; with >= 8
  // splits (or K <= 5) each split only keeps 16 (rows it drops are bounded by tau), which halves the
  // epilogue's insertion work.
  // A single-tile batch on single CTAs gets one split per SM (148): 8 rows per split are 1184 candidates, more than
  // the 64 that are re-scored, and keep the merge within its 2048-key register variant.
  const int planned = tc_planned_splits(Q, N, 2);
  int kp = planned > 128 ? 8 : ((planned >= 8 || K <= 5) ? 16 : RESCORE_KP);
  {   // experiments: EMR2A_RESCORE_KP = 8 / 16 / 32 overrides the list width per split
    const char* e = getenv("EMR2A_RESCORE_KP");
    const int v = (e && *e) ? atoi(e) : 0;
    if (v == 8 || v == 16 || v == 32) kp = v;
  }
  int rc = tc_topk_search(q_hi, nullptr, db_hi, nullptr, Q, N, D, ldq_bf16, lddb_bf16, q_fold, db_fold, idx_base,
                          kp, 1, nullptr, tc_ws, tc_ws_bytes, debug_scores, st, &parts, fold_sorted, 2);
  if (rc != EMR2A_OK) return rc;
  // several splits: re-score the 64 best approximate candidates of the query (rows outside the per-split
  // lists are bounded by tau); one split: its candidates are all there is
  *kpm = kp;
  *cand = parts.parts;
  *tau = parts.tau;
  if (parts.splits > 1) {
    *kpm = RESCORE_KPM;
    rc = emr2a_topk_merge(parts.parts, parts.splits, Q, kp, Q * kp, kp, RESCORE_KPM, approx, st);
    if (rc != EMR2A_OK) return rc;
    *cand = approx;
  }
  return EMR2A_OK;
}

static int topk_search_impl(const float* q_f32, int64_t ldq_f32, const uint16_t* q_hi, const uint16_t* q_lo,
                            int64_t ldq_bf16, const float* db_f32, int64_t lddb_f32, const uint16_t* db_hi,
                            const uint16_t* db_lo, int64_t lddb_bf16, int64_t Q, int64_t N, int D,
                            const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted, int64_t idx_base, int K,
                            int precision, const float* q_stats, const float* db_stats, uint64_t* out_keys,
                            int32_t* status, uint8_t* qflags, void* workspace, size_t ws_bytes, float* debug_scores,
                            const emr2a_lazy_rows* db_lazy, void* stream) {
  if (Q < 0 || N < 0 || D <= 0 || K <= 0 || !out_keys) return fail(EMR2A_ERR_INVALID, "topk_search: bad arguments (Q=%lld N=%lld D=%d K=%d)", (long long)Q, (long long)N, D, K);
  if ((q_fold == nullptr) != (db_fold == nullptr)) return fail(EMR2A_ERR_INVALID, "topk_search: q_fold and db_fold must be given together");
  if (idx_base < 0) return fail(EMR2A_ERR_INVALID, "topk_search: negative idx_base");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (Q == 0) return EMR2A_OK;
  if (N == 0) return zero_keys(out_keys, Q * K, st);
  switch (precision) {
    case EMR2A_PREC_FP32:
      if (!q_f32 || !db_f32) return fail(EMR2A_ERR_INVALID, "topk_search(fp32): q_f32/db_f32 required");
      if (ldq_f32 < D || lddb_f32 < D) return fail(EMR2A_ERR_INVALID, "topk_search(fp32): leading dimension smaller than D");
      return simt_topk_search(q_f32, db_f32, Q, N, D, ldq_f32, lddb_f32, q_fold, db_fold, idx_base, K, out_keys, workspace, ws_bytes, st);
    case EMR2A_PREC_BF16X3:
      return tc_topk_search(q_hi, q_lo, db_hi, db_lo, Q, N, D, ldq_bf16, lddb_bf16, q_fold, db_fold, idx_base, K, 3, out_keys, workspace, ws_bytes, debug_scores, st, nullptr, fold_sorted, 1);
    case EMR2A_PREC_BF16X1:
      return tc_topk_search(q_hi, nullptr, db_hi, nullptr, Q, N, D, ldq_bf16, lddb_bf16, q_fold, db_fold, idx_base, K, 1, out_keys, workspace, ws_bytes, debug_scores, st, nullptr, fold_sorted, 1);
    case EMR2A_PREC_BF16_RESCORE: {
      if (K > 10) return fail(EMR2A_ERR_UNSUPPORTED, "topk_search(rescore): K=%d > 10 (use EMR2A_PREC_BF16X3)", K);
      if (!q_f32 || (!db_f32 && !db_lazy)) return fail(EMR2A_ERR_INVALID, "topk_search(rescore): q_f32 and db_f32 (or db_lazy) required");
      if (ldq_f32 < D || (!db_lazy && lddb_f32 < D)) return fail(EMR2A_ERR_INVALID, "topk_search(rescore): leading dimension smaller than D");
      if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return fail(EMR2A_ERR_INVALID, "topk_search(rescore): workspace must be 256-byte aligned");
      const size_t a_bytes = align256(sizeof(uint64_t) * static_cast<size_t>(Q) * RESCORE_KPM);
      const size_t t_bytes = align256(tc_topk_workspace_bytes(Q, N, RESCORE_KP, D));
      const size_t r_bytes = align256(rescore_workspace_bytes(Q, K));
      if (ws_bytes < a_bytes + t_bytes + r_bytes) return fail(EMR2A_ERR_WORKSPACE, "topk_search(rescore): workspace %zu < %zu", ws_bytes, a_bytes + t_bytes + r_bytes);
      uint8_t* ws = static_cast<uint8_t*>(workspace);
      const uint64_t* cand = nullptr;
      const uint32_t* tau = nullptr;
      int kpm = 0;
      int rc = rescore_filter_stage(q_hi, ldq_bf16, db_hi, lddb_bf16, Q, N, D, q_fold, db_fold, fold_sorted, idx_base, K,
                                    reinterpret_cast<uint64_t*>(ws), ws + a_bytes, t_bytes, debug_scores, st, &cand, &kpm, &tau);
      if (rc != EMR2A_OK) return rc;
      return rescore_pipeline(cand, kpm, tau, q_f32, ldq_f32, db_f32, lddb_f32, db_lazy, db_hi, lddb_bf16, Q, N, D, idx_base, K, q_stats,
                              db_stats, q_fold, db_fold, out_keys, status, qflags, ws + a_bytes + t_bytes, r_bytes, st);
    }
    default:
      return fail(EMR2A_ERR_INVALID, "topk_search: unknown precision %d", precision);
  }
}

extern "C" int emr2a_topk_search(const float* q_f32, int64_t ldq_f32, const uint16_t* q_hi, const uint16_t* q_lo,
                                 int64_t ldq_bf16, const float* db_f32, int64_t lddb_f32, const uint16_t* db_hi,
                                 const uint16_t* db_lo, int64_t lddb_bf16, int64_t Q, int64_t N, int D,
                                 const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted, int64_t idx_base,
                                 int K, int precision, const float* q_stats, const float* db_stats,
                                 uint64_t* out_keys, int32_t* status_out, uint8_t* unverified_out, void* workspace,
                                 size_t ws_bytes, const emr2a_lazy_rows* db_lazy, void* stream) {
  if (db_lazy && precision != EMR2A_PREC_BF16_RESCORE) return fail(EMR2A_ERR_INVALID, "topk_search: db_lazy is for EMR2A_PREC_BF16_RESCORE only");
  return topk_search_impl(q_f32, ldq_f32, q_hi, q_lo, ldq_bf16, db_f32, lddb_f32, db_hi, db_lo, lddb_bf16, Q, N, D,
                          q_fold, db_fold, fold_sorted, idx_base, K, precision, q_stats, db_stats, out_keys,
                          status_out, unverified_out, workspace, ws_bytes, nullptr, db_lazy, stream);
}

// Diagnostics: same as emr2a_topk_search on the tensor-core arms, additionally dumping every
// score the epilogue saw to debug_scores [Q, N] (tests compare the GEMM itself with the oracle).
extern "C" int emr2a_debug_topk_search_dump(const uint16_t* q_hi, const uint16_t* q_lo, const uint16_t* db_hi,
                                            const uint16_t* db_lo, int64_t Q, int64_t N, int D, int64_t ldq,
                                            int64_t lddb, const uint8_t* q_fold, const uint8_t* db_fold,
                                            int64_t idx_base, int K, int precision, uint64_t* out_keys,
                                            void* workspace, size_t ws_bytes, float* debug_scores, void* stream) {
  if (precision != EMR2A_PREC_BF16X3 && precision != EMR2A_PREC_BF16X1)
    return fail(EMR2A_ERR_INVALID, "debug dump is for the tensor-core arms only");
  return topk_search_impl(nullptr, 0, q_hi, q_lo, ldq, nullptr, 0, db_hi, db_lo, lddb, Q, N, D, q_fold, db_fold, 0,
                          idx_base, K, precision, nullptr, nullptr, out_keys, nullptr, nullptr, workspace, ws_bytes,
                          debug_scores, nullptr, stream);
}

// Diagnostics: globaltimer stamps (start, end) of every work unit of the last CTA-pair launch made with
// EMR2A_TC_UNIT_CLOCK=1, plus its plan {m_tiles, n_tiles, splits, tiles_per_split, mg, sync_tiles, grid, n_units}.
extern "C" int emr2a_debug_unit_clocks(uint64_t* host_out, int64_t cap_units, int64_t* plan_out) {
  if (!host_out || !plan_out) return fail(EMR2A_ERR_INVALID, "debug_unit_clocks: null output");
  return tc_debug_unit_clocks(reinterpret_cast<unsigned long long*>(host_out), cap_units, plan_out);
}

// ---- cooperative shards: the RESCORE arm in stages, so that row shards verify ONE merged selection -------------------
extern "C" size_t emr2a_topk_filter_workspace_bytes(int64_t Q, int64_t N, int D, int K) {
  if (Q <= 0 || N <= 0 || K <= 0) return 256;
  return align256(tc_topk_workspace_bytes(Q, N, RESCORE_KP, D));
}

extern "C" int emr2a_topk_filter(const uint16_t* q_hi, int64_t ldq_bf16, const uint16_t* db_hi, int64_t lddb_bf16, int64_t Q,
                                 int64_t N, int D, const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted,
                                 int64_t idx_base, int K, uint64_t* cand_out, uint32_t* tau_out, float* kth_out,
                                 void* workspace, size_t ws_bytes, void* stream) {
  if (Q < 0 || N < 0 || D <= 0 || K <= 0 || !cand_out || !tau_out) return fail(EMR2A_ERR_INVALID, "topk_filter: bad arguments");
  if (K > 10) return fail(EMR2A_ERR_UNSUPPORTED, "topk_filter: K=%d > 10 (use EMR2A_PREC_BF16X3)", K);
  if ((q_fold == nullptr) != (db_fold == nullptr)) return fail(EMR2A_ERR_INVALID, "topk_filter: q_fold and db_fold must be given together");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (Q == 0) return EMR2A_OK;
  EMR2A_CUDA_TRY(cudaMemsetAsync(tau_out, 0, sizeof(uint32_t) * static_cast<size_t>(Q), st));
  if (N == 0) {
    const int rc = zero_keys(cand_out, Q * RESCORE_KPM, st);
    if (rc != EMR2A_OK) return rc;
  } else {
    if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return fail(EMR2A_ERR_INVALID, "topk_filter: workspace must be 256-byte aligned");
    const uint64_t* cand = nullptr;
    const uint32_t* tau = nullptr;
    int kpm = 0;
    int rc = rescore_filter_stage(q_hi, ldq_bf16, db_hi, lddb_bf16, Q, N, D, q_fold, db_fold, fold_sorted, idx_base, K,
                                  cand_out, workspace, ws_bytes, nullptr, st, &cand, &kpm, &tau);
    if (rc != EMR2A_OK) return rc;
    if (cand != cand_out) {      // a single split: pad its list to the fixed candidate width
      rc = emr2a_topk_merge(cand, 1, Q, kpm, Q * kpm, kpm, RESCORE_KPM, cand_out, st);
      if (rc != EMR2A_OK) return rc;
    }
    if (tau) EMR2A_CUDA_TRY(cudaMemcpyAsync(tau_out, tau, sizeof(uint32_t) * static_cast<size_t>(Q), cudaMemcpyDeviceToDevice, st));
  }
  if (kth_out) return rescore_kth_scores(cand_out, RESCORE_KPM, K, Q, kth_out, st);
  return EMR2A_OK;
}

extern "C" int emr2a_rescore_candidates(const uint64_t* cand, const uint32_t* tau, const float* kth_floor, const float* q_f32,
                                        int64_t ldq_f32, const float* db_f32, int64_t lddb_f32, int64_t Q, int64_t N, int D,
                                        int64_t idx_base, int K, const float* q_stats, const float* db_stats,
                                        uint64_t* out_keys, float* bound_out, const emr2a_lazy_rows* db_lazy,
                                        void* stream) {
  if (!cand || !tau || !q_f32 || (!db_f32 && !db_lazy) || !q_stats || !db_stats || !out_keys || !bound_out || Q < 0 || N < 0 ||
      D <= 0 || K <= 0 || K > 10 || ldq_f32 < D || (!db_lazy && lddb_f32 < D))
    return fail(EMR2A_ERR_INVALID, "rescore_candidates: bad arguments");
  if (Q == 0) return EMR2A_OK;
  return rescore_select_only(cand, RESCORE_KPM, tau, kth_floor, q_f32, ldq_f32, db_f32, lddb_f32, db_lazy, Q, N, D, idx_base,
                             K, q_stats, db_stats, out_keys, bound_out, static_cast<cudaStream_t>(stream));
}

extern "C" int emr2a_verify_merged(const uint64_t* keys, int K, int64_t Q, const float* bounds, int parts,
                                   int64_t bounds_stride, uint8_t* flags_out, int32_t* status_out, void* stream) {
  if (!keys || !bounds || !flags_out || !status_out || K <= 0 || Q < 0 || parts <= 0 || bounds_stride < Q)
    return fail(EMR2A_ERR_INVALID, "verify_merged: bad arguments");
  if (Q == 0) return EMR2A_OK;
  return rescore_verify_merged(keys, K, Q, bounds, parts, bounds_stride, flags_out, status_out, static_cast<cudaStream_t>(stream));
}

extern "C" size_t emr2a_exact_rescan_workspace_bytes(int n_flagged, int K) { return exact_rescan_workspace_bytes(n_flagged, K) + 256; }

extern "C" int emr2a_exact_rescan(const float* q_f32, int64_t ldq_f32, const float* db_f32, int64_t lddb_f32, int64_t N, int D,
                                  int64_t idx_base, int K, const uint8_t* q_fold, const uint8_t* db_fold,
                                  const int32_t* flag_list, int n_flagged, uint64_t* out_keys, void* workspace,
                                  size_t ws_bytes, const emr2a_lazy_rows* db_lazy, const uint16_t* db_hi,
                                  int64_t lddb_bf16, const float* q_stats, const float* db_stats,
                                  const uint64_t* seed_keys, void* stream) {
  if (!q_f32 || (!db_f32 && !db_lazy && N > 0) || !out_keys || N < 0 || D <= 0 || K <= 0 || n_flagged < 0 || ldq_f32 < D ||
      (!db_lazy && N > 0 && lddb_f32 < D) || (n_flagged > 0 && !flag_list))
    return fail(EMR2A_ERR_INVALID, "exact_rescan: bad arguments");
  if ((q_fold == nullptr) != (db_fold == nullptr)) return fail(EMR2A_ERR_INVALID, "exact_rescan: q_fold and db_fold must be given together");
  if (n_flagged == 0) return EMR2A_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (N == 0) return zero_keys(out_keys, static_cast<int64_t>(n_flagged) * K, st);
  return rescore_exact_rescan(q_f32, ldq_f32, db_f32, lddb_f32, db_lazy, N, D, idx_base, K, q_fold, db_fold, flag_list,
                              n_flagged, out_keys, workspace, ws_bytes, db_hi, lddb_bf16, q_stats, db_stats, seed_keys, st);
}

// The tensor-core filter of a range search or self-join, then range_refine of its candidates.  The kernel timing ring
// gets two entries: the filter (tc_range_filter records it around its launch) and the refine kernel.
template <class Filter, class Refine>
static int filter_then_refine(Filter filter, Refine refine, cudaStream_t st) {
  int rc = filter();
  if (rc != EMR2A_OK) return rc;
  tc_timing_record(0, st);
  rc = refine();
  tc_timing_record(1, st);
  return rc;
}

// ---- range search: every admissible pair with exact score >= min_score --------------------------------------------
extern "C" size_t emr2a_range_search_workspace_bytes(int64_t Q, int64_t N, int D) {
  if (Q <= 0 || N <= 0 || D <= 0) return 256;
  return align256(tc_topk_workspace_bytes(Q, N, 1, D));
}

extern "C" int emr2a_range_search(const float* q_f32, int64_t ldq_f32, const uint16_t* q_hi, int64_t ldq_bf16,
                                  const float* db_f32, int64_t lddb_f32, const uint16_t* db_hi, int64_t lddb_bf16,
                                  int64_t Q, int64_t N, int D, const uint8_t* q_fold, const uint8_t* db_fold,
                                  int fold_sorted, int64_t idx_base, float min_score, const float* q_stats,
                                  const float* db_stats, uint64_t* cand, int64_t cand_cap, uint64_t* results,
                                  int64_t result_cap, uint64_t* counts_out, void* workspace, size_t ws_bytes,
                                  const emr2a_lazy_rows* db_lazy, void* stream) {
  if (Q < 0 || N < 0 || D <= 0 || cand_cap < 0 || result_cap < 0 || !counts_out || (cand_cap > 0 && !cand) ||
      (result_cap > 0 && !results))
    return fail(EMR2A_ERR_INVALID, "range_search: bad arguments (Q=%lld N=%lld D=%d)", (long long)Q, (long long)N, D);
  if (!isfinite(min_score)) return fail(EMR2A_ERR_INVALID, "range_search: min_score must be finite");
  if ((q_fold == nullptr) != (db_fold == nullptr)) return fail(EMR2A_ERR_INVALID, "range_search: q_fold and db_fold must be given together");
  if (idx_base < 0) return fail(EMR2A_ERR_INVALID, "range_search: negative idx_base");
  if (!q_f32 || (!db_f32 && !db_lazy) || !q_stats || !db_stats)
    return fail(EMR2A_ERR_INVALID, "range_search: q_f32, db_f32 (or db_lazy), q_stats and db_stats required");
  if (ldq_f32 < D || (!db_lazy && lddb_f32 < D)) return fail(EMR2A_ERR_INVALID, "range_search: leading dimension smaller than D");
  if (Q == 0 || N == 0) return EMR2A_OK;
  if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return fail(EMR2A_ERR_INVALID, "range_search: workspace must be 256-byte aligned");
  // the refine stage's operand rules are checked before anything is launched: an error leaves the outputs untouched
  int rc = range_refine_check(q_f32, ldq_f32, db_f32, lddb_f32, db_lazy, D);
  if (rc != EMR2A_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(counts_out);
  return filter_then_refine(
      [&] { return tc_range_filter(q_hi, db_hi, Q, N, D, ldq_bf16, lddb_bf16, q_fold, db_fold, fold_sorted, idx_base,
                                   min_score, q_stats, db_stats, cand, cand_cap, counts, workspace, ws_bytes, st, false, 0); },
      [&] { return range_refine(cand, cand_cap, counts, results, result_cap, q_f32, ldq_f32, db_f32, lddb_f32, db_lazy, D,
                                idx_base, min_score, st); },
      st);
}

// ---- self-join: every pair i < j of one row set with exact score >= min_score ----------------------------------------
extern "C" size_t emr2a_self_join_workspace_bytes(int64_t n, int D) {
  return emr2a_range_search_workspace_bytes(n, n, D);      // fold padding of [0, n) and the counters of the band [0, n)
}

extern "C" int emr2a_self_join(const float* x_f32, int64_t ld_f32, const uint16_t* x_hi, int64_t ld_bf16, int64_t n, int D,
                               int64_t q_begin, int64_t q_end, const uint8_t* fold, int fold_sorted, float min_score,
                               const float* stats, uint64_t* cand, int64_t cand_cap, uint64_t* results,
                               int64_t result_cap, uint64_t* counts_out, void* workspace, size_t ws_bytes, void* stream) {
  if (n < 0 || D <= 0 || cand_cap < 0 || result_cap < 0 || !counts_out || (cand_cap > 0 && !cand) ||
      (result_cap > 0 && !results))
    return fail(EMR2A_ERR_INVALID, "self_join: bad arguments (n=%lld D=%d)", (long long)n, D);
  if (q_begin < 0 || q_begin > q_end || q_end > n)
    return fail(EMR2A_ERR_INVALID, "self_join: need 0 <= q_begin <= q_end <= n (q_begin=%lld q_end=%lld n=%lld)",
                (long long)q_begin, (long long)q_end, (long long)n);
  if (!isfinite(min_score)) return fail(EMR2A_ERR_INVALID, "self_join: min_score must be finite");
  if (!x_f32 || !x_hi || !stats) return fail(EMR2A_ERR_INVALID, "self_join: x_f32, x_hi and stats required");
  if (ld_f32 < D) return fail(EMR2A_ERR_INVALID, "self_join: leading dimension smaller than D");
  if (q_begin == q_end) return EMR2A_OK;
  if (!workspace || (reinterpret_cast<uintptr_t>(workspace) & 255)) return fail(EMR2A_ERR_INVALID, "self_join: workspace must be 256-byte aligned");
  int rc = range_refine_check(x_f32, ld_f32, x_f32, ld_f32, nullptr, D);
  if (rc != EMR2A_OK) return rc;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  unsigned long long* counts = reinterpret_cast<unsigned long long*>(counts_out);
  // queries [q_begin, q_end) against rows [q_begin, n): no row below q_begin is a partner j > i of these queries
  const uint16_t* band = x_hi + q_begin * ld_bf16;
  const uint8_t* band_fold = fold ? fold + q_begin : nullptr;
  // candidates carry global rows on both sides: re-scored against the whole row set
  return filter_then_refine(
      [&] { return tc_range_filter(band, band, q_end - q_begin, n - q_begin, D, ld_bf16, ld_bf16, band_fold, band_fold,
                                   fold_sorted, q_begin, min_score, stats, stats, cand, cand_cap, counts, workspace,
                                   ws_bytes, st, true, q_begin); },
      [&] { return range_refine(cand, cand_cap, counts, results, result_cap, x_f32, ld_f32, x_f32, ld_f32, nullptr, D, 0,
                                min_score, st); },
      st);
}

// Diagnostics: time the Top-K kernel of every search alone (CUDA events on the launching stream around its launch).
// A range search (emr2a_range_search) or a self-join (emr2a_self_join) adds two entries: its filter kernel, then its
// refine kernel.
// enable != 0 starts a fresh series; emr2a_debug_tc_elapsed waits for the timed launches and returns their durations
// (milliseconds, HOST array, oldest first, the last `cap` at most).
extern "C" int emr2a_debug_tc_timing(int enable) { return tc_timing_enable(enable); }
extern "C" int emr2a_debug_tc_elapsed(float* ms_out_host, int cap, int* n_out_host) {
  if (!ms_out_host || !n_out_host || cap <= 0) return fail(EMR2A_ERR_INVALID, "debug_tc_elapsed: bad arguments");
  return tc_timing_read(ms_out_host, cap, n_out_host);
}
