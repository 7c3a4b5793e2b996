/*
 * emr2a.h -- C-ABI of libemr2a.so: the B200 (sm_100a) retrieval hot path of EMR2A.
 *
 * The reference (Ali-Xiyao/emr2a-evidence-grounded-multimodal-retrieval) has no
 * FFI of its own: the path sits behind plain Python modules.  These entry
 * points are what the same-named Python modules shipped in this repository
 * (emr2a_b200/retrieval, emr2a_b200/utils) bind with ctypes; each one cites the
 * reference code it replaces.  Plain pointers and sizes only -- no torch types.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *     all work is stream-ordered, no call synchronises the device or allocates;
 *   - scratch memory is passed in (`workspace`), its size comes from the matching
 *     *_workspace_bytes query;
 *   - return value: EMR2A_OK or an error code; emr2a_last_error() gives the text
 *     (thread-local);
 *   - leading dimensions (`ld*`) are in ELEMENTS of the array they describe.
 *
 * Packed Top-K key (uint64), larger == better:
 *      bits 63..32  order-preserving image of the fp32 score
 *                   (b ^ 0x80000000 for b >= 0, ~b for negative floats)
 *      bits 31..0   0xFFFFFFFF - global database row index
 *   so sorting keys descending gives (score descending, index ascending): the
 *   deterministic tie rule that replaces np.argsort's unspecified order
 *   (utils/cv_evaluator.py:123).  Key 0 means "empty slot".
 */
#ifndef EMR2A_H
#define EMR2A_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EMR2A_ABI_VERSION 13

enum emr2a_status {
  EMR2A_OK = 0,
  EMR2A_ERR_INVALID = 1,      /* bad argument (maps to ValueError in the Python layer) */
  EMR2A_ERR_CUDA = 2,         /* a CUDA runtime / driver call failed */
  EMR2A_ERR_UNSUPPORTED = 3,  /* shape / mode not supported by the requested precision path */
  EMR2A_ERR_WORKSPACE = 4     /* workspace too small */
};

enum emr2a_dtype { EMR2A_F32 = 0, EMR2A_BF16 = 1 };

/* flags of emr2a_normalize_fuse */
enum emr2a_nf_flags {
  EMR2A_NF_SEGNORM = 1,     /* first scale each segment to unit length: x / (||x|| + 1e-8) */
  EMR2A_NF_ROWNORM = 2,     /* after weighting + concatenation divide the row by (||row|| + 1e-8) */
  EMR2A_NF_ZERO_GUARD = 4,  /* ROWNORM without epsilon, zero rows stay zero (utils/common.py:4-8) */
  EMR2A_NF_STANDARDIZE = 8  /* first apply the fitted StandardScaler per column, (x - mean) / scale in IEEE fp32
                               (utils/cv_evaluator.py:78-80, retrieval/evaluator.py:55-57), from col_std: the per-fold
                               scaler and the row normalisation are ONE pass over the raw rows */
};

/* arithmetic of emr2a_topk_search */
enum emr2a_precision {
  EMR2A_PREC_FP32 = 0,      /* fp32 FMA on CUDA cores: exact-order reference arithmetic, any shape */
  EMR2A_PREC_BF16X3 = 1,    /* tcgen05 bf16 tensor cores, 2-way split (hi*hi + hi*lo + lo*hi), fp32 accumulate: |err| ~ 1e-6 */
  EMR2A_PREC_BF16X1 = 2,    /* tcgen05 bf16 tensor cores, hi plane only (bf16-input variant), fp32 accumulate */
  EMR2A_PREC_BF16_RESCORE = 3 /* 1-pass bf16 tensor-core FILTER (16 or 32 candidates per query and database split, the
                                 64 best after merging), exact fp32 RE-SCORING of the candidates from the fp32 rows,
                                 selection VERIFIED against a rigorous error bound (K1 stats); queries the bound cannot
                                 verify are re-searched exactly in fp32.  K <= 10.  Scores are fp32 dot products
                                 (|err| ~ 1e-7); about 3x faster than BF16X3. */
};

/* score normalisation modes of emr2a_late_fuse_scores (retrieval/fusion.py:31-42) */
enum emr2a_score_mode { EMR2A_SCORE_NONE = 0, EMR2A_SCORE_ZSCORE = 1, EMR2A_SCORE_MINMAX = 2 };

int emr2a_abi_version(void);
const char* emr2a_last_error(void);

/* Number of SMs etc. of the current device; returns EMR2A_ERR_CUDA when no
 * sm_100 device is current (the product path never falls back to the CPU). */
int emr2a_device_check(int* sm_count, int* cc_major, int* cc_minor);

/*
 * K1 -- fused normalise + weight + concatenate (+ bf16 hi/lo split).
 * Replaces, in one pass over HBM:
 *   _normalize_rows            utils/cv_evaluator.py:95-97, retrieval/evaluator.py:75-77
 *   concat_fusion              utils/cv_evaluator.py:99-105   (seg0 = image, seg1 = text)
 *   early_fusion               retrieval/fusion.py:17-28      (seg0 = text,  seg1 = image)
 *   the per-call database re-normalisation of compute_cosine_similarity
 *                              retrieval/similarity.py:5-6
 *   l2_normalize / concat_embeddings  utils/common.py:4-22    (n = 1, ZERO_GUARD)
 *
 *   v_s   = seg_s                       (or seg_s / (||seg_s|| + 1e-8) with SEGNORM)
 *   row   = [w0 * v_0 ; w1 * v_1]
 *   out   = row                         (or row / (||row|| + 1e-8) with ROWNORM)
 *
 * seg1 may be NULL with d1 = 0.  Outputs are optional (NULL to skip):
 *   out_f32  [n, ld_f32]   fp32 rows (what the Python API returns)
 *   out_hi / out_lo [n, ld_bf16]  bf16 planes for the tensor-core search:
 *            hi = bf16(out), lo = bf16(out - hi); columns [d0+d1, ld_bf16) are zero-filled
 *   inv_norm_out [n]       1 / (||row|| + 1e-8) of the final division (1.0 without ROWNORM)
 *   col_std [3][d0+d1]     with EMR2A_NF_STANDARDIZE: per-column mean | scale | RN(1/scale) of the fitted scaler
 *                          (fp32, 16-byte aligned; fp32 rows in and out, up to 2048 columns); NULL otherwise
 *   row_div_out [n][4]     the divisors used per row (deferred fp32 rows, see emr2a_lazy_rows below); NULL otherwise
 *   stats_out [2]          running maxima over the rows (atomic max; zero it before the first call):
 *                          [0] = max ||out row||, [1] = max ||out row - bf16(out row)||; needs out_hi.
 *                          Input of the EMR2A_PREC_BF16_RESCORE error bound.
 */
int emr2a_normalize_fuse(const void* seg0, const void* seg1, int64_t n, int d0, int d1,
                         int64_t ld0, int64_t ld1, float w0, float w1, int flags, int in_dtype,
                         float* out_f32, int64_t ld_f32,
                         uint16_t* out_hi, uint16_t* out_lo, int64_t ld_bf16,
                         float* inv_norm_out, float* stats_out, const float* col_std,
                         float* row_div_out, void* stream);

/*
 * Deferred fp32 rows.  The EMR2A_PREC_BF16_RESCORE arm reads the fp32 rows of the DATABASE only for the few
 * candidates it re-scores (and for the rare exact re-scan), so K1 does not have to write them: with out_f32 = NULL
 * and row_div_out [n][4] (16-byte aligned; not with EMR2A_NF_STANDARDIZE) K1 records the divisors it used per row --
 *   [0] ||seg0|| + 1e-8, [1] ||seg1|| + 1e-8 (1.0 without SEGNORM), [2] the row divisor, [3] 1.0 if it was applied --
 * and the search re-creates an element from the RAW row on the fly: x -> RN(x / n_seg) -> * w -> RN(. / n_row), the
 * same correctly rounded IEEE operations on the same inputs, hence the same fp32 value bit for bit
 * (utils/cv_evaluator.py:95-105 are those operations in numpy).  K1 then moves 6 instead of 10 bytes per fp32 input
 * element and the database needs no fp32 copy in HBM.  This struct (HOST memory, device pointers inside) describes
 * such rows to emr2a_topk_search / emr2a_rescore_candidates / emr2a_exact_rescan in place of db_f32; the raw rows
 * must stay alive and unchanged until those calls have run.  Segment widths and leading dimensions must be multiples
 * of 4 elements, pointers 16-byte (fp32) / 8-byte (bf16) aligned.
 */
typedef struct emr2a_lazy_rows {
  const void* seg0;       /* raw rows as passed to emr2a_normalize_fuse */
  const void* seg1;       /* NULL with d1 = 0 */
  int32_t d0, d1;
  int64_t ld0, ld1;
  int32_t dtype;          /* EMR2A_F32 / EMR2A_BF16 */
  float w0, w1;
  int32_t flags;          /* emr2a_nf_flags of that call */
  const float* row_div;   /* row_div_out of that call */
} emr2a_lazy_rows;

/*
 * Full score matrix out[q, j] = <q_q, db_j> in fp32 (CUDA cores), for the API
 * surfaces that must return every score: compute_cosine_similarity
 * (retrieval/similarity.py:4-7 after K1, utils/cv_evaluator.py:107-112).
 */
int emr2a_scores(const float* q, const float* db, int64_t Q, int64_t N, int D,
                 int64_t ldq, int64_t lddb, float* out, int64_t ld_out, void* stream);

/* 1 - ||db_j - q|| / max_j ||db_j - q||   (retrieval/similarity.py:10-15).
 * workspace: emr2a_euclid_workspace_bytes(N). */
size_t emr2a_euclid_workspace_bytes(int64_t N);
int emr2a_euclid_scores(const float* q, const float* db, int64_t N, int D, int64_t lddb,
                        float* out, void* workspace, size_t ws_bytes, void* stream);

/*
 * Row-wise late fusion of two score matrices:
 *   out = w * norm(text) + (1 - w) * norm(image),  norm in {none, zscore, minmax}
 * (retrieval/fusion.py:4-14, 31-42).  `one_minus_w` is passed separately because
 * the reference forms it in float64 before the fp32 multiply.
 */
int emr2a_late_fuse_scores(const float* text_scores, const float* image_scores, int64_t Q, int64_t N,
                           int64_t ld, float w_text, float one_minus_w, int mode,
                           float* out, int64_t ld_out, void* stream);

/*
 * K2 -- similarity + Top-K without materialising the score matrix.
 * Replaces np.dot + np.argsort(...)[-k:][::-1] per query
 * (utils/cv_evaluator.py:112,123,233-237; retrieval/evaluator.py:188-189,219-220).
 *
 * Operands are the rows K1 produced (weights and inverse norms already folded
 * in, so score = plain dot product):
 *   EMR2A_PREC_FP32         : q_f32 [Q, ldq_f32], db_f32 [N, lddb_f32]
 *   EMR2A_PREC_BF16X3       : q_hi,q_lo [Q, ldq_bf16] and db_hi,db_lo [N, lddb_bf16]
 *                             (bf16 bits; ld >= round_up(D,64), ld % 8 == 0, zero padded, 16-byte aligned)
 *   EMR2A_PREC_BF16X1       : q_hi, db_hi only
 *   EMR2A_PREC_BF16_RESCORE : q_hi, db_hi AND q_f32, db_f32, plus q_stats / db_stats (the float[2] K1
 *                             wrote for each side) and status_out; the hi planes must be bf16_rn of the
 *                             fp32 rows (K1 writes both from the same values) -- the error bound is built
 *                             per query from the fp32 query row, clamped by q_stats
 * q_fold / db_fold (uint8 0..254, nullable together): a pair with equal fold ids is
 * excluded -- the CV rule that a case is never retrieved from its own fold
 * (utils/cv_evaluator.py:349-376).  `fold_sorted` != 0 promises both fold
 * vectors are non-decreasing so whole tiles of a single fold can be skipped.
 * idx_base is added to the local row number (row-sharded databases).
 * out_keys [Q, K]: packed keys, best first; slots beyond the number of
 * admissible rows are 0.
 * status_out (int32[4], nullable except for BF16_RESCORE; zero it before the call):
 *   [0] number of queries whose selection the error bound could not verify (they were re-searched
 *       exactly), [1] != 0: more such queries than the re-scan list holds (about 4 % of Q, 64..1024) -- the caller
 *       must repeat the call with EMR2A_PREC_BF16X3 or EMR2A_PREC_FP32, for all queries or only for those
 *       marked in unverified_out.
 * unverified_out (uint8 [Q], nullable, BF16_RESCORE only): 1 for every query the bound could not verify
 *   (complete even when the re-scan list overflowed), 0 otherwise.
 * db_lazy (nullable, BF16_RESCORE only): deferred fp32 database rows (see emr2a_lazy_rows) instead of db_f32.
 */
size_t emr2a_topk_search_workspace_bytes(int64_t Q, int64_t N, int D, int K, int precision);
int emr2a_topk_search(const float* q_f32, int64_t ldq_f32,
                      const uint16_t* q_hi, const uint16_t* q_lo, int64_t ldq_bf16,
                      const float* db_f32, int64_t lddb_f32,
                      const uint16_t* db_hi, const uint16_t* db_lo, int64_t lddb_bf16,
                      int64_t Q, int64_t N, int D,
                      const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted,
                      int64_t idx_base, int K, int precision,
                      const float* q_stats, const float* db_stats,
                      uint64_t* out_keys, int32_t* status_out, uint8_t* unverified_out,
                      void* workspace, size_t ws_bytes, const emr2a_lazy_rows* db_lazy, void* stream);

/*
 * K2 in stages for COOPERATIVE ROW SHARDS (EMR2A_PREC_BF16_RESCORE arithmetic).  When the database is row-sharded
 * over GPUs, emr2a_topk_search on every shard re-scores 64 candidates per query and verifies its LOCAL selection --
 * work that does not shrink with the shard.  The staged calls let the shards verify ONE merged selection instead
 * (the reference scores every query against the whole database, utils/cv_evaluator.py:112,123 -- a shard only has
 * to contribute the rows that can reach the GLOBAL Top-K):
 *   1. emr2a_topk_filter        tensor-core filter of the shard: cand_out [Q, 64] approximate keys (best first, 0 =
 *                               empty), tau_out [Q] (order-preserving image of the largest filter score a row outside
 *                               the candidate lists can have; 0 = none), kth_out [Q] (nullable) = the shard's K-th
 *                               best FILTER score (-inf if it holds fewer than K admissible rows);
 *   2. the caller reduces kth_out with MAX over the shards (NCCL all-reduce, 4*Q bytes): a lower bound of the global
 *      K-th best filter score, because the shard that attains the maximum alone holds K rows at or above it;
 *   3. emr2a_rescore_candidates exact fp32 scores of the candidates whose filter score is >= kth_floor - 2E (E = the
 *                               per-query error bound of csrc/rescore.cu); a candidate below that cannot be among the
 *                               exact global K best.  out_keys [Q, K]: the shard's exact best; bound_out [Q]: an
 *                               upper bound (tau + E) of the exact score of every shard row that is NOT a candidate,
 *                               -inf if every admissible row is one.  kth_floor may be NULL (single shard);
 *   4. the caller all-gathers out_keys and bound_out and merges the keys (emr2a_topk_merge);
 *   5. emr2a_verify_merged      flags_out [Q] = 1 where the merged exact K-th best does not exceed EVERY shard's
 *                               bound (bounds[p * bounds_stride + q]), status_out[0] += the number of such queries
 *                               (zero it first).  Unflagged queries are exact: the rows not re-scored either are
 *                               candidates cut in step 3 or are bounded by bound_out;
 *   6. emr2a_exact_rescan       for the (rare) flagged queries: flag_list [n_flagged] query numbers (identical, in
 *                               the same order, on every shard); exact fp32 search of the whole shard, compact
 *                               lists out_keys [n_flagged, K]; the caller merges them across shards and writes
 *                               them over the flagged rows.  With seed_keys [n_flagged, K] -- exact keys already
 *                               known for these queries (the merged lists) -- plus db_hi (the shard's bf16 plane),
 *                               q_stats and db_stats (all nullable together) the search is FILTERED: it streams the
 *                               plane (half the bytes of the fp32 rows), computes the filter score on the CUDA cores
 *                               and scores a row exactly only if that score is within the error bound E of the best
 *                               known K-th exact score (the seed's, then the running one).  Every row that belongs
 *                               to the exact Top-K passes; a shard may return fewer than K keys (rows that cannot
 *                               beat the seed's K-th best are dropped), the merge over the shards is the exact Top-K.
 * Results are bit-identical to emr2a_topk_search on the unsharded database (same fp32 re-scoring arithmetic, same
 * tie rule).  Operand requirements are those of EMR2A_PREC_BF16_RESCORE (K <= 10); db_lazy (nullable) replaces db_f32
 * as in emr2a_topk_search.
 */
size_t emr2a_topk_filter_workspace_bytes(int64_t Q, int64_t N, int D, int K);
int emr2a_topk_filter(const uint16_t* q_hi, int64_t ldq_bf16, const uint16_t* db_hi, int64_t lddb_bf16,
                      int64_t Q, int64_t N, int D,
                      const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted,
                      int64_t idx_base, int K,
                      uint64_t* cand_out, uint32_t* tau_out, float* kth_out,
                      void* workspace, size_t ws_bytes, void* stream);
int emr2a_rescore_candidates(const uint64_t* cand, const uint32_t* tau, const float* kth_floor,
                             const float* q_f32, int64_t ldq_f32, const float* db_f32, int64_t lddb_f32,
                             int64_t Q, int64_t N, int D, int64_t idx_base, int K,
                             const float* q_stats, const float* db_stats,
                             uint64_t* out_keys, float* bound_out, const emr2a_lazy_rows* db_lazy, void* stream);
int emr2a_verify_merged(const uint64_t* keys, int K, int64_t Q, const float* bounds, int parts,
                        int64_t bounds_stride, uint8_t* flags_out, int32_t* status_out, void* stream);
size_t emr2a_exact_rescan_workspace_bytes(int n_flagged, int K);
int emr2a_exact_rescan(const float* q_f32, int64_t ldq_f32, const float* db_f32, int64_t lddb_f32,
                       int64_t N, int D, int64_t idx_base, int K,
                       const uint8_t* q_fold, const uint8_t* db_fold,
                       const int32_t* flag_list, int n_flagged,
                       uint64_t* out_keys, void* workspace, size_t ws_bytes,
                       const emr2a_lazy_rows* db_lazy,
                       const uint16_t* db_hi, int64_t lddb_bf16, const float* q_stats, const float* db_stats,
                       const uint64_t* seed_keys, void* stream);

/*
 * Range search: EVERY admissible pair (q, d) with exact score s(q, d) >= min_score, not a fixed K.  Replaces the full
 * score matrix of emr2a_scores followed by a threshold on the host (the reference's compute_cosine_similarity,
 * retrieval/similarity.py:4-7, scores everything), and with fold vectors it is the all-pairs pass of a cross-fold
 * near-duplicate audit of a CV cohort (the CV rule of utils/cv_evaluator.py:349-376).
 * Exactness, in three lines:  the filter score s~ of the 1-pass tensor-core GEMM obeys |s~ - s| <= E (the error bound
 * of EMR2A_PREC_BF16_RESCORE, from q_stats / db_stats); the filter emits every pair with s~ >= min_score - E (rounded
 * down), a superset of the answer; every emitted pair is re-scored exactly in fp32 and kept iff s >= min_score.
 * Operands are those of EMR2A_PREC_BF16_RESCORE in emr2a_topk_search (hi planes, fp32 rows or db_lazy, both stats);
 * q_fold / db_fold / fold_sorted / idx_base as there.  The scores are bit-identical to the ones emr2a_topk_search
 * reports for the same pair with EMR2A_PREC_BF16_RESCORE.
 * Buffers (device, caller-provided):
 *   cand [cand_cap][2]       uint64 (query, packed key of the FILTER score) -- scratch of the call;
 *   results [result_cap][2]  uint64 (query, packed key of the EXACT score), in unspecified order;
 *   counts_out [2]           uint64, zeroed by the caller: [0] number of filter candidates (exact, also past cand_cap),
 *                            [1] number of results (exact, also past result_cap, whenever [0] <= cand_cap; if the
 *                            candidates overflowed, no pair is re-scored and [1] stays 0).
 *   Either count above its capacity means the outputs are incomplete; one retry with cand_cap >= counts_out[0] and
 *   result_cap >= counts_out[1] (>= counts_out[0] if the candidates overflowed: results are a subset) succeeds.
 * A non-finite min_score is EMR2A_ERR_INVALID; the plane rules of the tensor-core arms give EMR2A_ERR_UNSUPPORTED.
 * workspace: emr2a_range_search_workspace_bytes(Q, N, D), 256-byte aligned.
 */
size_t emr2a_range_search_workspace_bytes(int64_t Q, int64_t N, int D);
int emr2a_range_search(const float* q_f32, int64_t ldq_f32, const uint16_t* q_hi, int64_t ldq_bf16,
                       const float* db_f32, int64_t lddb_f32, const uint16_t* db_hi, int64_t lddb_bf16,
                       int64_t Q, int64_t N, int D,
                       const uint8_t* q_fold, const uint8_t* db_fold, int fold_sorted, int64_t idx_base,
                       float min_score, const float* q_stats, const float* db_stats,
                       uint64_t* cand, int64_t cand_cap, uint64_t* results, int64_t result_cap,
                       uint64_t* counts_out, void* workspace, size_t ws_bytes,
                       const emr2a_lazy_rows* db_lazy, void* stream);

/*
 * Self-join: EVERY pair i < j of ONE row set x [n] with exact score s(i, j) >= min_score, each pair once -- the
 * near-duplicate pairs of a cohort (the reference scores all pairs with compute_cosine_similarity,
 * retrieval/similarity.py:4-7) and, with a fold vector, the cross-fold pairs of a CV cohort (the CV rule of
 * utils/cv_evaluator.py:349-376).  A call covers the query band [q_begin, q_end): every pair with q_begin <= i < q_end,
 * i < j < n, fold[i] != fold[j] when fold is given, and s >= min_score.  Bands that partition [0, n) give each pair
 * exactly once in total (the multi-GPU audit runs one band per GPU).
 * Exactness, in three lines:  the filter score s~ of the 1-pass tensor-core GEMM obeys |s~ - s| <= E (the error bound
 * of EMR2A_PREC_BF16_RESCORE, from stats); the filter emits every pair i < j with s~ >= min_score - E (rounded down), a
 * superset of the answer; every emitted pair is re-scored exactly in fp32 and kept iff s >= min_score.
 * Only the upper triangle is computed: 256-row tiles with every j <= i are skipped, and on the tiles the diagonal
 * crosses the scores with j <= i are masked (also for identical rows), so a row is never paired with itself.
 * Operands: one row set as K1 writes it for EMR2A_PREC_BF16_RESCORE: fp32 rows x_f32 [n][ld_f32], the hi plane x_hi
 * [n][ld_bf16] and its stats[2].  fold [n] (optional) and fold_sorted as in emr2a_range_search.
 * Results: (i, packed key of the EXACT score and j) in global row numbers; the scores are bit-identical to the ones
 * emr2a_range_search reports for the pair (i, j) with x as both operands.
 * Buffers, counts_out[2] and the one-retry rule: as emr2a_range_search.
 * Errors (before anything is launched; the outputs stay untouched): EMR2A_ERR_INVALID unless 0 <= q_begin <= q_end <= n,
 * for a non-finite min_score, missing rows / plane / stats, ld_f32 < D or a workspace that is not 256-byte aligned; the
 * plane rules of the tensor-core arms give EMR2A_ERR_UNSUPPORTED.
 * workspace: emr2a_self_join_workspace_bytes(n, D) is enough for any band of the row set; 256-byte aligned.
 */
size_t emr2a_self_join_workspace_bytes(int64_t n, int D);
int emr2a_self_join(const float* x_f32, int64_t ld_f32, const uint16_t* x_hi, int64_t ld_bf16, int64_t n, int D,
                    int64_t q_begin, int64_t q_end, const uint8_t* fold, int fold_sorted, float min_score,
                    const float* stats, uint64_t* cand, int64_t cand_cap, uint64_t* results, int64_t result_cap,
                    uint64_t* counts_out, void* workspace, size_t ws_bytes, void* stream);

/*
 * K3 -- merge `parts` partial Top-K lists per query into one.  Every input list must be sorted
 * best-first with its empty slots (0) at the end, as K2 and this function produce them.
 *   keys_in[(p * part_stride) + q * q_stride + j], j < K_in   ->  keys_out[q * K_out + j]
 * Used for the per-CTA partial lists of K2 and for the lists gathered from the
 * other GPUs (row-sharded database; NCCL all-gather).
 */
int emr2a_topk_merge(const uint64_t* keys_in, int parts, int64_t Q, int K_in,
                     int64_t part_stride, int64_t q_stride, int K_out,
                     uint64_t* keys_out, void* stream);

/*
 * Row-id mapping for shards that are not one contiguous range of the database (fold-balanced shards of the
 * all-queries CV, SURVEY 8e: "each shard holds ~N/(5G) rows of every fold"): K2 numbers the rows of the operand it is
 * given as idx_base + local row; this rewrites the index field of every non-empty key to row_ids[index - idx_base]
 * (scores untouched).  row_ids must be ASCENDING in the local row order so that the tie rule (score descending,
 * GLOBAL index ascending) -- and with it the order inside every list -- is preserved; then sharded results stay
 * bit-identical to the single-GPU ones.  The reference's equivalent is the train_ids list that turns a position in
 * the fold's train matrix back into a patient (utils/cv_evaluator.py:124-129, 366-371).
 */
int emr2a_keys_map_rows(uint64_t* keys, int64_t n_keys, const uint32_t* row_ids, int64_t n_rows,
                        int64_t idx_base, void* stream);

/*
 * K4 -- unpack Top-K, gather labels, vote and count.
 * Replaces the per-query python of evaluate_fold (utils/cv_evaluator.py:232-310):
 * top-1 prediction, Counter majority vote (ties -> label seen first), weighted
 * vote (score sums in rank order; wacc_f32 = 0: float64 sums as in
 * utils/cv_evaluator.py:255-260, wacc_f32 = 1: float32 sums as in
 * retrieval/evaluator.py:224-230), hit@k for each k in k_list_host (a HOST array, nk <= 16)
 * (true label in top_labels[:k]), and the two confusion matrices
 * (utils/metrics.py:56-75).
 *
 *   db_labels [>= max index + 1 - label_base]  int32 class code per database row
 *   q_labels  [Q] int32 true class codes;  q_group [Q] uint8 (nullable): counters are
 *             kept per group (the fold) -- n_groups >= 1
 * Per-query outputs (each nullable): top_idx int64 [Q,K] (-1 = empty), top_scores f32 [Q,K],
 *   top_labels int32 [Q,K] (-1 = empty), pred_top1 / pred_vote / pred_weighted int32 [Q].
 * Counters (must be zeroed by the caller, accumulated with atomics):
 *   hit_counts  uint64 [n_groups, nk]
 *   vote_counts uint64 [n_groups, 3]   (#top1 correct, #majority correct, #weighted correct)
 *   confusion   uint64 [n_groups, 2, C, C]   ([.,0]=top-1, [.,1]=majority; index [true][pred])
 *   group_sizes uint64 [n_groups]
 */
int emr2a_vote_metrics(const uint64_t* keys, int64_t Q, int K,
                       const int32_t* db_labels, int64_t label_base,
                       const int32_t* q_labels, const uint8_t* q_group, int n_groups, int C,
                       const int32_t* k_list_host, int nk, int wacc_f32,
                       int64_t* top_idx, float* top_scores, int32_t* top_labels,
                       int32_t* pred_top1, int32_t* pred_vote, int32_t* pred_weighted,
                       unsigned long long* hit_counts, unsigned long long* vote_counts,
                       unsigned long long* confusion, unsigned long long* group_sizes,
                       void* stream);

/*
 * Ingest: mean over the slices of each patient,
 *   out[p, :] = mean(x[offsets[p] : offsets[p+1], :], axis=0)
 * (pipelines/step3_retrieval/evaluate_retrieval.py:66-67 `embeddings[pid].mean(axis=0)`,
 * analysis/run_cv_experiments.py:316-333 aggregate_embeddings).  x [total_slices, ld] fp32,
 * offsets int64 [n_segments + 1] (device), slices added in order in fp32 then divided by the count.
 */
int emr2a_segment_mean(const float* x, int64_t ld, const int64_t* offsets, int64_t n_segments, int D,
                       float* out, int64_t ld_out, void* stream);

/*
 * Per-fold preprocessing (StandardScaler -> PCA fitted on the train fold: utils/cv_evaluator.py:73-93,
 * retrieval/evaluator.py:44-73): the HBM-bound passes, the float64 covariance contraction and the projection are
 * kernels of this library; only the D x D symmetric eigen-decomposition is a library call made by the host layer
 * (emr2a_b200/preprocess.py).
 *
 * emr2a_column_moments: sum[c] = SUM_r (x[r,c] - shift[c]), sumsq[c] = SUM_r (x[r,c] - shift[c])^2 over the n rows,
 *   accumulated in float64 (StandardScaler reduces float32 input in float64: sklearn _incremental_mean_and_var).
 *   shift (float[D], nullable = 0) guards the variance against cancellation.  Deterministic: fixed row partition,
 *   ordered second stage, no atomics.  workspace: emr2a_column_moments_workspace_bytes(n, D), 8-byte aligned.
 * emr2a_standardize: out[r,c] = (x[r,c] - mean[c]) / scale[c] in IEEE fp32, mean/scale already cast to float32 --
 *   the arithmetic of StandardScaler.transform on a float32 array (`X -= astype(mean_, X.dtype); X /= astype(scale_,
 *   X.dtype)`).  out may alias x.
 * emr2a_gram_f64: gram[a,b] = SUM_r z[r,a] z[r,b] and zsum[a] = SUM_r z[r,a] in float64, where z = the standardised
 *   row computed on the fly, z[r,c] = fp32((x[r,c] - mean[c]) / scale[c]) (mean/scale nullable: z = x) -- the
 *   covariance input of the PCA fit (PCA.fit on the scaler's output, utils/cv_evaluator.py:89-90) without writing
 *   the standardised matrix.  Hand-written float64 FMA contraction, deterministic (fixed row partition, ordered
 *   second stage).  gram is the full symmetric D x D matrix, row-major.  workspace:
 *   emr2a_gram_f64_workspace_bytes(n, D), 8-byte aligned.
 * emr2a_project: out[r,j] = SUM_c z[r,c] * w[j,c] - bias[j]  (PCA.transform: `X @ components_.T - mean_ @
 *   components_.T`, utils/cv_evaluator.py:90-91) with z standardised on the fly as above, fp32 FMA in ascending c
 *   (bit-identical to emr2a_standardize followed by emr2a_scores and the subtraction).  bias nullable.
 */
size_t emr2a_gram_f64_workspace_bytes(int64_t n, int D);
int emr2a_gram_f64(const float* x, int64_t ld, int64_t n, int D, const float* mean, const float* scale,
                   double* gram, double* zsum, void* workspace, size_t ws_bytes, void* stream);
int emr2a_project(const float* x, int64_t ld, int64_t n, int D, const float* mean, const float* scale,
                  const float* w, int64_t ldw, int P, const float* bias, float* out, int64_t ld_out, void* stream);
size_t emr2a_column_moments_workspace_bytes(int64_t n, int D);
int emr2a_column_moments(const float* x, int64_t ld, int64_t n, int D, const float* shift,
                         double* sum, double* sumsq, void* workspace, size_t ws_bytes, void* stream);
int emr2a_standardize(const float* x, int64_t ld, int64_t n, int D, const float* mean, const float* scale,
                      float* out, int64_t ld_out, void* stream);

/*
 * Late fusion with z-score / min-max score normalisation without the [Q, N] score matrix
 * (retrieval/fusion.py:4-14, 31-42; retrieval/evaluator.py:150-157).  Per query the fused score is an affine map
 *     fused[d] = < [g_t * Tq ; g_i * Iq], [Td ; Id] > - c
 * of the two similarity vectors, so the Top-K is the ordinary fused search with per-row scaled query segments
 * and the constant applied to the winning scores afterwards:
 * emr2a_scale_segments: x[r, 0:d0] *= g0[r], x[r, d0:d0+d1] *= g1[r]   (fp32 rows, in place; g1 nullable if d1 = 0)
 * emr2a_keys_add_offset: score of every non-empty key of query q += offset[q] (order within a query is unchanged).
 */
int emr2a_scale_segments(float* x, int64_t n, int d0, int d1, int64_t ld, const float* g0, const float* g1,
                         void* stream);
int emr2a_keys_add_offset(uint64_t* keys, int64_t Q, int K, const float* offset, void* stream);

/* Top-K of a given score matrix (the *_from_scores helpers and get_all_top_labels,
 * retrieval/evaluator.py:195-208, 235-275): keys out [Q, K]. */
int emr2a_topk_from_scores(const float* scores, int64_t Q, int64_t N, int64_t ld, int K,
                           uint64_t* out_keys, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EMR2A_H */
