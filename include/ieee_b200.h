/*
 * ieee_b200.h -- C ABI of libieee_b200.so: the B200 (sm_100a) implementation of the
 * test-time retrieval hot path of ziwang1121/IEEE (a torchreid fork).
 *
 * The reference has no FFI for this path: it is three Python module-level functions plus one
 * CPython extension (file:line relative to the reference tree):
 *
 *   torchreid/metrics/distance.py:6          compute_distance_matrix(input1, input2, metric)
 *   torchreid/metrics/rank.py:246            evaluate_rank(distmat, q_pids, g_pids, q_camids, g_camids, max_rank, ...)
 *   torchreid/metrics/rank_cylib/rank_cy.pyx:26   evaluate_cy(...)          (the one native seam)
 *   torchreid/utils/rerank.py:31             re_ranking(q_g_dist, q_q_dist, g_g_dist, k1, k2, lambda_value)
 *   torchreid/engine/engine.py:391-417       Engine._evaluate: normalise -> distmat -> [rerank] -> evaluate_rank
 *
 * The entry points below are what a binding for those functions calls (ctypes stub in
 * INTEGRATION.md; ieee_b200/_lib.py is that stub).  Conventions:
 *
 *   - every pointer is a DEVICE pointer unless the parameter name ends in _host;
 *   - nothing is allocated on the caller's behalf: outputs and workspaces are passed in, workspace
 *     sizes come from the matching *_workspace_bytes() function; workspaces need 256-byte alignment;
 *   - all work is enqueued on `stream` (a cudaStream_t) and is asynchronous unless the function
 *     name ends in _sync;
 *   - return value: IEEE_OK or an ieee_status; ieee_last_error() gives the text (thread local);
 *   - no CPU fallback anywhere: without a CUDA device every compute call returns IEEE_ERR_CUDA.
 *
 * Matrices are row-major with an explicit leading dimension in ELEMENTS.
 */
#ifndef IEEE_B200_H_
#define IEEE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IEEE_B200_ABI_VERSION 4

typedef void* ieee_stream_t; /* cudaStream_t */

typedef enum {
  IEEE_OK = 0,
  IEEE_ERR_INVALID = 1,        /* bad argument (shape, alignment, enum)                        */
  IEEE_ERR_CUDA = 2,           /* CUDA runtime / driver error, or no device                    */
  IEEE_ERR_WORKSPACE = 3,      /* workspace too small or misaligned                            */
  IEEE_ERR_NO_VALID_QUERY = 4, /* rank.py:165 "all query identities do not appear in gallery" */
  IEEE_ERR_SHORT_RANK_LIST = 5,/* a valid query keeps fewer than max_rank gallery items
                                  (ragged ValueError in rank.py:167, stale buffer in rank_cy.pyx) */
  IEEE_ERR_CAPACITY = 6        /* a per-query list exceeded the capacity given by the caller   */
} ieee_status;

/* distance.py:36-44; NEG_DOT = -(a . b), the similarity GNN re-ranking starts from (gnn_reranking.py:31) as a distance */
typedef enum { IEEE_METRIC_EUCLIDEAN = 0, IEEE_METRIC_COSINE = 1, IEEE_METRIC_NEG_DOT = 2 } ieee_metric;
typedef enum { IEEE_DTYPE_F32 = 0, IEEE_DTYPE_BF16 = 1 } ieee_dtype;

/* Arithmetic of the distance contraction (always fp32 accumulation in TMEM / registers):
 *   F16X3     fp32 features scaled per row by a power of two, split into fp16 hi + lo (22 mantissa bits), three
 *             tcgen05 MMAs per k-step (hi*hi, hi*lo, lo*hi) into one accumulator; the dropped lo*lo term is
 *             <= 2^-24 relative: fp32-grade products.  Default for fp32 inputs; meets the 1e-4 parity bound.
 *   BF16      one tcgen05 MMA per k-step on bf16-rounded features (exact products for bf16 inputs).
 *   FP32_SIMT plain fp32 FMA kernel (no tensor cores); cross-check for the tensor path.           */
typedef enum { IEEE_PREC_F16X3 = 0, IEEE_PREC_BF16 = 1, IEEE_PREC_FP32_SIMT = 2 } ieee_precision;

const char* ieee_last_error(void);
int ieee_abi_version(void);
/* Number of SMs / compute capability (major*10+minor) of the current device; IEEE_ERR_CUDA without one. */
int ieee_device_info(int* sm_count, int* compute_capability);
/* Tensor-core kernel pairing: 2 (default) = tcgen05 cta_group::2, one 256 x 256 tile per SM pair;
 * 1 = cta_group::1, one 128 x 256 tile per SM.  Returns the previous value.  (Env: IEEE_B200_CTA_GROUP.) */
int ieee_set_cta_group(int cta_group);
/* Accumulation chunking of the tensor-core contraction: the tcgen05 fp32 accumulator truncates, so
 * every `k_slices` 64-wide K-slices the partial sums are moved to registers and added there with round-to-nearest.
 * 0 = accumulate the whole K in TMEM (fastest, ~1e-5 relative bias on the dot product); default 6 (F16X3 mode;
 * the 1-pass BF16 mode always accumulates the whole K in TMEM).
 * Returns the previous value. */
int ieee_set_accum_chunk(int k_slices);
/* Tile raster of the contraction: m tiles (256 query rows each with cta_group 2) per panel; inside a panel m runs
 * fastest, so one panel's query rows stay L2-resident while it sweeps every gallery tile.  0 (default) sizes the
 * panel for ~40 MB of query operand.  Negative: query only.  Returns the previous value. */
int ieee_set_raster_panel(int m_tiles);
/* Warps that stream one query's distance row together in the count stage, for rows of 4 K .. 64 K columns: 1, 2, 4 or
 * 8 (shorter rows always take one warp, longer ones the whole CTA of 8).  Other values: query only.  Returns the
 * previous value.  Results do not depend on it. */
int ieee_set_count_team(int warps_per_query);
/* Whether the one-call entry points (ieee_distmat, ieee_retrieve_eval) centre euclidean operands on the query
 * set's mean (see ieee_feature_center).  Default 1; 0 reproduces the uncentred arithmetic of ABI 2 (accuracy
 * studies).  Negative: query only.  Returns the previous value. */
int ieee_set_centering(int on);
/* Diagnostics for kernel tuning (results are WRONG when non-zero): bit 0 = tensor-core epilogue skips its global
 * stores, bit 1 = epilogue also skips the TMEM reads, bit 2 = no TMA store, bit 3 = chunk BF16 mode too, bit 4 = count
 * stage always uses the CTA-per-query kernel with shared atomics (results stay correct), bit 5 = no near-duplicate
 * fix-up pass (results stay within the accumulator's floor), bit 7 = step timeline (results stay correct): the
 * one-call entry points record a CUDA event after every launch they make on the caller's stream.  Returns the
 * previous value. */
int ieee_set_debug_flags(int flags);
/* Number of CUDA kernels this library has launched in this process (bench.py reports the per-step delta).
 * ieee_note_launches adds n to it -- for a caller that replays a captured CUDA graph of this library's launches,
 * which the library cannot see -- and returns the new count. */
int64_t ieee_launch_count(void);
int64_t ieee_note_launches(int64_t n);
/* Step timeline (debug bit 7), per calling thread: _reset forgets the marks; ieee_debug_timeline waits for the last
 * mark and writes one line per mark, "name\tus since the previous mark\tus since the first mark", into buf (NUL
 * terminated, truncated to cap).  Returns the number of marks, -1 on a CUDA error.  At most 96 marks are kept. */
void ieee_debug_timeline_reset(void);
int ieee_debug_timeline(char* buf, size_t cap);

/* ------------------------------------------------------------------------------------------------
 * Distance matrix.   Replaces distance.py:49-64 (euclidean_squared_distance: ||a||^2 + ||b||^2 - 2ab^T,
 * squared, unclamped) and distance.py:67-80 (cosine_distance: 1 - normalize(a) normalize(b)^T, eps 1e-12).
 * `normalize` != 0 applies engine.py:391-394 (F.normalize of both sets) first.
 *
 * Packed operand = what the tensor-core kernel consumes: a 16-bit hi plane (+ lo plane for F16X3), each
 * [rows, Dp] with Dp = D rounded up to 64, zero padded, plus two fp32 per row (squared norm and the
 * power-of-two row scale).  Pack a gallery once, reuse it for every query block.
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_packed_bytes(int64_t rows, int64_t D, int precision);
/* center: NULL, or float32[D] (16-byte aligned) subtracted from every (normalised) row before it is split; euclidean
 * only.  |q - g|^2 does not change when the same vector is subtracted from q and g, but the fp32 evaluation of
 * |q|^2 + |g|^2 - 2 q.g loses |q|^2 + |g|^2 times a few ulps to cancellation (distance.py:59-64 does too): with the
 * common component of the post-ReLU features removed, that scale shrinks to the spread of the data and the tensor
 * core's truncating accumulator sees mixed-sign products.  Both operands of a contraction MUST be packed with the
 * same centre. */
int ieee_pack_features(const void* x, int dtype, int64_t ld, int64_t rows, int64_t D, int metric, int normalize,
                       int precision, const float* center, void* packed, ieee_stream_t stream);
/* Centre for ieee_pack_features: column mean over up to max_rows (0: 64) evenly strided rows of x, scaled to unit
 * length when `normalize` is set (the rows will be).  Deterministic (fixed summation order).  center: float32[D];
 * workspace: ieee_feature_center_workspace_bytes(D). */
size_t ieee_feature_center_workspace_bytes(int64_t D);
int ieee_feature_center(const void* x, int dtype, int64_t ld, int64_t rows, int64_t D, int normalize, int64_t max_rows,
                        float* center, void* workspace, ieee_stream_t stream);
/* fixup_workspace: NULL, or ieee_distmat_fixup_bytes(Q) bytes (8-byte aligned).  With it (euclidean, F16X3) every
 * output below 2^-6 of its scale |q|^2 + |g|^2 -- near-duplicate pairs, where the expansion |q|^2 + |g|^2 - 2 q.g only
 * keeps the ABSOLUTE accuracy of its terms -- is listed by the contraction and recomputed as sum_k (q_k - g_k)^2 by
 * a second small kernel: all distances then sit within 1e-4 relative of the exact value.  Word 0 of the workspace
 * holds the number of 128-output spans flagged; the list keeps 2 Q + 4096 of them, and when there are more the second
 * kernel re-tests every span of the block instead, so none is missed. */
size_t ieee_distmat_fixup_bytes(int64_t Q);
int ieee_distmat_packed(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                        int precision, float* out, int64_t ldo, void* fixup_workspace, ieee_stream_t stream);
size_t ieee_distmat_workspace_bytes(int64_t Q, int64_t G, int64_t D, int precision);
/* One call: [centre on q's rows ->] pack both sides into the workspace, then the contraction.  out[Q, G] float32,
 * leading dim ldo. */
int ieee_distmat(const void* q, const void* g, int dtype, int64_t ldq, int64_t ldg, int64_t Q, int64_t G, int64_t D,
                 int metric, int normalize, int precision, float* out, int64_t ldo, void* workspace,
                 size_t workspace_bytes, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Ranking + CMC / mAP, Market-1501 protocol.   Replaces rank.py:103-171 (eval_market1501) and
 * rank_cy.pyx:156-243 (eval_market1501_cy).  Sort-free: the metrics depend only on the positions of the
 * relevant gallery items among the kept ones, pos(r) = #{kept g : (d[q,g], g) <lex (d[q,r], r)} -- ties are
 * broken by gallery index (the order the reference leaves to NumPy's unstable argsort), NaN ranks last.
 *
 * Three stream-ordered stages so that a gallery sharded over several GPUs can exchange between them:
 *   group   : sort the (local) gallery by pid once                        -> ieee_gallery_group
 *   gather  : per query, its relevant / junk gallery items and distances  -> ieee_rank_gather
 *             [all-gather of the relevant lists across shards]
 *   count   : one streaming pass over the (local) distance rows           -> ieee_rank_count
 *             [all-reduce SUM of the integer counts across shards]
 *   finalize: AP in fp64, CMC hit counts, means                           -> ieee_rank_finalize
 * ieee_eval_market1501 runs all of them for the single-GPU case.
 * ---------------------------------------------------------------------------------------------- */

/* Result block written by ieee_rank_finalize / ieee_eval_market1501 (device memory, 64 bytes + cmc). */
typedef struct {
  double mAP;              /* mean of per-query AP over valid queries (float64, rank.py:169)            */
  double sum_ap;           /* sum of AP (for merging query blocks: mAP = sum_ap / num_valid)            */
  int64_t num_valid;       /* queries with at least one relevant kept gallery item (rank.py:142-144)    */
  int64_t num_ties;        /* (relevant item, other kept item) pairs with bit-equal distance            */
  int64_t num_short;       /* valid queries that keep fewer than max_rank gallery items                 */
  int32_t max_rank;        /* effective K' = min(max_rank, G_total) (rank.py:110-115)                   */
  int32_t status;          /* IEEE_OK / IEEE_ERR_NO_VALID_QUERY / IEEE_ERR_SHORT_RANK_LIST              */
  int64_t list_overflow;   /* 0, or the list capacity a query needed when it exceeded the caller's `cap` hint
                              (ieee_retrieve_eval*: every other field is then meaningless, call again)     */
  double mINP;             /* mean inverse negative penalty over valid queries: R / (1-based rank of the hardest
                              relevant item among the kept ones) (README.rst:45; Ye et al., TPAMI 2021)     */
} ieee_eval_summary;

/* Group the (local) gallery by identity once: the blob holds an open-addressing hash table pid -> (offset, count)
 * into the gallery indices grouped by pid, so a query finds all gallery items of its identity with one probe
 * instead of scanning G labels.  g_pids: int64[G], G < 2^30; the value 0x8080808080808080 is reserved. */
size_t ieee_gallery_group_bytes(int64_t G);
int ieee_gallery_group(const int64_t* g_pids, int64_t G, void* group /* ieee_gallery_group_bytes(G), 256-aligned */,
                       ieee_stream_t stream);
/* Largest number of (local) gallery items sharing an identity with any of the Q queries = the list capacity
 * `cap` the gather/count stages need.  cap_dev: one int32 of device memory (written asynchronously);
 * the _sync form also copies it to the host and synchronises the stream. */
int ieee_rank_list_cap(const void* group, int64_t G, const int64_t* q_pids, int64_t Q, int32_t* cap_dev,
                       ieee_stream_t stream);
int ieee_rank_list_cap_sync(const void* group, int64_t G, const int64_t* q_pids, int64_t Q, int32_t* scratch_dev,
                            int32_t* cap_host, ieee_stream_t stream);

/* gather: for each of Q queries, rel[q, 0..n) = packed (orderable distance key << 32 | global gallery index) of
 * the relevant local items (same pid, other camera), junk[q, ...] likewise for the junk items (same pid, same
 * camera, rank.py:136).  `cap` = list capacity per query (>= ieee_rank_list_cap).  Unsorted.
 * rel is uint64[Q, cap + 1]: entry [q, cap] holds the list length, so ONE all-gather of rel moves lists and lengths;
 * n_rel / n_junk (int32[Q]) receive the lengths as well.  junk is uint64[Q, cap].
 * g_offset = global index of local gallery row 0 (0 on one GPU). */
int ieee_rank_gather(const float* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids,
                     const int64_t* q_camids, const int64_t* g_camids, const void* group, int64_t g_offset,
                     int32_t cap, uint64_t* rel, int32_t* n_rel, uint64_t* junk, int32_t* n_junk,
                     int32_t* overflow_flag, ieee_stream_t stream);

/* count: thresholds of query q = union over the `shards` relevant lists rel_all[s][q][cap + 1] (the all-gathered
 * buffers; shards = 1 and rel_all = rel on one GPU).  Streams the local distance row once and writes
 * counts[q, k] = #{local kept g : (d, g) <lex T_k} for the k-th smallest threshold, k < R[q] (= lengths summed over
 * shards), plus counts[q, W] = this shard's number of relevant items (n_rel) and counts[q, W + 1] = its number of
 * junk items.  counts is int32[Q, W + 2] with row width W = out_cap (0: W = shards*cap, always enough); it is
 * summed over shards by the caller (all-reduce) before query_metrics / finalize, which read R[q] from it -- call
 * those with shards = 1, cap = W.  A merged list is rarely as long as shards*cap: passing the longest one seen
 * before (stats[1] of an earlier call with the same labels) as out_cap shrinks the all-reduce by ~the shard count.
 * stats (uint64[2], may be NULL): [0] accumulates bit-equal (threshold, other kept item) pairs, [1] receives the
 * longest merged list (max-updated).  stats[1] > out_cap means some rows were too narrow and their counts were
 * NOT written: run again with out_cap >= stats[1]. */
size_t ieee_rank_count_smem_bytes(int32_t shards, int32_t cap);
int ieee_rank_count(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, int32_t shards,
                    int32_t cap, int32_t out_cap, const uint64_t* rel_all, const int32_t* n_rel,
                    const uint64_t* junk, const int32_t* n_junk, int32_t* counts, unsigned long long* stats,
                    ieee_stream_t stream);

/* finalize = ieee_rank_query_metrics (per query) followed by ieee_rank_reduce (over queries); the two halves
 * are exported separately so that query blocks can share one final reduction.
 *
 * query_metrics: pos_k = counts[q,k] (already summed over shards); ap[q] = (1/R) sum_k (k+1)/(pos_k+1) in
 * float64 (rank.py:155-160), first[q] = pos_0 (-1: invalid query, rank.py:142-144), short_list[q] = 1 when
 * the query keeps fewer than max_rank gallery items.  G_total = gallery size over all shards.
 * reduce: cmc[0..K') float32 = float32(hits_j) / float32(num_valid) exactly as rank.py:167-168 and
 * mAP = mean(ap) (float64, fixed reduction tree: bitwise reproducible), K' = min(max_rank, G_total). */
int ieee_rank_query_metrics(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards, int32_t cap,
                            int32_t max_rank, double* ap, int32_t* first, int32_t* short_list,
                            double* inp /* double[Q] inverse negative penalty, may be NULL */, ieee_stream_t stream);
int ieee_rank_reduce(const double* ap, const int32_t* first, const int32_t* short_list, int64_t Q, int32_t max_rank,
                     const unsigned long long* ties, float* cmc, ieee_eval_summary* summary,
                     const double* inp /* may be NULL: mINP = 0 */, ieee_stream_t stream);
/* per_query_ap (double[Q]) / per_query_first (int32[Q]) may be NULL.  workspace: ieee_rank_finalize_workspace_bytes(Q). */
size_t ieee_rank_finalize_workspace_bytes(int64_t Q);
int ieee_rank_finalize(const int32_t* counts, int64_t Q, int64_t G_total, int32_t shards, int32_t cap,
                       int32_t max_rank, const unsigned long long* ties, float* cmc,
                       ieee_eval_summary* summary, double* per_query_ap, int32_t* per_query_first, void* workspace,
                       ieee_stream_t stream);

/* Single-GPU evaluate_rank on a device distmat: group + gather + count + finalize.  Synchronises the stream
 * once (ieee_rank_list_cap_sync) to size the per-query lists.  `cap` = list capacity the workspace was sized
 * for (0: sized with the default of ieee_eval_workspace_bytes); IEEE_ERR_CAPACITY if a query needs more.
 * cmc: float[max_rank] device, summary: device. */
size_t ieee_eval_workspace_bytes(int64_t Q, int64_t G, int32_t cap /* 0 = min(G, 4096) */);
int ieee_eval_market1501(const float* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids,
                         const int64_t* g_pids, const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank,
                         int32_t cap, float* cmc, ieee_eval_summary* summary, void* workspace, size_t workspace_bytes,
                         ieee_stream_t stream);

/* Gallery side of an evaluation in ONE call: identity grouping (on an internal high-priority side stream), [centre
 * from the query rows q], feature packing of the gallery and, when q_packed is given, of the query rows too.
 *   q != NULL and no IEEE_PREPARE_KEEP_CENTER: the column mean of (a sample of) q is written to center (float32[D]) and used;
 *   otherwise center is an INPUT (or NULL: uncentred).
 *   q_packed != NULL: the Q rows of q are packed there as well (ieee_packed_bytes(Q, D, precision)) and can be handed to
 *   ieee_retrieve_eval_prepared* -- the caller's host work between the two calls then hides behind that kernel.
 *   IEEE_PREPARE_DEFER_JOIN: the grouping is left running on the side stream; a stream must call
 *   ieee_gallery_group_join before it reads `group` (ieee_retrieve_eval_prepared* do that themselves, right before
 *   their gather stage: the label-only kernels then run beside the contraction instead of holding it up).
 * g_pids / group may be NULL to skip the grouping.  workspace: not used any more (the centre is one launch); may be
 * NULL.  ieee_gallery_prepare_workspace_bytes is kept for callers that still size one. */
#define IEEE_PREPARE_DEFER_JOIN 1
#define IEEE_PREPARE_KEEP_CENTER 2
size_t ieee_gallery_prepare_workspace_bytes(int64_t D);
int ieee_gallery_prepare(const void* gf, int64_t ldg, int dtype, int64_t G, int64_t D, int metric, int normalize,
                         int precision, const int64_t* g_pids, const void* q, int64_t ldq, int64_t Q, float* center,
                         void* g_packed, void* group, void* q_packed, int flags, void* workspace, ieee_stream_t stream);
/* `stream` waits for the grouping most recently left on this device's side stream (no-op if there is none). */
int ieee_gallery_group_join(ieee_stream_t stream);

/* The same for a FLOAT64 distance matrix, ranked in float64 order: evaluate_py (rank.py:117, the function this fork
 * runs) argsorts the matrix in the dtype it is given, so distances that differ below float32 resolution are ordered
 * there and must not be tied by a float32 copy.  Same workspace as ieee_eval_market1501; at most 4096 same-identity
 * gallery items per query. */
int ieee_eval_market1501_f64(const double* distmat, int64_t ld, int64_t Q, int64_t G, const int64_t* q_pids,
                             const int64_t* g_pids, const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank,
                             int32_t cap, float* cmc, ieee_eval_summary* summary, void* workspace,
                             size_t workspace_bytes, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Retrieval + evaluation in ONE call: the tail of Engine._evaluate (engine.py:391-417) --
 * [normalise] -> distance matrix -> Market-1501 CMC / mAP -- enqueued back to back on `stream` from C, so a
 * binding pays one foreign call per evaluation instead of one per kernel.
 *
 * ieee_retrieve_eval           raw query AND gallery features + labels in, (cmc, summary) out; euclidean operands
 *                              are centred on the query set (ieee_set_centering).
 * ieee_retrieve_eval_prepared  the gallery side was prepared once (ieee_pack_features + ieee_gallery_group)
 *                              and is reused for every query set.
 * cap > 0  : list-capacity HINT (e.g. the value a previous call reported); fully asynchronous.  If a query needs
 *            more, summary->list_overflow holds the needed capacity and the other results are meaningless.
 * cap <= 0 : the capacity is queried first (one stream synchronisation, ieee_rank_list_cap_sync) and written to
 *            *cap_host_out when that is not NULL.
 * distmat  : float32 [Q, ld] scratch for the distance block, ld >= G (ld % 32 == 0 keeps the TMA-store epilogue);
 *            holds the distance matrix on return (compute_distance_matrix's result, distance.py:6).
 * cmc: float[max_rank] device; summary: device; per_query_ap (double[Q]) / per_query_first (int32[Q]) may be NULL.
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_retrieve_workspace_bytes(int64_t Q, int64_t G, int64_t D, int precision, int32_t cap /* 0 = min(G, 4096) */);
int ieee_retrieve_eval(const void* qf, int64_t ldq, const void* gf, int64_t ldg, int dtype, int64_t Q, int64_t G,
                       int64_t D, int metric, int normalize, int precision, const int64_t* q_pids,
                       const int64_t* g_pids, const int64_t* q_camids, const int64_t* g_camids, int32_t max_rank,
                       int32_t cap, int32_t* cap_host_out, float* distmat, int64_t ld, float* cmc,
                       ieee_eval_summary* summary, double* per_query_ap, int32_t* per_query_first, void* workspace,
                       size_t workspace_bytes, ieee_stream_t stream);
size_t ieee_retrieve_prepared_workspace_bytes(int64_t Q, int64_t D, int precision, int32_t cap);
int ieee_retrieve_eval_prepared(const void* qf, int64_t ldq, int dtype, int64_t Q, int64_t D, int metric, int normalize,
                                int precision, const void* g_packed, const void* group,
                                const float* center /* the centre g_packed was packed with, or NULL */, int64_t G,
                                const int64_t* q_pids, const int64_t* q_camids, const int64_t* g_camids,
                                int32_t max_rank, int32_t cap, int32_t* cap_host_out, float* distmat, int64_t ld,
                                float* cmc, ieee_eval_summary* summary, double* per_query_ap,
                                int32_t* per_query_first,
                                const void* q_packed /* NULL, or the query rows as packed by ieee_gallery_prepare (qf is
                                                        then not read and may be NULL) */,
                                void* workspace, size_t workspace_bytes, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Junk-masked top-k ranked list: the first k entries of rank.py:117 + :136-140 per query (what
 * torchreid/utils/reidtools.py:49,111 walks), ascending (distance, index); rows with fewer than k kept
 * items are padded with index -1 / +inf.  Pass q_pids = NULL for an unmasked top-k (re-ranking, rerank.py:48).
 * idx: int32[Q, k] GLOBAL gallery indices (local + g_offset), val: float[Q, k].  k <= 1024.
 * ---------------------------------------------------------------------------------------------- */
int ieee_topk(const float* distmat, int64_t ld, int64_t Q, int64_t G, int64_t g_offset, const int64_t* q_pids,
              const int64_t* q_camids, const int64_t* g_pids, const int64_t* g_camids, int32_t k, int32_t* idx,
              float* val, ieee_stream_t stream);
/* Merge `shards` per-shard top-k lists (idx_all[s][Q][k], val_all[s][Q][k]) into the global top-k. */
int ieee_topk_merge(const int32_t* idx_all, const float* val_all, int32_t shards, int64_t Q, int32_t k,
                    int32_t* idx, float* val, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * k-reciprocal re-ranking.   Replaces rerank.py:31-113.  Inputs are the three device distance matrices
 * (float32): q_g [Q,G], q_q [Q,Q], g_g [G,G]; out: float32 [Q, G] (leading dim ldo).
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_rerank_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2);
int ieee_rerank(const float* q_g, int64_t ld_qg, const float* q_q, int64_t ld_qq, const float* g_g, int64_t ld_gg,
                int64_t Q, int64_t G, int32_t k1, int32_t k2, double lambda_value, float* out, int64_t ldo,
                void* workspace, size_t workspace_bytes, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * k-reciprocal re-ranking, streamed: the same result as ieee_rerank, computed from packed features (ieee_pack_features,
 * both operands with the same centre) without any N x N or Q x Q matrix, N = Q + G.
 *   ieee_rerank_stream_prepare computes the virtual matrix [[qq, qg], [qg^T, gg]] in column strips (of width
 *   strip_bytes / ~8N, a multiple of 256 columns) twice with the contraction: the first pass yields the column
 *   maxima `colmax` (float32 [N]) and the first k1 + 1 neighbours `rank` (int32 [N, k1 + 1]) of every sample, the second
 *   the weights of the k-reciprocal sets.  The strips live in `scratch` (ieee_rerank_stream_scratch_bytes), which is
 *   free again when the call's work on the stream is done.  The sparse state (V, its query expansion, the inverted
 *   index) stays in `workspace` (ieee_rerank_stream_workspace_bytes, linear in N), which must outlive the block calls.
 *   No host synchronisation.
 *   ieee_rerank_stream_block turns the distances of queries [row0, row0 + rows) to the gallery (float32 [rows, G],
 *   leading dim ld, as the contraction of those packed query rows against g_packed writes them) into their re-ranked
 *   distances, in place; scratch holds rows * G floats.  Q, G, k1, k2 and colmax are those given to the prepare call.
 * Bit-identical to ieee_rerank on the three matrices the contraction writes for the same packed operands.  Limits as
 * ieee_rerank: k1 + 1 <= 512 and <= N, 1 <= k2 <= k1 + 1, k2 * (k1+1) * (round(k1/2)+2) <= 16384 entries per row,
 * N < 2^24; precision F16X3 or BF16.  The size queries need no GPU and return 0 (with ieee_last_error set) when the
 * parameters are out of range.
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_rerank_stream_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2);
size_t ieee_rerank_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes);
int ieee_rerank_stream_prepare(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int metric,
                               int precision, int32_t k1, int32_t k2, size_t strip_bytes, float* colmax, int32_t* rank,
                               void* workspace, size_t workspace_bytes, void* scratch, size_t scratch_bytes,
                               ieee_stream_t stream);
int ieee_rerank_stream_block(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, const float* colmax,
                             int64_t row0, int64_t rows, double lambda_value, float* block, int64_t ld, void* scratch,
                             size_t scratch_bytes, ieee_stream_t stream);

/* k-reciprocal re-ranking, streamed, in phases: the prepare call split so that S processes, each holding a gallery slice
 * [g0, g0 + Gs) (the slices tiling [0, G) in order) and the replicated queries, share its strips and end with the state
 * of their own slice.  ieee_rerank_stream_prepare is pass 0, pass 1 and finish over every sample with the window
 * (0, G); ieee_rerank_stream_block is ieee_rerank_stream_block_window with Gs = G.  Same limits as above.
 *   ieee_rerank_stream_pass needs the whole gallery packed (g_packed, G rows, as for the prepare call) and computes the
 *   strips of the owned samples only: queries [q0, q1) and gallery rows [g0, g1), each range starting at a multiple of
 *   256 of its segment and ending at one or at the segment's end (an empty range is allowed).  The bits do not depend on
 *   the ranges or on strip_bytes.
 *     pass 0 writes colmax and rank of the owned samples (colmax[i], rank[i, :] for i in [q0, q1) and [Q + g0, Q + g1)).
 *       workspace may be null.  Exchange: every process needs colmax [N] and rank [N, k1 + 1] of all samples before
 *       pass 1 (an all-gather of the owned rows).
 *     pass 1 writes V's columns and counts of all N rows (from rank alone, the same on every process) and V's values of
 *       the owned rows.  workspace: ieee_rerank_stream_window_workspace_bytes of this process's window (V comes first).
 *       Exchange: every process needs V's values of all rows before finish; ieee_rerank_stream_v_layout says where they
 *       are (an all-gather of the owned rows of a [N, cap] float32 array).
 *   ieee_rerank_stream_finish builds the query expansion and the inverted index of the gallery window [g0, g0 + Gs) from
 *   rank and V of every sample; the workspace then serves block calls for that window only.
 *   ieee_rerank_stream_block_window re-ranks the distances of queries [row0, row0 + rows) to the window's Gs gallery rows
 *   (float32 [rows, Gs], leading dim ld), in place: the same bits as columns [g0, g0 + Gs) of ieee_rerank_stream_block on
 *   the whole gallery's distances.  scratch holds rows * Gs floats.
 *   ieee_rerank_stream_window_workspace_bytes: V of N rows plus expansion and index of Q + Gs rows, about
 *   8 c N + 16 k2 c (Q + Gs) bytes with c = (k1+1)(round(k1/2)+2) (k2 = 1: 8 c N + 8 c (Q + Gs)); for Gs = G it is
 *   ieee_rerank_stream_workspace_bytes.  Returns 0 with ieee_last_error set when out of range.
 *   ieee_rerank_stream_v_layout: V in the workspace is three arrays of N rows, cap entries each: columns (int32 [N, cap])
 *   at byte offset off_col, values (float32 [N, cap]) at off_val, counts (int32 [N]) at off_cnt; row i holds cnt[i] valid
 *   entries.  The same for every window.  Needs no GPU.
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_rerank_stream_window_workspace_bytes(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs);
int ieee_rerank_stream_v_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t* cap, size_t* off_col, size_t* off_val,
                                size_t* off_cnt);
int ieee_rerank_stream_pass(int32_t pass, const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D,
                            int metric, int precision, int32_t k1, int32_t k2, size_t strip_bytes, int64_t q0, int64_t q1,
                            int64_t g0, int64_t g1, float* colmax, int32_t* rank, void* workspace, size_t workspace_bytes,
                            void* scratch, size_t scratch_bytes, ieee_stream_t stream);
int ieee_rerank_stream_finish(void* workspace, size_t workspace_bytes, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t g0,
                              int64_t Gs, const int32_t* rank, ieee_stream_t stream);
int ieee_rerank_stream_block_window(const void* workspace, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t Gs,
                                    const float* colmax, int64_t row0, int64_t rows, double lambda_value, float* block,
                                    int64_t ld, void* scratch, size_t scratch_bytes, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GNN re-ranking (alternative `rerank` mode).   Replaces torchreid/utils/GPU-Re-Ranking/gnn_reranking.py:27-59 with its
 * extensions build_adjacency_matrix_kernel.cu:10-17 and gnn_propagate_kernel.cu:8-22.
 * neg_score: float32 [N, lds] = -(X_u X_u^T) over queries followed by gallery (ieee_distmat with IEEE_METRIC_NEG_DOT),
 * N = Q + G.  A: float32 [N, ldA] with ldA = N rounded up to 32, receives the propagated, row-normalised adjacency
 * features; the re-ranked similarity is A[:Q] A[Q:]^T (gnn_reranking.py:55) -- one more contraction by the caller.
 * k1 <= 1024 neighbours, k2 <= k1 of them propagate (k2 == 1: no propagation, as in the reference).
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_gnn_rerank_workspace_bytes(int64_t N, int32_t k1);
int ieee_gnn_rerank(const float* neg_score, int64_t lds, int64_t N, int32_t k1, int32_t k2, float* A, int64_t ldA,
                    void* workspace, size_t workspace_bytes, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * GNN re-ranking, streamed: the A of ieee_gnn_rerank held sparse, computed from packed features (ieee_pack_features with
 * IEEE_METRIC_NEG_DOT, no centre) without any N x N matrix, N = Q + G.  Memory grows linearly in N and in the number
 * of adjacency entries.
 *   ieee_gnn_stream_neighbours computes -(X_u X_u^T) in row strips (queries, then gallery; strip_bytes / ~4N rows, a
 *   multiple of 256) with the contraction, and from each strip the first k1 neighbours `rank` (int32 [N, k1], ties by
 *   index) and S = score^2 (float32 [N, k1]).  No host synchronisation.
 *   ieee_gnn_stream_graph_bytes_sync (symbolic phase) derives every adjacency structure from `rank` alone and waits for
 *   its sizes: sizes (host int64[6]) = {nnz of A, nnz of A's gallery rows, work bytes of ieee_gnn_stream_graph, and
 *   three sizes that call reads back}.  It keeps an index in `scratch` for the next call.
 *   ieee_gnn_stream_graph (numeric phase) writes A as CSR (a_ptr int64 [N + 1], a_col int32 ascending, a_val float32)
 *   and A's gallery rows as CSC (g_ptr int64 [N + 1] over the N columns, g_row int32 gallery indices ascending, g_val
 *   float32).  Structural entries whose value is 0 are kept.  `work` is free again when its work on the stream is done.
 *   ieee_gnn_stream_block writes -(A[q] . A[Q + g]) for queries [row0, row0 + rows) into block (float32 [rows, G],
 *   leading dim ld), summed in float64 (scratch: rows * G doubles) in ascending column order and rounded once: the bits
 *   do not depend on the block size.
 * rank, S and A have the bits ieee_gnn_rerank gives on the -(X_u X_u^T) the contraction writes for the same packed rows;
 * only the final product differs from the dense path's tensor-core contraction (k2 == 1: A holds 0 and 1 and the products
 * are the same integers).  Limits: 1 <= k2 <= k1 <= min(N, 1024), N <= 2^20; precision F16X3 or BF16.
 * ieee_gnn_stream_scratch_bytes needs no GPU and returns 0 (with ieee_last_error set) when the parameters are out of range.
 * ---------------------------------------------------------------------------------------------- */
size_t ieee_gnn_stream_scratch_bytes(int64_t Q, int64_t G, int32_t k1, size_t strip_bytes);
int ieee_gnn_stream_neighbours(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision,
                               int32_t k1, size_t strip_bytes, int32_t* rank, float* S, void* scratch, size_t scratch_bytes,
                               ieee_stream_t stream);
int ieee_gnn_stream_graph_bytes_sync(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                                     size_t scratch_bytes, int64_t* sizes, ieee_stream_t stream);
int ieee_gnn_stream_graph(const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch,
                          size_t scratch_bytes, void* work, size_t work_bytes, const int64_t* sizes, int64_t* a_ptr,
                          int32_t* a_col, float* a_val, int64_t* g_ptr, int32_t* g_row, float* g_val, ieee_stream_t stream);
int ieee_gnn_stream_block(const int64_t* a_ptr, const int32_t* a_col, const float* a_val, const int64_t* g_ptr,
                          const int32_t* g_row, const float* g_val, int64_t Q, int64_t G, int64_t row0, int64_t rows,
                          float* block, int64_t ld, void* scratch, size_t scratch_bytes, ieee_stream_t stream);

/* GNN re-ranking, streamed, in phases: the calls above split so that S processes, each holding the whole gallery and the
 * whole query set, share the work that grows as N^2 and end with the same state.  Every row-parallel kernel computes a
 * row from `rank`, S and the structures before it only, so which process computes a row does not change its bits.
 * ieee_gnn_stream_neighbours is ieee_gnn_stream_neighbours_rows over all rows; ieee_gnn_stream_graph_bytes_sync is
 * ieee_gnn_stream_symbolic over all rows followed by ieee_gnn_stream_sizes_sync; ieee_gnn_stream_graph is the numeric
 * steps (k2 == 1: step 3 only) followed by ieee_gnn_stream_csc, over all rows.  Same limits as above.
 * The owned rows of a process are queries [q0, q1) and gallery rows [g0, g1) (rows Q + g0 to Q + g1 of the N samples),
 * each range starting at a multiple of 256 of its segment and ending at one or at the segment's end, or empty; the CSC
 * columns with the same indices are its owned columns.  Other ranges give IEEE_ERR_INVALID.
 *   ieee_gnn_stream_neighbours_rows writes rank and S of the owned rows.  Exchange: every process needs rank and S of all
 *   N rows before the next call (an all-gather of the owned rows).
 *   ieee_gnn_stream_symbolic builds the index in scratch (every process, all rows: linear in N k1) and counts the nnz of
 *   B1, A1, B2 and A2 of the owned rows into four int32 [N] arrays of scratch (k2 == 1: nothing to count).  No host
 *   synchronisation.  Exchange: every process needs the four counts of all rows (an all-gather of the owned rows; offsets
 *   from ieee_gnn_stream_layout).
 *   ieee_gnn_stream_sizes_sync scans the counts into row offsets and waits for the totals: sizes as
 *   ieee_gnn_stream_graph_bytes_sync gives them, the same on every process.  The one host round trip.
 *   ieee_gnn_stream_numeric, step 0: B1, 1: A1, 2: B2 (after the transpose of the whole A1, computed by every process),
 *   3: A2 into a_ptr (all rows), a_col and a_val.  B1, A1 and B2 are CSR arrays in `work` (offsets from
 *   ieee_gnn_stream_layout).  Each step writes the owned rows' entries and, unless every row is owned, sets every other
 *   row's entries to 0.  Exchange: every process needs all of B1 before step 1, all of A1 before step 2, all of B2 before
 *   step 3, and A2's gallery rows (entries [sizes[0] - sizes[1], sizes[0])) before ieee_gnn_stream_csc.  Because every
 *   entry is 0 on all processes but the one that owns its row, an all-reduce that sums these arrays as int32 moves each
 *   entry's bits exactly.  With k2 == 1 only step 3 exists (A2 = A0).
 *   ieee_gnn_stream_csc builds the CSC of A2's gallery rows (g_ptr of all columns, every process), sorts the owned
 *   columns and, unless every column is owned, sets every other column's entries to 0.  Exchange: g_row and g_val as
 *   above.  Then every process holds the a_ptr, A2's gallery rows and the CSC one process builds, and ieee_gnn_stream_block
 *   serves any of its owned query rows.
 *   ieee_gnn_stream_layout needs no GPU: off[0..3] = byte offsets in scratch of the counts of B1, A1, B2, A2; with sizes
 *   (those of ieee_gnn_stream_sizes_sync), off[4..9] = byte offsets in work of B1's columns and values, A1's columns and
 *   values, B2's columns and values (k2 != 1).
 * Memory: every process holds B1, A1, B2 and the CSC whole while the state is built, as one process does.
 * ---------------------------------------------------------------------------------------------- */
int ieee_gnn_stream_neighbours_rows(const void* q_packed, int64_t Q, const void* g_packed, int64_t G, int64_t D, int precision,
                                    int32_t k1, size_t strip_bytes, int64_t q0, int64_t q1, int64_t g0, int64_t g1, int32_t* rank,
                                    float* S, void* scratch, size_t scratch_bytes, ieee_stream_t stream);
int ieee_gnn_stream_layout(int64_t Q, int64_t G, int32_t k1, int32_t k2, const int64_t* sizes, size_t* off);
int ieee_gnn_stream_symbolic(const int32_t* rank, int64_t Q, int64_t G, int32_t k1, int32_t k2, int64_t q0, int64_t q1, int64_t g0,
                             int64_t g1, void* scratch, size_t scratch_bytes, ieee_stream_t stream);
int ieee_gnn_stream_sizes_sync(int64_t Q, int64_t G, int32_t k1, int32_t k2, void* scratch, size_t scratch_bytes, int64_t* sizes,
                               ieee_stream_t stream);
int ieee_gnn_stream_numeric(int32_t step, const int32_t* rank, const float* S, int64_t Q, int64_t G, int32_t k1, int32_t k2,
                            int64_t q0, int64_t q1, int64_t g0, int64_t g1, void* scratch, size_t scratch_bytes, void* work,
                            size_t work_bytes, const int64_t* sizes, int64_t* a_ptr, int32_t* a_col, float* a_val,
                            ieee_stream_t stream);
int ieee_gnn_stream_csc(int64_t Q, int64_t G, int32_t k1, int64_t q0, int64_t q1, int64_t g0, int64_t g1, void* scratch,
                        size_t scratch_bytes, const int64_t* a_ptr, const int32_t* a_col, const float* a_val, int64_t* g_ptr,
                        int32_t* g_row, float* g_val, ieee_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Peer exchange: the two exchange steps of a gallery sharded over the GPUs of one box (relevant lists to every rank,
 * partial counts to every rank) as STORES into NVLink peer memory from inside the rank kernels, with flag words for
 * the hand-over -- no collective launches between the kernels of a step.
 *
 * Every rank allocates one exchange buffer (ieee_peer_alloc: cudaMalloc, zeroed, plus its 64-byte cudaIpc handle),
 * the handles are exchanged once through the host (any process group), every rank maps its peers' buffers
 * (ieee_peer_open).  Per query block all ranks then call, with identical Qb / cap / W / epoch and their own my_shard:
 *
 *   ieee_rank_gather_peer    lists of this shard -> slot my_shard of EVERY rank's list table
 *   ieee_rank_count_peer     waits for all lists; streams the local rows; partial counts -> slot my_shard of EVERY
 *                            rank's count table
 *   ieee_rank_metrics_peer   waits for all partial counts; sums them (integers: exact in any order); AP / first hit /
 *                            mINP term of every query of the block into this rank's result arrays; on the LAST block
 *                            of the evaluation (q_base + Qb == Qtot) the kernel's last CTA also runs the fixed-tree
 *                            reduction over all Qtot queries: bit-identical (cmc, summary) on every rank without a
 *                            result broadcast.  cmc / summary may be NULL for earlier blocks.  stats_out (int64[3],
 *                            device, may be NULL) receives {list overflow (needed capacity or 0), tie pairs, longest
 *                            merged list} over all shards.
 * Two hand-overs per block suffice (a first version had a third, owner -> everybody): seeing a peer's count flag of block n
 * says its count kernel is done with the lists, seeing its list flag of block n + 1 says its metrics kernel is done
 * with the count rows, so the next block may overwrite both.
 * A kernel that waits spins on flags in its OWN buffer (bounded: it traps after ~4 s); it never waits for a kernel of
 * the same rank that is queued behind it, so the ranks cannot deadlock as long as all of them issue the same calls.
 * `epoch` must grow by one per query block (never reuse a value with the same buffers).
 * ---------------------------------------------------------------------------------------------- */
#define IEEE_MAX_PEERS 16
typedef struct {
  int32_t shards, my_shard;
  uint64_t epoch;
  void* base[IEEE_MAX_PEERS]; /* exchange buffer of every shard as mapped into THIS process (base[my_shard]: own) */
  int64_t Qb_max, Qb, Qtot, q_base; /* rows of the largest block (sizes the buffer); rows of this block; rows of the
                                       whole evaluation; first row of this block */
  int32_t cap, W;             /* per-shard list capacity; count-row width (>= longest merged list, <= shards * cap) */
} ieee_peer_exchange;

size_t ieee_peer_exchange_bytes(int64_t Qb_max, int64_t Qtot, int32_t cap, int32_t W, int32_t shards);
int ieee_peer_alloc(size_t bytes, void** ptr, void* ipc_handle_out /* 64 bytes, host */);
int ieee_peer_open(const void* ipc_handle /* 64 bytes, host */, void** ptr);
int ieee_peer_close(void* ptr);
int ieee_peer_free(void* ptr);
/* stats: uint64[4] of device memory private to this rank, zeroed by the caller once per evaluation:
 * [0] gather overflow (int32), [1] tie pairs, [2] longest merged list. */
int ieee_rank_gather_peer(const float* distmat, int64_t ld, int64_t G, const int64_t* q_pids, const int64_t* q_camids,
                          const int64_t* g_camids, const void* group, int64_t g_offset, int32_t* n_rel, uint64_t* junk,
                          int32_t* n_junk, unsigned long long* stats, const ieee_peer_exchange* ex, ieee_stream_t stream);
int ieee_rank_count_peer(const float* distmat, int64_t ld, int64_t G, int64_t g_offset, const int32_t* n_rel,
                         const uint64_t* junk, const int32_t* n_junk, unsigned long long* stats,
                         const ieee_peer_exchange* ex, ieee_stream_t stream);
int ieee_rank_metrics_peer(int64_t G_total, int32_t max_rank, const unsigned long long* stats, float* cmc,
                           ieee_eval_summary* summary, int64_t* stats_out, const ieee_peer_exchange* ex,
                           ieee_stream_t stream);
/* One query block of a sharded evaluation in ONE call (the sharded counterpart of ieee_retrieve_eval_prepared): pack the
 * queries -> contraction against this rank's packed gallery slice -> gather / count / metrics with the peer
 * exchange.  `ex` describes one block of Q rows (Qb == Qtot == Q, q_base == 0) with the list capacity and row width
 * every rank agreed on; G_total / g_offset place the slice in the whole gallery.  stats_out as in ieee_rank_metrics_peer:
 * stats_out[0] != 0 or stats_out[2] > ex->W mean the sizes were too small and the call must be repeated with larger ones. */
size_t ieee_retrieve_prepared_peer_workspace_bytes(int64_t Q, int64_t D, int precision, int32_t cap);
int ieee_retrieve_eval_prepared_peer(const void* qf, int64_t ldq, int dtype, int64_t Q, int64_t D, int metric, int normalize,
                                     int precision, const void* g_packed, const void* group, const float* center, int64_t G,
                                     int64_t G_total, int64_t g_offset, const int64_t* q_pids, const int64_t* q_camids,
                                     const int64_t* g_camids, int32_t max_rank, float* distmat, int64_t ld, float* cmc,
                                     ieee_eval_summary* summary, int64_t* stats_out,
                                     double* per_query_ap /* double[Q], may be NULL: then in the exchange buffer */,
                                     int32_t* per_query_first /* int32[Q], may be NULL */, const ieee_peer_exchange* ex,
                                     const void* q_packed /* as in ieee_retrieve_eval_prepared */, void* workspace,
                                     size_t workspace_bytes, ieee_stream_t stream);
/* Byte offset of a per-query result array inside an exchange buffer: which = 0 AP (double[Qtot]), 1 first hit
 * (int32[Qtot]), 2 mINP term (double[Qtot]), 3 short-list flag (int32[Qtot]). */
size_t ieee_peer_result_offset(int which, int64_t Qb_max, int64_t Qtot, int32_t cap, int32_t W, int32_t shards);

#ifdef __cplusplus
}
#endif
#endif /* IEEE_B200_H_ */
