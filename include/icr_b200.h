/*
 * icr_b200.h — C ABI of the B200-native retrieval hot path (cosine scoring + top-k,
 * dense cos_sim, MultipleNegativesRankingLoss fwd/bwd, shard-candidate merge).
 *
 * This header is the drop-in boundary. The reference (chen-bowen/instacart_next_order_
 * recommendation) has no FFI of its own: the calls replaced are Python calls into
 * sentence-transformers 5.2.2 + torch. Each entry point cites the reference call site it
 * stands in for. INTEGRATION.md shows the ctypes binding a reference maintainer would add.
 *
 * Conventions
 *   - Plain C, no C++ types or exceptions cross this line.
 *   - Every pointer except `stream` is a DEVICE pointer owned by the caller. The library
 *     never allocates or frees device memory and keeps no pointer after return.
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued on it and the call
 *     returns without synchronising.
 *   - Matrices are row-major, contiguous in the embedding dimension, `ld*` = row stride in
 *     ELEMENTS. Row starts must be 16-byte aligned.
 *   - Return value: 0 = ok, negative = icr_status; icr_last_error_string() gives the text
 *     for the calling thread. There is no CPU fallback: a device that is not sm_100 is
 *     ICR_ERR_DEVICE.
 */
#ifndef ICR_B200_H
#define ICR_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ICR_ABI_VERSION 3
#define ICR_MAX_K 256 /* largest k of one fused top-k call (reference: top_k <= 100, schemas.py:34) */

typedef enum {
  ICR_OK = 0,
  ICR_ERR_ARG = -1,       /* bad shape / stride / null pointer           */
  ICR_ERR_DTYPE = -2,     /* dtype not supported by this entry point     */
  ICR_ERR_ALIGN = -3,     /* pointer or row stride not 16-byte aligned   */
  ICR_ERR_K = -4,         /* k < 1 or k > ICR_MAX_K                      */
  ICR_ERR_WORKSPACE = -5, /* workspace too small (see *_workspace_bytes) */
  ICR_ERR_CUDA = -6,      /* CUDA runtime / driver error                 */
  ICR_ERR_DEVICE = -7     /* current device is not sm_100                */
} icr_status;

typedef enum {
  ICR_F32 = 0,
  ICR_BF16 = 1,
  ICR_F16 = 2 /* embeddings as the reference's fp16-autocast training produces them (train_sbert.py:210,232); the MNRL entry
                points, and catalogs of icr_cos_topk / icr_cos_sim_dense: 2 bytes per element like bf16, 8x finer rounding */
} icr_dtype;

/* which kernel family serves a cos_topk call */
typedef enum {
  ICR_PATH_AUTO = 0,
  ICR_PATH_GEMV = 1, /* K1: streaming CUDA-core GEMV + fused top-k, small query batches */
  ICR_PATH_GEMM = 2  /* K2: tcgen05/TMEM GEMM + threshold-filter epilogue                */
} icr_path;
/* OR-ed into `path`: the workspace is RESIDENT — the caller zero-filled it once and since then only icr_cos_topk calls of
 * the same shape, on one stream, have used it. The GEMV path then skips re-zeroing its two counters - the merge ticket and
 * the slab-chunk counter of the ring kernel, both left at zero by the merging CTA: one memset less on the latency path of
 * a request. */
#define ICR_PATH_WS_RESIDENT 0x100

int icr_abi_version(void);
const char* icr_last_error_string(void);
/* 1 if the CURRENT device is compute capability 10.x, 0 otherwise, <0 on CUDA error. */
int icr_device_supported(void);

/* ---------------------------------------------------------------------------------------
 * Catalog preparation (once per index load; replaces the per-call re-normalisation that
 * sentence_transformers.util.cos_sim does on every /recommend,
 * reference src/inference/serve_recommendations.py:214,250).
 *   inv_norms[r] = 1 / max(||x_r||_2, 1e-12)            (F.normalize's eps; x: ICR_F32, ICR_BF16 or ICR_F16)
 * ------------------------------------------------------------------------------------- */
int icr_row_inv_norms(const void* x, int64_t rows, int64_t dim, int64_t ld, int dtype,
                      float* inv_norms, void* stream);

/* fp32 rows -> L2-normalised, scaled by 2^8 and split into an fp16 (hi | lo) pair per row:
 * planes[r, 0:dim] = hi, planes[r, dim_pad:dim_pad+dim] = lo, row stride 2*dim_pad fp16
 * elements, dim_pad = dim rounded up to 64, padding zero-filled. This is the operand
 * format of the fp32-parity DENSE tensor-core path (icr_cos_sim_dense: three fp16 MMAs with fp32 accumulation builds these
 * per call); exported for callers that want the planes themselves. */
int icr_split_f16_planes(const float* x, int64_t rows, int64_t dim, int64_t ld,
                         uint16_t* planes, void* stream);
int64_t icr_planes_row_elems(int64_t dim); /* = 2 * round_up(dim, 64) */

/* fp32 rows -> the SCREENING operand of the tensor-core top-k path: plane[r, 0:dim] = fp16(256 * x_r / max(||x_r||, 1e-12)),
 * row stride dim_pad = round_up(dim, 64) fp16 elements, padding zero-filled; inv_norms[r] (optional, may be NULL) as
 * icr_row_inv_norms. One fp16 MMA term on these planes bounds every cosine to within 2^-10; icr_cos_topk keeps every row
 * whose screened score lies within twice that of the k-th best and re-scores those few rows exactly in fp32 from the
 * caller's rows, so the returned scores and ids are those of the fp32 computation. */
int icr_screen_plane(const float* x, int64_t rows, int64_t dim, int64_t ld,
                     uint16_t* plane, float* inv_norms, void* stream);
int64_t icr_screen_plane_row_elems(int64_t dim); /* = round_up(dim, 64) */

/* Catalog upload helper: fp32 rows as the reference stores them on disk (embeddings.npy,
 * src/inference/serve_recommendations.py:127) -> the HBM-resident form: ICR_F32, ICR_BF16 or ICR_F16
 * (round to nearest even, bit for bit torch's .to(); fp16 overflows to +-inf and keeps subnormals), optionally
 * L2-normalised first (x / max(||x||, 1e-12) in fp32, the reference normalises at encode time, :195-200). x and out are
 * device pointers; dim % 4 == 0. */
int icr_convert_rows(const float* x, int64_t rows, int64_t dim, int64_t ldx,
                     void* out, int64_t ldo, int out_dtype, int normalize, void* stream);

/* ---------------------------------------------------------------------------------------
 * Fused cosine top-k  ==  torch.topk(cos_sim(queries, catalog), k, dim=1, sorted=True)
 * with ties broken by the lower catalog row.
 * Stands in for: cos_sim + argsort + walk (serve_recommendations.py:213-225, 250-262);
 * cos_sim + torch.topk(100) + heap merge inside InformationRetrievalEvaluator (constructed
 * at src/training/train_sbert.py:197-202); cos_sim + np.argsort per row
 * (src/baselines/content_based.py:54-63, scripts/compare_untrained_vs_trained.py:74-84).
 *
 *   queries      [Q, D] dtype, row stride ldq
 *   catalog      [N, D] dtype, row stride ldc          (the shard's rows when sharded)
 *   dtype        ICR_F32, ICR_BF16 or ICR_F16, shared by queries and catalog; the 16-bit types need D % 8 == 0.
 *                ICR_F16 scores are fp32 arithmetic on the fp16 values (products of two fp16 numbers are exact in
 *                fp32): no screening, no re-scoring
 *   cat_planes   optional (may be NULL): the plane of icr_screen_plane(catalog), [N, round_up(D, 64)] fp16;
 *                used by the GEMM path for ICR_F32 catalogs; if NULL it is built in the workspace per call
 *   cat_inv_norms optional (may be NULL): icr_row_inv_norms(catalog); used by the GEMM path (ICR_BF16, ICR_F16:
 *                epilogue scaling; ICR_F32: exact re-scoring of the screened rows); if NULL it is computed per call
 *   exclude_mask optional (may be NULL): N bytes, non-zero = row never returned
 *                (exclude_product_ids semantics, serve_recommendations.py:216-221)
 *   row_offset   added to every returned id (global numbering of a row shard)
 *   out_scores   [Q, k] f32 descending; out_ids [Q, k] i64. If fewer than k rows are
 *                eligible the tail is (-inf, -1). Both are only ever written; they may be pinned,
 *                device-mapped HOST memory (cudaHostAlloc): the last kernel of the call then
 *                delivers the result over PCIe itself and a request needs no device-to-host copy
 *                (DeviceCatalog.topk_request; every other pointer must be device memory).
 * ------------------------------------------------------------------------------------- */
size_t icr_cos_topk_workspace_bytes(int64_t Q, int64_t N, int64_t D, int dtype, int k, int path,
                                    int have_planes);
int icr_cos_topk(const void* queries, int64_t Q, int64_t ldq,
                 const void* catalog, int64_t N, int64_t ldc,
                 int64_t D, int dtype,
                 const uint16_t* cat_planes, const float* cat_inv_norms,
                 const uint8_t* exclude_mask,
                 int k, int64_t row_offset, int path,
                 float* out_scores, int64_t* out_ids,
                 void* workspace, size_t workspace_bytes, void* stream);

/* Per-query exclusions: a bitmap `bits` uint32 [ceil(N/32)][Q] (device memory, 4-byte aligned). Row r of the catalog
 * (a local row, before row_offset) is excluded for query q when bit r % 32 of bits[r / 32][q] is set. The word index
 * is outermost: the 32 rows a kernel filters together share one word, and 32 consecutive queries read one 128-byte
 * line. Q * ceil(N/32) * 4 bytes: 6.2 KB per query on a 49,688-row catalog.
 *
 * icr_query_exclusion_bits builds it from a CSR list (the convention of icr_ir_metrics): query q excludes
 * rows[offsets[q] .. offsets[q+1]), in any order, duplicates allowed; rows outside [0, N) are ignored, as the
 * reference skips excluded ids that are not in the catalog. offsets [Q + 1] and rows are device memory. One memset and
 * one scatter kernel on `stream`; a caller that reuses an exclusion set across calls builds it once. */
int icr_query_exclusion_bits(const int64_t* offsets, const int64_t* rows, int64_t Q, int64_t N,
                             uint32_t* bits, void* stream);

/* icr_cos_topk with per-query exclusions `excl_bits` (the bitmap above, for these Q queries and N rows; NULL = none,
 * which is exactly icr_cos_topk). Given together with exclude_mask, a row is excluded when either says so. Same
 * workspace (icr_cos_topk_workspace_bytes) and the same plan: the bitmap changes only which rows are eligible. If fewer
 * than k rows are eligible for a query, its tail is (-inf, -1). Not available on the sharded entry. */
int icr_cos_topk_excl(const void* queries, int64_t Q, int64_t ldq,
                      const void* catalog, int64_t N, int64_t ldc,
                      int64_t D, int dtype,
                      const uint16_t* cat_planes, const float* cat_inv_norms,
                      const uint8_t* exclude_mask, const uint32_t* excl_bits,
                      int k, int64_t row_offset, int path,
                      float* out_scores, int64_t* out_ids,
                      void* workspace, size_t workspace_bytes, void* stream);

/* number of kernel launches the last icr_cos_topk call on this thread enqueued */
int icr_last_launch_count(void);

/* Optional timing of the dominant kernel of subsequent calls made by this thread (used by bench.py for
 * the roofline figure): CUDA events are recorded on the call's stream around each launch of the GEMV /
 * GEMM scoring kernel. collect() waits for the recorded events and returns their summed duration;
 * kernel_id 1 = gemv_topk, 2 = gemm_topk; mma_terms = fp16 MMA products issued per algorithmic product. */
int icr_profile_enable(int on);
int icr_profile_collect(float* total_ms, int* launches, int* kernel_id, int* mma_terms);

/* ---------------------------------------------------------------------------------------
 * Dense cosine similarity  ==  sentence_transformers.util.cos_sim(a, b) -> f32 [Qa, Nb]
 * (hook-compatible path: MNRL similarity_fct, evaluator score_functions).
 * a and b share dtype: ICR_F32, ICR_BF16 or ICR_F16 (16-bit types: D % 8 == 0).
 * ------------------------------------------------------------------------------------- */
size_t icr_cos_sim_dense_workspace_bytes(int64_t Qa, int64_t Nb, int64_t D, int dtype);
int icr_cos_sim_dense(const void* a, int64_t Qa, int64_t lda,
                      const void* b, int64_t Nb, int64_t ldb,
                      int64_t D, int dtype,
                      float* out, int64_t ldo,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Shard-candidate merge (K4): G lists of k_in (score, id) per query, as gathered by an
 * allgather of every rank's icr_cos_topk output, -> global top-k_out. Replaces the
 * per-chunk Python heapq merge of InformationRetrievalEvaluator.
 *   cand_scores [G, Q, k_in] f32, cand_ids [G, Q, k_in] i64 (id < 0 = empty slot)
 * ------------------------------------------------------------------------------------- */
size_t icr_topk_merge_workspace_bytes(int64_t Q, int G, int k_in, int k_out);
int icr_topk_merge(const float* cand_scores, const int64_t* cand_ids,
                   int64_t Q, int G, int k_in, int k_out,
                   float* out_scores, int64_t* out_ids,
                   void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * Shard-candidate exchange over NVLink peer memory (K4x): the all-gather of every rank's
 * icr_cos_topk output without NCCL. No reference counterpart (the reference is single-GPU).
 * The host allocates one symmetric buffer of icr_peer_buffer_bytes() per rank, zero-filled,
 * mapped into every peer (e.g. torch.distributed._symmetric_memory), and passes the world's
 * buffer addresses AS SEEN FROM THIS PROCESS in `peer_buffers` (HOST array, index = rank).
 * `epoch` is the 1-based count of exchange calls on this buffer, identical on all ranks.
 *   scores [n] f32, ids [n] i64: this rank's candidates (n = Q * k <= n_max)
 * On return (stream order) the local buffer holds scores [world][n] at *scores_off and
 * ids [world][n] at *ids_off (byte offsets from the local buffer's base), the inputs
 * icr_topk_merge expects with G = world. Every rank must make the same call.
 * ------------------------------------------------------------------------------------- */
#define ICR_MAX_PEERS 16
size_t icr_peer_buffer_bytes(int64_t n_max, int world);
int icr_peer_exchange(const float* scores, const int64_t* ids, int64_t n, int rank, int world,
                      const uint64_t* peer_buffers, uint32_t epoch, int64_t n_max,
                      size_t* scores_off, size_t* ids_off, void* stream);

/* Exchange AND merge in one kernel (K4f): this rank's [Q, k] lists (descending or not) are pushed to every peer as in
 * icr_peer_exchange, and the same launch waits for the peers' lists and writes the global top-k of every query to
 * out_scores / out_ids [Q, k] - the result of icr_peer_exchange followed by icr_topk_merge(G = world, k_in = k_out = k).
 * Same buffers, epochs and lock-step rule as icr_peer_exchange (the two may be mixed call by call, and a rank may use one
 * while its peers use the other). Global ids must lie below 2^32 - 1, as for icr_topk_merge. */
int icr_peer_exchange_merge(const float* scores, const int64_t* ids, int64_t Q, int k, int rank, int world,
                            const uint64_t* peer_buffers, uint32_t epoch, int64_t n_max,
                            float* out_scores, int64_t* out_ids, void* stream);

/* One rank's call of a search over a ROW-SHARDED catalog: icr_cos_topk over this rank's shard (arguments and dtypes as there;
 * row_offset = global id of the shard's first row), the exchange of every rank's [Q, k] candidates over NVLink peer memory
 * and the merge - out_scores / out_ids [Q, k] receive the GLOBAL top-k, identical on every rank. Every rank of the group
 * makes the same call (same Q, k, epoch; the shards may differ in size). Request-sized batches (Q <= 7 on the GEMV path,
 * world * k keys within the kernel's merge buffer) are ONE launch: the CTA that merges the shard's partial lists pushes the
 * result to the peers, waits for theirs and merges them, all in the kernel's tail. Larger batches: the local search, then
 * the K4f kernel. No reference counterpart (the reference is single-GPU); the single-GPU call it extends stands in for
 * serve_recommendations.py:213-225. */
size_t icr_cos_topk_sharded_workspace_bytes(int64_t Q, int64_t N, int64_t D, int dtype, int k, int path,
                                            int have_planes);
int icr_cos_topk_sharded(const void* queries, int64_t Q, int64_t ldq,
                         const void* catalog, int64_t N, int64_t ldc,
                         int64_t D, int dtype,
                         const uint16_t* cat_planes, const float* cat_inv_norms,
                         const uint8_t* exclude_mask,
                         int k, int64_t row_offset, int path,
                         int rank, int world, const uint64_t* peer_buffers, uint32_t epoch, int64_t n_max,
                         float* out_scores, int64_t* out_ids,
                         void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * MultipleNegativesRankingLoss (sentence-transformers; constructed at
 * src/training/train_sbert.py:182-185):
 *   loss = mean_i CE( scale * cos_sim(A, P)[i, :], i )
 * fwd saves per-row lse / inverse norms for bwd. Internal math is fp32.
 *   a, p        [B, D] dtype (ICR_F32, ICR_BF16 or ICR_F16);  loss: 1 float;  lse, inv_a, inv_p: B floats each
 *   grad_out    1 float (dL/dloss);  grad_a, grad_p [B, D] dtype (row strides ldga, ldgp)
 * ------------------------------------------------------------------------------------- */
size_t icr_mnrl_workspace_bytes(int64_t B, int64_t D);
int icr_mnrl_fwd(const void* a, int64_t lda, const void* p, int64_t ldp,
                 int64_t B, int64_t D, int dtype, float scale,
                 float* loss, float* lse, float* inv_a, float* inv_p,
                 void* workspace, size_t workspace_bytes, void* stream);
int icr_mnrl_bwd(const void* a, int64_t lda, const void* p, int64_t ldp,
                 int64_t B, int64_t D, int dtype, float scale,
                 const float* lse, const float* inv_a, const float* inv_p,
                 const float* grad_out,
                 void* grad_a, int64_t ldga, void* grad_p, int64_t ldgp,
                 void* workspace, size_t workspace_bytes, void* stream);
/* Forward and backward in one call: loss plus the gradients for dL/dloss = 1 (a training step always wants both; the
 * caller multiplies by the incoming gradient). Same outputs as icr_mnrl_fwd followed by icr_mnrl_bwd with grad_out = 1. */
int icr_mnrl_fwd_bwd(const void* a, int64_t lda, const void* p, int64_t ldp,
                     int64_t B, int64_t D, int dtype, float scale,
                     float* loss, float* lse, float* inv_a, float* inv_p,
                     void* grad_a, int64_t ldga, void* grad_p, int64_t ldgp,
                     void* workspace, size_t workspace_bytes, void* stream);
/* out = grad * grad_out[0] for the two [n]-element gradients of icr_mnrl_fwd_bwd (n = B * D, contiguous): what
 * autograd's backward does with the incoming dL/dloss. grad_out is a device scalar. */
int icr_mnrl_scale_grads(const void* grad_a, const void* grad_p, int64_t n, int dtype, const float* grad_out,
                         void* out_a, void* out_p, void* stream);

/* Rectangular form for cross-device in-batch negatives (sentence-transformers'
 * gather_across_devices=True; not enabled by the reference, src/training/train_sbert.py:184-185):
 * B local anchors against Bc >= B candidates (the positives of all ranks, gathered), the positive
 * of anchor i at candidate i + label_offset (= rank * B).
 *   loss = mean_i CE( scale * cos_sim(A, C)[i, :], i + label_offset )
 * grad_c [Bc, D] is this rank's contribution to every candidate's gradient (the host
 * reduce-scatters it). Tensor-core path only: D % 8 == 0. */
size_t icr_mnrl_rect_workspace_bytes(int64_t B, int64_t Bc, int64_t D);
int icr_mnrl_fwd_rect(const void* a, int64_t lda, const void* c, int64_t ldc,
                      int64_t B, int64_t Bc, int64_t label_offset, int64_t D, int dtype, float scale,
                      float* loss, float* lse, float* inv_a, float* inv_c,
                      void* workspace, size_t workspace_bytes, void* stream);
int icr_mnrl_bwd_rect(const void* a, int64_t lda, const void* c, int64_t ldc,
                      int64_t B, int64_t Bc, int64_t label_offset, int64_t D, int dtype, float scale,
                      const float* lse, const float* inv_a, const float* inv_c,
                      const float* grad_out,
                      void* grad_a, int64_t ldga, void* grad_c, int64_t ldgc,
                      void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------
 * IR metric arithmetic over the retrieved ids (the evaluator's host tail, on the device).
 * Stands in for the per-query Python loops of sentence-transformers'
 * InformationRetrievalEvaluator.compute_metrics (evaluator built at
 * src/training/train_sbert.py:197-202, key read at :220) and of the in-tree
 * src/baselines/metrics.py:13-176 (compute_ir_metrics), whose NDCG / AP normalisers differ:
 * the *_RETRIEVED kinds follow metrics.py (:112-119 ideal ordering of the retrieved
 * relevances; :66-72 AP / min(|relevant|, |ranked|)).
 *
 *   ids         [Q, K] i64 (row stride ld_ids), best first, id < 0 = no result (K <= ICR_MAX_K)
 *   rel_offsets [Q+1] i64, rel_rows[rel_offsets[q] : rel_offsets[q+1]] = the relevant catalog
 *               rows of query q that exist in the catalog, ASCENDING
 *   n_relevant  [Q] i32 = len(relevant_docs[qid]) (may exceed the segment length when a
 *               relevant id is not in the catalog); a query with 0 scores 0 on every metric
 *   kinds, ks   HOST arrays of M metric kinds / cut-offs (copied into the launch parameters)
 *   per_query   [Q, M] f64 out: metric m of query q
 *   means       [M] f64 out: mean over the Q queries, summed in a fixed order
 * ------------------------------------------------------------------------------------- */
typedef enum {
  ICR_METRIC_ACCURACY = 0,
  ICR_METRIC_PRECISION = 1,
  ICR_METRIC_RECALL = 2,
  ICR_METRIC_MRR = 3,
  ICR_METRIC_NDCG = 4,           /* IDCG = min(n_relevant, k) ones (sentence-transformers) */
  ICR_METRIC_MAP = 5,            /* AP / min(k, n_relevant)   (sentence-transformers)      */
  ICR_METRIC_NDCG_RETRIEVED = 6, /* IDCG = the retrieved hits moved to the front (metrics.py:112-119) */
  ICR_METRIC_MAP_RETRIEVED = 7   /* AP / min(n_relevant, #retrieved in the first k) (metrics.py:66-72) */
} icr_metric_kind;
#define ICR_MAX_METRICS 32
int icr_ir_metrics(const int64_t* ids, int64_t Q, int K, int64_t ld_ids,
                   const int64_t* rel_offsets, const int64_t* rel_rows, const int32_t* n_relevant,
                   const int32_t* kinds, const int32_t* ks, int M,
                   double* per_query, double* means, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ICR_B200_H */
