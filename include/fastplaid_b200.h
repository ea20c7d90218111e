/*
 * fastplaid_b200.h -- C ABI of the B200-native PLAID search engine.
 *
 * This is the drop-in boundary for the search hot path of lightonai/fast-plaid
 * (v1.4.6 @ 87f96f6).  In the reference that path sits behind the PyO3 module
 * `fast_plaid.fast_plaid_rust` (rust/lib.rs:366-383).  Each entry point below names the
 * reference interface it replaces.  Conventions:
 *
 *   - plain C types only; every pointer named `d_*` is a DEVICE pointer on the index's
 *     GPU, every pointer named `h_*` is a HOST pointer, `stream` is a cudaStream_t
 *     passed as void* (NULL = legacy default stream);
 *   - every function returns 0 on success or a negative code; the message is available
 *     from fpb_last_error() (thread-local).  No exception crosses the boundary.  The
 *     reference's PyValueError / PyRuntimeError (rust/utils/errors.rs:5-7) are raised by
 *     the Python host from these codes;
 *   - all entry points are asynchronous w.r.t. the host on `stream` unless their name
 *     ends in `_host` (those synchronise the stream before returning);
 *   - an fpb_index is immutable after creation and may be searched concurrently from
 *     several host threads on different streams with different workspaces, like the
 *     reference's `LoadedIndex` (`unsafe impl Send/Sync`, rust/search/load.rs:58-59).
 *     It does NOT own the big arrays: the caller (PyTorch) keeps them alive.
 */
#ifndef FASTPLAID_B200_H_
#define FASTPLAID_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FPB_OK 0
#define FPB_ERR_INVALID (-1)  /* bad argument -> Python ValueError  (errors.rs:5-7)   */
#define FPB_ERR_CUDA (-2)     /* CUDA runtime failure -> RuntimeError                  */
#define FPB_ERR_UNSUPPORTED (-3)
#define FPB_ERR_WORKSPACE (-4) /* workspace too small                                  */
#define FPB_ERR_NO_IVF (-5)   /* compress_only index: search refused (search.rs:227-232) */

typedef struct fpb_index fpb_index;
struct fpb_record;

/* Thread-local message of the last failing call in this thread. */
const char* fpb_last_error(void);
/* ABI version (bumped on any signature change). */
int fpb_abi_version(void);

/*
 * fpb_index_create  -- replaces `construct_index` (rust/search/load.rs:122-186) and
 * `ResidualCodec::load` (rust/utils/residual_codec.rs:72-152).
 *
 *   d_centroids       f16 [n_centroids, dim], row-major            (load.rs:145)
 *   d_bucket_weights  f16 [1 << nbits]                              (load.rs:150)
 *   d_doc_offsets     i64 [n_docs + 1], exclusive cumsum of doclens (tensor.rs:221-224)
 *   d_doc_codes       i32 [n_tokens]   (narrowed from the on-disk int64 by the loader)
 *   d_doc_residuals   u8  [n_tokens, dim*nbits/8]
 *   d_token_norms     f16 [n_tokens]  OUTPUT, caller-owned like the other arrays: filled here with the fp16 norm of
 *                     every decompressed token (the `norm(...)` of decompress_residuals, search.rs:86-93), which the
 *                     MaxSim / reconstruct kernels then read instead of recomputing it per (query, document) pair
 *   d_ivf_offsets     i64 [n_centroids + 1]  or NULL for a compress_only index
 *   d_ivf_pids        i32 [n_ivf]            (LOCAL doc ids, ascending within a list)
 *   doc_id_base       global id of local doc 0 (document sharding; 0 on one GPU)
 *
 * The two 256-entry LUTs of the reference collapse into one (1<<nbits)-entry permuted
 * weight table w_perm[i] = bucket_weights[bitrev_nbits(i)] built here on the host.
 */
int fpb_index_create(fpb_index** out, int device, int nbits, int dim, int64_t n_centroids,
                     const void* d_centroids, const void* d_bucket_weights, int64_t n_docs,
                     const int64_t* d_doc_offsets, const int32_t* d_doc_codes,
                     const uint8_t* d_doc_residuals, void* d_token_norms, const int64_t* d_ivf_offsets,
                     const int32_t* d_ivf_pids, int64_t n_ivf, int64_t max_doc_len,
                     int64_t doc_id_base);
void fpb_index_destroy(fpb_index* index);

/* Search parameters -- mirrors `SearchParameters` (rust/search/search.rs:171-200).
 * `batch_size` (document batch of the approximate stage) only bounds memory in the
 * reference and does not change values (search.rs:558-586); it is accepted and ignored. */
typedef struct fpb_params {
  int32_t n_ivf_probe;   /* search.rs:185, default 8    */
  int32_t n_full_scores; /* search.rs:179, default 4096 */
  int32_t top_k;         /* search.rs:182               */
  int32_t batch_size;    /* search.rs:176, ignored      */
  int32_t flags;         /* FPB_FLAG_*                  */
} fpb_params;

/* The workspace carries the per-query subset structures (search.rs:494-517, :544-547). */
#define FPB_FLAG_SUBSET 1
/* Approximate stage (search.rs:554-592).  By default it is computed in two exact passes: a bound pass
 * that gathers only the score rows of "high" centroids and yields, per candidate, an upper and a lower
 * bound of its approximate score (equal when the candidate is resolved), then an exact pass over the
 * unresolved candidates whose upper bound reaches the n_full_scores/4-th best lower bound.  Every
 * candidate that can enter the pruned list carries its exact score; the others keep an upper bound that
 * is strictly below the pruning threshold, so the pruned list, its scores and everything after it are
 * bit-identical to scoring every candidate.
 *   FPB_FLAG_APPROX_EXACT_ALL : also refine the candidates below the threshold (off_approx then holds
 *                               the exact score of EVERY candidate; parity tests)
 *   FPB_FLAG_APPROX_DIRECT    : one-pass scoring of every candidate (the A/B alternative)
 *   FPB_FLAG_APPROX_TWO_PASS  : two passes whatever the size of the job
 * With none of them the library picks: the two passes carry ~0.5 ms of fixed cost (threshold sample, bitmap,
 * refine list), so a call whose batch x index is too small to repay it (B * n_tokens < 2e8) is scored in one pass. */
#define FPB_FLAG_APPROX_EXACT_ALL 2
#define FPB_FLAG_APPROX_DIRECT 4
#define FPB_FLAG_APPROX_TWO_PASS 8

/* Byte offsets of every intermediate inside the workspace, so the parity tests can read
 * each stage (S, probed cells, candidates, approx scores, rerank list, exact scores)
 * exactly as the oracle dumps them.  All offsets are multiples of 256. */
typedef struct fpb_layout {
  int64_t total_bytes;
  int32_t B, Q, Qp, n_tiles, R, n_probe, cand_cap, bitmap_words;
  int32_t cbitmap_words, reserved0;
  int64_t off_queries;   /* f16 [B, Qp, D]  zero-padded queries                       */
  int64_t off_S;         /* f16 [B, K, Qp]  centroid scores          (search.rs:491)  */
  int64_t off_tmax;      /* f16 [B, Qp, n_tiles] per-128-centroid-tile column maxima  */
  int64_t off_cells;     /* i32 [B, Q, n_probe]  probed cells        (search.rs:520-528) */
  int64_t off_bitmap;    /* u32 [B, bitmap_words]                                     */
  int64_t off_n_cand;    /* i32 [B]                                                   */
  int64_t off_cand;      /* i32 [B, cand_cap] sorted unique doc ids  (search.rs:535-541) */
  int64_t off_approx;    /* f32 [B, cand_cap]                        (search.rs:554-592) */
  int64_t off_work;      /* i32 [B + 8] chunk prefix + counters                       */
  int64_t off_n_rerank;  /* i32 [B]                                                   */
  int64_t off_rerank;    /* i32 [B, R] doc ids, (approx desc, id asc) (search.rs:602-619) */
  int64_t off_rerank_approx; /* f32 [B, R]                                            */
  int64_t off_exact;     /* f32 [B, R]                               (search.rs:651-656) */
  /* only with FPB_FLAG_SUBSET (otherwise zero-sized): */
  int64_t off_cbitmap;   /* u32 [B, cbitmap_words] centroids present in the subset docs (search.rs:496-503) */
  int64_t off_clist;     /* i32 [B, K] the same as a sorted list                      */
  int64_t off_n_clist;   /* i32 [B]                                                   */
  int64_t off_sbitmap;   /* u32 [B, bitmap_words] the subset's documents              */
  /* two-pass approximate stage: */
  int64_t off_tau;       /* f16 [B, Qp]  per query token the "high" score threshold (+inf on padded columns) */
  int64_t off_hibits;    /* u32 [B, hb_words] centroid c is high: exists q with S[b,c,q] >= tau[b,q] */
  int64_t off_lb;        /* f32 [B, cand_cap] lower bound of the approximate score (== off_approx entry when resolved) */
  int64_t off_refine;    /* i32 [B, cand_cap] candidate indices re-scored exactly by the second pass */
  int64_t off_n_refine;  /* i32 [B]                                                   */
  int64_t off_thresh;    /* f32 [B] pruning threshold used by the second pass (-inf: refine all) */
  int64_t off_work2;     /* i32 [B + 8] chunk prefix + counter of the second pass     */
  int64_t off_stats;     /* u64 [8] counters: [0] rows gathered by the bound pass, [1] tokens walked by it,
                            [2] rows gathered by the exact pass (accumulated until the caller clears them) */
  int32_t hb_words, flags; /* flags = params->flags the layout was made for */
} fpb_layout;

/* Workspace sizing for a batch of B queries of Q tokens. */
int fpb_workspace_layout(const fpb_index* index, int B, int Q, const fpb_params* params,
                         fpb_layout* out);

/*
 * fpb_search_batch -- replaces `pysearch` -> `search_many` -> `search`
 * (rust/lib.rs:195-223, rust/search/search.rs:219-288, :471-696) for a whole batch.
 *
 *   d_queries     f16 [B, Q, dim]  (already cast to fp16, fast_plaid.py:241)
 *   d_out_ids     i64 [B, top_k]   global doc ids, rank order
 *   d_out_scores  f32 [B, top_k]
 *   d_out_counts  i32 [B]          min(top_k, #reranked)  (search.rs:666)
 * Unused tail entries are id -1 / score -inf.
 */
int fpb_search_batch(const fpb_index* index, const void* d_queries, int B, int Q,
                     const fpb_params* params, void* d_workspace, size_t workspace_bytes,
                     int64_t* d_out_ids, float* d_out_scores, int32_t* d_out_counts,
                     void* stream);

/* Search restricted, per query, to a subset of documents (`subset=` of FastPlaid.search,
 * search.rs:494-517 + :544-547): probing is limited to the centroids that occur in the subset's
 * documents and the candidate set is intersected with the subset.
 *   d_subset_ids      i32 [total]  GLOBAL doc ids, query b owns [offsets[b], offsets[b+1])
 *   d_subset_offsets  i64 [B+1]
 *   max_subset_len    the largest per-query subset length (grid sizing)
 * params->flags must contain FPB_FLAG_SUBSET (it sizes the workspace). */
int fpb_search_batch_subset(const fpb_index* index, const void* d_queries, int B, int Q,
                            const fpb_params* params, const int32_t* d_subset_ids,
                            const int64_t* d_subset_offsets, int64_t max_subset_len, void* d_workspace,
                            size_t workspace_bytes, int64_t* d_out_ids, float* d_out_scores,
                            int32_t* d_out_counts, void* stream);

/* Same call with HOST buffers: H2D of the queries, the search, D2H of the results and a
 * stream synchronise all happen inside.  d_out_* are device scratch of the same shapes. */
int fpb_search_batch_host(const fpb_index* index, const void* h_queries, int B, int Q,
                          const fpb_params* params, void* d_workspace, size_t workspace_bytes,
                          void* d_queries_staging, int64_t* d_out_ids, float* d_out_scores,
                          int32_t* d_out_counts, int64_t* h_out_ids, float* h_out_scores,
                          int32_t* h_out_counts, void* stream);

/* ---- stage-level entry points (parity tests, roofline bench).  Each runs one stage of
 * search.rs on the workspace laid out by fpb_workspace_layout. ---- */
int fpb_stage_centroid_scores(const fpb_index*, const void* d_queries, int B, int Q,
                              const fpb_params*, void* d_workspace, size_t, void* stream); /* search.rs:491 */
int fpb_stage_subset(const fpb_index*, const int32_t* d_subset_ids, const int64_t* d_subset_offsets,
                     int64_t max_subset_len, int B, int Q, const fpb_params*, void* d_workspace, size_t,
                     void* stream); /* search.rs:496-503: run between centroid_scores and probe */
int fpb_stage_probe(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace,
                    size_t, void* stream); /* search.rs:520-532 */
int fpb_stage_candidates(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace,
                         size_t, void* stream); /* search.rs:535-541 */
int fpb_stage_approx(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace,
                     size_t, void* stream); /* search.rs:554-592 */
int fpb_stage_select(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace,
                     size_t, void* stream); /* search.rs:602-619 */
int fpb_stage_maxsim(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace,
                     size_t, void* stream); /* search.rs:626-656 (+ decompress :53-107) */
int fpb_stage_rank(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace,
                   size_t, int64_t* d_out_ids, float* d_out_scores, int32_t* d_out_counts,
                   void* stream); /* search.rs:659-666 */

int fpb_stage_keys(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace, size_t,
                   uint64_t* d_keys, void* stream); /* sharded two-step mode: emit [B, R] approx keys */
int fpb_stage_records(const fpb_index*, int B, int Q, const fpb_params*, void* d_workspace, size_t,
                      struct fpb_record* d_records, void* stream); /* sharded mode: emit [B, R] records */

/* ---- document-sharded search (new; the reference replicates the index and splits the
 * query list, fast_plaid.py:893-928).  Each rank runs fpb_search_shard on its shard and
 * emits R fixed-size records per query; the host all-gathers them (NCCL) and every rank
 * runs fpb_merge_shards, which re-applies the reference's GLOBAL pruning rule
 * (top n_full_scores/4 by approximate score, search.rs:605-619) before the final sort. */
struct fpb_record {
  float approx;   /* -inf for padding */
  float exact;
  int64_t doc_id; /* global id, -1 for padding */
};
typedef struct fpb_record fpb_record;

int fpb_search_shard(const fpb_index* index, const void* d_queries, int B, int Q,
                     const fpb_params* params, void* d_workspace, size_t workspace_bytes,
                     fpb_record* d_records /* [B, R] */, void* stream);
int fpb_merge_shards(const fpb_record* d_all_records /* [n_shards, B, R] */, int n_shards,
                     int B, int R, int top_k, int64_t* d_out_ids, float* d_out_scores,
                     int32_t* d_out_counts, void* stream);

/* Two-step variant (exact-scores only the documents that survive the GLOBAL pruning, so the
 * MaxSim work divides by the number of shards):
 *   1. fpb_shard_approx_keys : stages up to the local pruning; emits [B, R] 64-bit keys
 *                              (approx score, then smaller global id first; 0 = padding)
 *   2. all-gather of the keys; fpb_shard_apply_threshold finds, per query, the R-th best key of
 *      the whole index and shrinks this shard's re-rank list to the entries at or above it
 *   3. fpb_shard_exact_records : MaxSim on the shrunk lists, emits [B, R] fpb_record
 *   4. all-gather of the records; fpb_merge_shards ranks them. */
int fpb_shard_approx_keys(const fpb_index* index, const void* d_queries, int B, int Q,
                          const fpb_params* params, void* d_workspace, size_t workspace_bytes,
                          uint64_t* d_keys /* [B, R] */, void* stream);
/* Step 1 with a `subset` (search.rs:493-515, :544-551).  The reference restricts probing to the centroids
 * that the subset documents touch; with the documents sharded that set is the UNION over the shards:
 *   1a. fpb_shard_subset_begin : centroid scores + this shard's document bitmap and centroid bitmap;
 *                                copies the centroid bitmap ([B, layout.cbitmap_words] uint32) out
 *   1b. all-gather of the bitmaps; fpb_shard_subset_keys ORs them, probes, and continues like
 *       fpb_shard_approx_keys.  Subset ids are GLOBAL document ids (ids outside this shard are ignored).
 * params->flags must contain FPB_FLAG_SUBSET in both calls and in the later steps' layout. */
int fpb_shard_subset_begin(const fpb_index* index, const void* d_queries, int B, int Q,
                           const fpb_params* params, const int32_t* d_subset_ids,
                           const int64_t* d_subset_offsets, int64_t max_subset_len, void* d_workspace,
                           size_t workspace_bytes, uint32_t* d_cbitmap_out, void* stream);
int fpb_shard_subset_keys(const fpb_index* index, int B, int Q, const fpb_params* params, void* d_workspace,
                          size_t workspace_bytes, const uint32_t* d_all_cbitmaps /* [n_shards, B, words] */,
                          int n_shards, uint64_t* d_keys /* [B, R] */, void* stream);
int fpb_shard_apply_threshold(const fpb_index* index, const uint64_t* d_all_keys /* [n_shards, B, R] */,
                              int n_shards, int shard_rank, int B, int Q, const fpb_params* params,
                              void* d_workspace, size_t workspace_bytes, void* stream);
int fpb_shard_exact_records(const fpb_index* index, int B, int Q, const fpb_params* params,
                            void* d_workspace, size_t workspace_bytes, fpb_record* d_records, void* stream);

/* ---- the same exchange below the C ABI (SURVEY.md 8e: fpb_comm_init / fpb_search_batch_sharded) ----
 * An fpb_comm wraps one NCCL communicator (libnccl.so.2 is resolved at run time; without it these calls
 * return FPB_ERR_UNSUPPORTED and everything else keeps working).  Rank 0 makes the id with
 * fpb_comm_unique_id, the host distributes the FPB_COMM_ID_BYTES bytes by whatever means it has, every
 * rank calls fpb_comm_create (collective).
 *
 * fpb_search_batch_sharded searches the WHOLE batch on a grid of  n_query_groups x (nranks/n_query_groups)
 * document shards: rank r holds document shard r % n_shards (contiguous range, `doc_id_base` of its index)
 * and searches the queries of group r / n_shards (B split into n_query_groups contiguous slices).  Both
 * ncclAllGather calls (approximate-score keys, then the records of the globally surviving documents) are
 * issued on `stream` from inside the call; every rank returns the result of every query.
 *   d_queries  f16 [B, Q, dim]  the same batch on every rank
 *   d_ws       workspace of fpb_workspace_layout(index, ceil(B / n_query_groups), Q, params)
 *   d_scratch  fpb_sharded_scratch_bytes(ceil(B / n_query_groups), n_full_scores / 4, nranks) bytes */
#define FPB_COMM_ID_BYTES 128
typedef struct fpb_comm fpb_comm;
int fpb_comm_unique_id(void* out_id /* FPB_COMM_ID_BYTES */);
int fpb_comm_create(fpb_comm** out, int nranks, int rank, const void* unique_id, int device);
void fpb_comm_destroy(fpb_comm* comm);
int fpb_comm_nccl_version(void); /* 0 when NCCL is not loadable */
int64_t fpb_sharded_scratch_bytes(int b_local, int R, int nranks);
int fpb_search_batch_sharded(const fpb_index* index, fpb_comm* comm, int n_query_groups, const void* d_queries,
                             int B, int Q, const fpb_params* params, void* d_workspace, size_t workspace_bytes,
                             void* d_scratch, size_t scratch_bytes, int64_t* d_out_ids, float* d_out_scores,
                             int32_t* d_out_counts, void* stream);
/* The same with HOST buffers (H2D of the queries, D2H of the results, stream synchronise inside). */
int fpb_search_batch_sharded_host(const fpb_index* index, fpb_comm* comm, int n_query_groups, const void* h_queries,
                                  int B, int Q, const fpb_params* params, void* d_workspace, size_t workspace_bytes,
                                  void* d_scratch, size_t scratch_bytes, void* d_queries_staging, int64_t* d_out_ids,
                                  float* d_out_scores, int32_t* d_out_counts, int64_t* h_out_ids, float* h_out_scores,
                                  int32_t* h_out_counts, void* stream);

/* ---- by-products of the MaxSim kernel ("next" rows of SURVEY.md 8f-3) ---- */
/* reconstruct_embeddings (rust/utils/embeddings.rs:12-69): decompressed, normalised
 * fp16 rows of the given local docs, concatenated.  d_out: f16 [sum(len), dim]. */
int fpb_reconstruct(const fpb_index* index, const int32_t* d_doc_ids, int n, const int64_t* d_out_offsets,
                    void* d_out, void* stream);
/* token matrices of search_many_with_token_scores (search.rs:668-686):
 * d_out f16 [n, max_len, Q] row t = doc token, col = query token, for n (query, doc) pairs. */
int fpb_token_scores(const fpb_index* index, const void* d_queries, int Q, const int32_t* d_query_of,
                     const int32_t* d_doc_ids, int n, int64_t max_len, void* d_out, void* stream);

/* ---- index build: the encode step of create_index (rust/index/create.rs:404-428) ----
 * codes[t] = argmax_k fp16(<x_t, c_k>) (compress_into_codes, create.rs:148-170; ties -> smallest k),
 * residuals[t] = packed bucket indices of fp16(x_t - c[codes[t]]) against `cutoffs`
 * (bucketize right=false + LSB-first bits + big-endian packbits, create.rs:413-427, :176-184).
 *   d_tokens f16 [n_tokens, dim], d_centroids f16 [n_centroids, dim], d_cutoffs f32 [(1<<nbits)-1]
 *   d_codes i32 [n_tokens], d_residuals u8 [n_tokens, dim*nbits/8] */
/* Host utility: round-to-nearest-even fp32 -> fp16 cast of a query batch (the cast search_on_device does
 * on the host, fast_plaid.py:241), single-threaded with F16C.  The _portable variant is the same
 * conversion in plain C, exported so the tests can compare the two. */
int fpb_cast_f32_to_f16_host(const float* h_src, void* h_dst, size_t n);
int fpb_cast_f32_to_f16_host_portable(const float* h_src, void* h_dst, size_t n);

int fpb_encode(int device, int nbits, int dim, int64_t n_centroids, const void* d_centroids,
               const void* d_tokens, int64_t n_tokens, const float* d_cutoffs, int32_t* d_codes,
               uint8_t* d_residuals, void* stream);

/* ---- index build: Lloyd iterations of the centroid k-means (python/fast_plaid/search/kmeans.py:60-223) ----
 * fpb_kmeans_assign : assign[i] = argmax_k (<x_i, c_k> + bias[k]) in fp32 on the tensor cores; with
 *                     bias[k] = -|c_k|^2 / 2 that is the nearest centroid by squared distance (kmeans.py:153-160);
 *                     ties -> smallest k.   d_points f16 [n, 128], d_centroids f16 [K, 128], d_bias f32 [K]
 * fpb_kmeans_update : centroid k <- mean of its points, as a deterministic segmented sum: d_order i64 [n] = point
 *                     indices sorted by assignment, d_seg_offsets i64 [K+1]; empty segments are left untouched
 *                     (the caller re-seeds them, kmeans.py:196-205); d_shift f32 [K] (optional) receives
 *                     |new - old| per centroid for the convergence test */
int fpb_kmeans_assign(int device, int dim, int64_t n_centroids, const void* d_centroids, const float* d_bias,
                      const void* d_points, int64_t n_points, int32_t* d_assign, void* stream);
int fpb_kmeans_update(int device, int dim, int64_t n_centroids, const void* d_points, const int64_t* d_order,
                      const int64_t* d_seg_offsets, void* d_centroids, float* d_shift, void* stream);

/* ---- index update: outlier search of the centroid expansion (python/fast_plaid/search/update.py:121-150) ----
 * fpb_nearest_centroid : the fpb_kmeans_assign argmax, plus d_best f32 [n] = the maximum itself,
 *                        max_k (<x_i, c_k> + bias[k]) accumulated in fp32.  With bias[k] = -|c_k|^2 / 2 the caller
 *                        gets min_k |x_i - c_k|^2 = |x_i|^2 - 2 d_best[i], which update_centroids compares with the
 *                        squared cluster threshold.  dim 128 only (FPB_ERR_UNSUPPORTED otherwise). */
int fpb_nearest_centroid(int device, int dim, int64_t n_centroids, const void* d_centroids, const float* d_bias,
                         const void* d_points, int64_t n_points, int32_t* d_assign, float* d_best, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FASTPLAID_B200_H_ */
