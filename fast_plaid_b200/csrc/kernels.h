// Internal launchers (one per pipeline stage).  All are asynchronous on `stream`.
#pragma once
#include <cuda.h>

#include "common.cuh"

struct Ws {
  const fpb_layout* L;
  char* base;
  __half* queries() const { return reinterpret_cast<__half*>(base + L->off_queries); }
  __half* S() const { return reinterpret_cast<__half*>(base + L->off_S); }
  __half* tmax() const { return reinterpret_cast<__half*>(base + L->off_tmax); }
  int32_t* cells() const { return reinterpret_cast<int32_t*>(base + L->off_cells); }
  uint32_t* bitmap() const { return reinterpret_cast<uint32_t*>(base + L->off_bitmap); }
  int32_t* n_cand() const { return reinterpret_cast<int32_t*>(base + L->off_n_cand); }
  int32_t* cand() const { return reinterpret_cast<int32_t*>(base + L->off_cand); }
  float* approx() const { return reinterpret_cast<float*>(base + L->off_approx); }
  int32_t* work() const { return reinterpret_cast<int32_t*>(base + L->off_work); }
  int32_t* n_rerank() const { return reinterpret_cast<int32_t*>(base + L->off_n_rerank); }
  int32_t* rerank() const { return reinterpret_cast<int32_t*>(base + L->off_rerank); }
  float* rerank_approx() const { return reinterpret_cast<float*>(base + L->off_rerank_approx); }
  float* exact() const { return reinterpret_cast<float*>(base + L->off_exact); }
  uint32_t* cbitmap() const { return reinterpret_cast<uint32_t*>(base + L->off_cbitmap); }
  int32_t* clist() const { return reinterpret_cast<int32_t*>(base + L->off_clist); }
  int32_t* n_clist() const { return reinterpret_cast<int32_t*>(base + L->off_n_clist); }
  uint32_t* sbitmap() const { return reinterpret_cast<uint32_t*>(base + L->off_sbitmap); }
  __half* tau() const { return reinterpret_cast<__half*>(base + L->off_tau); }
  uint32_t* hibits() const { return reinterpret_cast<uint32_t*>(base + L->off_hibits); }
  float* lb() const { return reinterpret_cast<float*>(base + L->off_lb); }
  int32_t* refine() const { return reinterpret_cast<int32_t*>(base + L->off_refine); }
  int32_t* n_refine() const { return reinterpret_cast<int32_t*>(base + L->off_n_refine); }
  float* thresh() const { return reinterpret_cast<float*>(base + L->off_thresh); }
  int32_t* work2() const { return reinterpret_cast<int32_t*>(base + L->off_work2); }
  unsigned long long* stats() const { return reinterpret_cast<unsigned long long*>(base + L->off_stats); }
};

// TMA descriptor of an fp16 [K, 128] centroid table: 2-D, box 64 x 128 (one SWIZZLE_128B K block of a 128-centroid
// tile), SWIZZLE_128B, rows past K zero-filled.  Returns nullptr on success, else why no map could be made.
const char* encode_centroid_tmap(CUtensorMap* tm, const void* d_centroids, int64_t K);

int launch_pad_queries(const fpb_index* ix, const Ws& ws, const __half* d_queries, cudaStream_t st);
int launch_centroid_scores(const fpb_index* ix, const Ws& ws, cudaStream_t st);   // K1 (dispatch)
int launch_centroid_scores_v2(const fpb_index* ix, const Ws& ws, cudaStream_t st, bool* handled);  // K1 on tcgen05
int launch_probe(const fpb_index* ix, const Ws& ws, bool subset, cudaStream_t st);       // K1b
int launch_candidates(const fpb_index* ix, const Ws& ws, bool subset, cudaStream_t st);  // K2
int launch_subset_mark(const fpb_index* ix, const Ws& ws, const int32_t* d_ids, const int64_t* d_offsets,
                       int64_t max_len, cudaStream_t st);
int launch_subset_compact(const fpb_index* ix, const Ws& ws, cudaStream_t st);
int launch_subset_merge(const fpb_index* ix, const Ws& ws, const uint32_t* d_all, int n_shards, cudaStream_t st);
int launch_subset(const fpb_index* ix, const Ws& ws, const int32_t* d_ids, const int64_t* d_offsets,
                  int64_t max_len, cudaStream_t st);                                      // subset structures
int launch_compact(const uint32_t* bitmap, const uint32_t* mask, int words, int32_t* out, int cap, int32_t* n_out,
                   int B, cudaStream_t st);
int launch_approx(const fpb_index* ix, const Ws& ws, int flags, cudaStream_t st); // K3 (flags: FPB_FLAG_APPROX_*)
int launch_select(const fpb_index* ix, const Ws& ws, cudaStream_t st);            // K3b
int launch_maxsim(const fpb_index* ix, const Ws& ws, cudaStream_t st);            // K5 (dispatch)
int launch_token_norms(const fpb_index* ix, __half* d_out, cudaStream_t st);      // per-token fp16 norms (index load)
int launch_maxsim_v4(const fpb_index* ix, const Ws& ws, cudaStream_t st, bool* handled);  // K5 v4 (register operands)
int launch_maxsim_v5(const fpb_index* ix, const Ws& ws, cudaStream_t st, bool* handled);  // K5 v5 (tcgen05, 20 decode warps)
int launch_rank(const fpb_index* ix, const Ws& ws, int top_k, int64_t* d_out_ids, float* d_out_scores,
                int32_t* d_out_counts, cudaStream_t st);                          // K6
int launch_emit_keys(const fpb_index* ix, const Ws& ws, uint64_t* d_keys, cudaStream_t st);
int launch_apply_threshold(const Ws& ws, const uint64_t* d_all_keys, int n_shards, int rank, cudaStream_t st,
                           int b_stride = 0);
int launch_merge(const fpb_record* d_all_records, int n_shards, int b_stride, int n_queries, int R, int top_k,
                 int64_t* d_out_ids, float* d_out_scores, int32_t* d_out_counts, cudaStream_t stream);
int launch_emit_records(const fpb_index* ix, const Ws& ws, fpb_record* d_records, cudaStream_t st);
