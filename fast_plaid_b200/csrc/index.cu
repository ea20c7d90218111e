// Index handle, error reporting and workspace layout of the C ABI.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <cuda.h>

#include "kernels.h"

// The driver-API entry point is resolved at run time (no link against libcuda).
typedef CUresult (*fpb_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*,
                                        CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                        CUtensorMapFloatOOBfill);

const char* encode_centroid_tmap(CUtensorMap* tm, const void* d_centroids, int64_t K) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    cudaGetLastError();
    return "cuTensorMapEncodeTiled is not available from this driver";
  }
  const cuuint64_t gdim[2] = {128, cuuint64_t(K)};
  const cuuint64_t gstride[1] = {128 * 2};
  const cuuint32_t box[2] = {64, 128};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = reinterpret_cast<fpb_encode_tiled_fn>(fn)(
      tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(d_centroids), gdim, gstride, box, estr,
      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? nullptr : "cuTensorMapEncodeTiled failed";
}

static thread_local char g_err[512] = "";

void fpb_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* fpb_last_error(void) { return g_err; }
extern "C" int fpb_abi_version(void) { return 6; }  // 6: d_token_norms of fpb_index_create; 5: two-pass approximate stage (layout fields, FPB_FLAG_APPROX_*), fpb_comm_* + fpb_search_batch_sharded

static int bitrev(int x, int nbits) {
  int r = 0;
  for (int k = 0; k < nbits; ++k)
    if (x & (1 << k)) r |= 1 << (nbits - 1 - k);
  return r;
}

extern "C" int fpb_index_create(fpb_index** out, int device, int nbits, int dim, int64_t n_centroids,
                                const void* d_centroids, const void* d_bucket_weights,
                                int64_t n_docs, const int64_t* d_doc_offsets,
                                const int32_t* d_doc_codes, const uint8_t* d_doc_residuals, void* d_token_norms,
                                const int64_t* d_ivf_offsets, const int32_t* d_ivf_pids,
                                int64_t n_ivf, int64_t max_doc_len, int64_t doc_id_base) {
  if (!out) {
    fpb_set_error("fpb_index_create: out is NULL");
    return FPB_ERR_INVALID;
  }
  *out = nullptr;
  if (nbits != 2 && nbits != 4) {
    fpb_set_error("unsupported nbits=%d (2 and 4 are supported)", nbits);
    return FPB_ERR_UNSUPPORTED;
  }
  const int pd = dim * nbits / 8;
  if ((dim != 64 && dim != 128) || (pd != 16 && pd != 32 && pd != 64)) {
    fpb_set_error("unsupported embedding dim=%d with nbits=%d: this build supports dim 64 and 128", dim, nbits);
    return FPB_ERR_UNSUPPORTED;
  }
  if (n_centroids <= 0 || n_docs < 0 || !d_centroids || !d_bucket_weights || !d_doc_offsets) {
    fpb_set_error("fpb_index_create: bad sizes or NULL codec/offset pointers");
    return FPB_ERR_INVALID;
  }
  if (n_docs >= (int64_t(1) << 31) || n_centroids >= (int64_t(1) << 31)) {
    fpb_set_error("fpb_index_create: n_docs and n_centroids must fit in int32 per shard");
    return FPB_ERR_UNSUPPORTED;
  }
  FPB_CUDA_CHECK(cudaSetDevice(device));
  fpb_index* ix = new fpb_index();
  memset(ix, 0, sizeof(*ix));
  ix->device = device;
  ix->nbits = nbits;
  ix->dim = dim;
  ix->pd = pd;
  ix->K = n_centroids;
  ix->N = n_docs;
  ix->n_ivf = n_ivf;
  ix->max_doc_len = max_doc_len;
  ix->doc_id_base = doc_id_base;
  ix->centroids = static_cast<const __half*>(d_centroids);
  ix->doc_offsets = d_doc_offsets;
  ix->doc_codes = d_doc_codes;
  ix->doc_residuals = d_doc_residuals;
  ix->token_norms = static_cast<const __half*>(d_token_norms);
  ix->ivf_offsets = d_ivf_offsets;
  ix->ivf_pids = d_ivf_pids;
  cudaDeviceProp prop;
  cudaError_t e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) {
    delete ix;
    fpb_set_error("cudaGetDeviceProperties failed: %s", cudaGetErrorString(e));
    return FPB_ERR_CUDA;
  }
  ix->sm_count = prop.multiProcessorCount;
  uint16_t w[16];
  e = cudaMemcpy(w, d_bucket_weights, sizeof(uint16_t) * (1 << nbits), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    delete ix;
    fpb_set_error("copy of bucket_weights failed: %s", cudaGetErrorString(e));
    return FPB_ERR_CUDA;
  }
  for (int i = 0; i < 16; ++i) ix->w_perm_bits[i] = 0;
  for (int i = 0; i < (1 << nbits); ++i) ix->w_perm_bits[i] = w[bitrev(i, nbits)];
  int64_t n_tokens = 0;
  if (n_docs > 0) {
    e = cudaMemcpy(&n_tokens, d_doc_offsets + n_docs, sizeof(int64_t), cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      delete ix;
      fpb_set_error("copy of doc_offsets[N] failed: %s", cudaGetErrorString(e));
      return FPB_ERR_CUDA;
    }
  }
  ix->E = n_tokens;
  if (n_tokens > 0 && !d_token_norms) {
    delete ix;
    fpb_set_error("fpb_index_create: d_token_norms (f16 [n_tokens], filled here) is NULL");
    return FPB_ERR_INVALID;
  }
  if (n_tokens > 0) {  // derive the per-token norms once (default stream, synchronous: creation is not a hot path)
    const int rc = launch_token_norms(ix, static_cast<__half*>(d_token_norms), nullptr);
    e = rc == FPB_OK ? cudaDeviceSynchronize() : cudaSuccess;
    if (rc != FPB_OK || e != cudaSuccess) {
      delete ix;
      if (rc == FPB_OK) fpb_set_error("token norm kernel failed: %s", cudaGetErrorString(e));
      return rc != FPB_OK ? rc : FPB_ERR_CUDA;
    }
  }
  // without a tensor map K1 runs the mma.sync kernel
  static_assert(sizeof(CUtensorMap) == sizeof(ix->tmap_centroids), "CUtensorMap is 128 bytes");
  ix->has_tmap =
      dim == 128 && !encode_centroid_tmap(reinterpret_cast<CUtensorMap*>(ix->tmap_centroids), d_centroids, n_centroids);
  *out = ix;
  return FPB_OK;
}

extern "C" void fpb_index_destroy(fpb_index* index) { delete index; }

extern "C" int fpb_workspace_layout(const fpb_index* ix, int B, int Q, const fpb_params* p,
                                    fpb_layout* L) {
  if (!ix || !p || !L) {
    fpb_set_error("fpb_workspace_layout: NULL argument");
    return FPB_ERR_INVALID;
  }
  if (B <= 0 || Q <= 0) {
    fpb_set_error("fpb_workspace_layout: B=%d Q=%d must be positive", B, Q);
    return FPB_ERR_INVALID;
  }
  if (Q > 256) {
    fpb_set_error("queries with more than 256 tokens are not supported (Q=%d)", Q);
    return FPB_ERR_UNSUPPORTED;
  }
  if (p->n_ivf_probe < 1 || p->n_ivf_probe > 32) {
    fpb_set_error("n_ivf_probe=%d outside the supported range [1,32]", p->n_ivf_probe);
    return FPB_ERR_UNSUPPORTED;
  }
  if (p->n_full_scores < 1 || p->top_k < 1) {
    fpb_set_error("n_full_scores and top_k must be >= 1");
    return FPB_ERR_INVALID;
  }
  int R = p->n_full_scores / 4;
  if (R < 1) R = 1;
  if (R > 4096) {
    fpb_set_error("n_full_scores=%d: more than 4096 re-ranked documents per query is not supported",
                  p->n_full_scores);
    return FPB_ERR_UNSUPPORTED;
  }
  memset(L, 0, sizeof(*L));
  int Qp = fpb_next_pow2(Q < 16 ? 16 : Q);
  L->B = B;
  L->Q = Q;
  L->Qp = Qp;
  L->n_tiles = int((ix->K + 127) / 128);
  L->R = R;
  L->n_probe = p->n_ivf_probe;
  L->cand_cap = int(ix->N > 0 ? ix->N : 1);
  L->bitmap_words = int((ix->N + 31) / 32) + 1;
  int64_t off = 0;
  auto take = [&](int64_t bytes) {
    int64_t o = off;
    off += fpb_align256(bytes);
    return o;
  };
  L->off_queries = take(int64_t(B) * Qp * ix->dim * 2);
  L->off_S = take(int64_t(B) * ix->K * Qp * 2);
  L->off_tmax = take(int64_t(B) * Qp * L->n_tiles * 2);
  L->off_cells = take(int64_t(B) * Q * L->n_probe * 4);
  L->off_bitmap = take(int64_t(B) * L->bitmap_words * 4);
  L->off_n_cand = take(int64_t(B) * 4);
  L->off_cand = take(int64_t(B) * L->cand_cap * 4);
  L->off_approx = take(int64_t(B) * L->cand_cap * 4);
  L->off_work = take(int64_t(B + 8) * 4);
  L->off_n_rerank = take(int64_t(B) * 4);
  L->off_rerank = take(int64_t(B) * R * 4);
  L->off_rerank_approx = take(int64_t(B) * R * 4);
  L->off_exact = take(int64_t(B) * R * 4);
  const bool sub = (p->flags & FPB_FLAG_SUBSET) != 0;
  L->cbitmap_words = int((ix->K + 31) / 32) + 1;
  L->off_cbitmap = take(sub ? int64_t(B) * L->cbitmap_words * 4 : 0);
  L->off_clist = take(sub ? int64_t(B) * ix->K * 4 : 0);
  L->off_n_clist = take(sub ? int64_t(B) * 4 : 0);
  L->off_sbitmap = take(sub ? int64_t(B) * L->bitmap_words * 4 : 0);
  // two-pass approximate stage (k3_approx.cu); hb_words is a multiple of 4 so a query's bitmap is uint4-copyable
  const bool direct = (p->flags & FPB_FLAG_APPROX_DIRECT) != 0;
  L->hb_words = int(((ix->K + 31) / 32 + 3) / 4 * 4);
  L->off_tau = take(direct ? 0 : int64_t(B) * Qp * 2);
  L->off_hibits = take(direct ? 0 : int64_t(B) * L->hb_words * 4);
  L->off_lb = take(direct ? 0 : int64_t(B) * L->cand_cap * 4);
  L->off_refine = take(direct ? 0 : int64_t(B) * L->cand_cap * 4);
  L->off_n_refine = take(int64_t(B) * 4);
  L->off_thresh = take(int64_t(B) * 4);
  L->off_work2 = take(int64_t(B + 8) * 4);
  L->off_stats = take(8 * 8);
  L->flags = p->flags;
  L->total_bytes = off;
  return FPB_OK;
}
