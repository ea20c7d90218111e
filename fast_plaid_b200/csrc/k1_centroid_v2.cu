// K1 v2 : centroid scores S = fp16(C . q^T) on tcgen05 (search.rs:491), dim = 128, Qp <= 128.
//
// GEMM view: D[token][centroid] = sum_k Qtok[token][k] * C[centroid][k] with M = 128 query tokens
// (A operand, resident for the CTA's lifetime), N = 128 centroids per tile (B operand, streamed
// through a 3-stage shared-memory ring in the K-major SWIZZLE_128B layout), K = 128, fp32
// accumulators in TMEM (2 x 128 columns, double buffered).  One accumulator row = one query
// token, so the per-128-centroid-tile column maximum K1b needs is a per-thread max over the
// columns, and the fp16 tile is transposed through shared memory into [centroid][q] blocks
// that are contiguous in S[b][k][q] and leave with one bulk-async copy each
// (cp.async.bulk.global.shared::cta, SASS UBLKCP) -- the 1 GB write of S never touches the LSU.
//
// The centroid tiles arrive by TMA (cp.async.bulk.tensor.2d with a SWIZZLE_128B tensor map, SASS
// UTMALDG): one elected thread arms the stage's mbarrier with the byte count and issues two
// 64-column boxes; rows past K are zero-filled by the TMA unit.
//
// grid = (token tiles, centroid splits); warps 0-7 epilogue (TMEM lane quarter w % 4, column half
// w / 4 of the 128-centroid tile), warp 8 issues the MMAs, warp 9 is the TMA producer.  (With four
// epilogue warps the epilogue -- 128 conversions + stores per thread and tile -- was the critical
// path: 0.33 ms.)
#include <string.h>

#include "kernels.h"
#include "tc05.cuh"

namespace {

constexpr int G1_THREADS = 320;
constexpr int G1_PRODUCER_WARP = 9;
constexpr int G1_STAGING = 128 * 128 * 2;  // 32 KB fp16 output tile

struct G1Smem {
  static constexpr int a_off = 0;
  static constexpr int b_off = CT_TILE;
  static constexpr int st_off = b_off + CT_STAGES * CT_TILE;
  static constexpr int bar_off = st_off + 2 * G1_STAGING;
  static constexpr int pmax_off = bar_off + 256;               // fp32 [128] partial tile maxima of the upper half
  static constexpr int bytes = pmax_off + 512 + 1024;
};

__global__ void __launch_bounds__(G1_THREADS, 1)
k1_centroid_v2_kernel(const __grid_constant__ CUtensorMap tmap_c, int K, const __half* __restrict__ Qpad, int B, int Qp,
                      __half* __restrict__ S, __half* __restrict__ tmax, int n_ctiles, int tiles_per_split) {
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = SMEM_ALIGN1024(smem_dyn);
  unsigned char* smA = base + G1Smem::a_off;
  unsigned char* smB = base + G1Smem::b_off;
  unsigned char* smS = base + G1Smem::st_off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + G1Smem::bar_off);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  float* pmax = reinterpret_cast<float*>(base + G1Smem::pmax_off);
  const CtileBars ring(bars);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tt = blockIdx.x;                      // token tile
  const int ct_begin = blockIdx.y * tiles_per_split;
  const int ct_end = min(n_ctiles, ct_begin + tiles_per_split);
  const int n_tokens = B * Qp;

  // ---- setup: A tile (128 query tokens), barriers, TMEM ----
  for (int i = tid; i < 128 * 16; i += G1_THREADS) {
    const int r = i >> 4, c = i & 15;
    const int tok = tt * 128 + r;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (tok < n_tokens) v = *reinterpret_cast<const uint4*>(Qpad + int64_t(tok) * 128 + c * 8);
    *reinterpret_cast<uint4*>(smA + sw128_off(r, c)) = v;
  }
  fence_proxy_async();
  if (tid == 0) ring.init(8);
  if (warp == 8) tmem_alloc<CT_TMEM_COLS>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int n_my = ct_end - ct_begin;

  if (warp == G1_PRODUCER_WARP) {
    // =========================== TMA producer: centroid tiles -> swizzled smem ===========================
    if (lane == 0) ctile_produce(&tmap_c, ring, smB, ct_begin, n_my, 0);
    __syncwarp();
  } else if (warp == 8) {
    // =========================== MMA issuer ===========================
    if (lane == 0) ctile_mma(ring, smA, smB, tmem_base, n_my, 0);
    __syncwarp();
  } else if (warp < 8) {
    // =========================== epilogue ===========================
    const int quarter = warp & 3, half = warp >> 2;  // TMEM lanes 32*quarter.., columns 64*half..
    const int trow = quarter * 32 + lane;        // token row inside the tile == TMEM lane
    const int tok = tt * 128 + trow;
    const bool tok_valid = tok < n_tokens;
    const int b = tok / Qp, q = tok % Qp;
    const int blk = trow / Qp;                   // query block inside the tile
    const int n_blk = 128 / Qp;
    const uint32_t blk_bytes = uint32_t(128 * Qp * 2);
    for (int i = 0; i < n_my; ++i) {
      const int acc = i & 1, sb = i & 1;
      const int ct = ct_begin + i;
      const int k0 = ct * 128;
      const int rows_valid = min(128, K - k0);
      unsigned char* stg = smS + sb * G1_STAGING;
      // the bulk stores issued from this staging buffer two tiles ago must have finished reading it
      if (tid < n_blk) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
      asm volatile("bar.sync 1, 256;" ::: "memory");
      mbar_wait(ring.tfull + 8 * acc, (i >> 1) & 1);
      tc_fence_after();
      float mx = -INFINITY;
      unsigned char* my = stg + blk * blk_bytes + q * 2;
#pragma unroll 1
      for (int c0 = 64 * half; c0 < 64 * half + 64; c0 += 32) {
        float v[32];
        tmem_ld32(tmem_base + (uint32_t(quarter * 32) << 16) + acc * 128 + c0, v);
#pragma unroll
        for (int x = 0; x < 32; ++x) {
          if (c0 + x < rows_valid) mx = fmaxf(mx, v[x]);
          *reinterpret_cast<__half*>(my + (c0 + x) * (Qp * 2)) = __float2half_rn(v[x]);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(ring.tempty + 8 * acc);
      if (half == 1) pmax[trow] = mx;
      fence_proxy_async();
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (half == 0 && tok_valid)
        tmax[(int64_t(b) * Qp + q) * n_ctiles + ct] = __float2half_rn(fmaxf(mx, pmax[trow]));
      if (tid < n_blk) {
        const int bb = (tt * 128) / Qp + tid;    // query of block `tid`
        if (bb < B) {
          const __half* dst = S + (int64_t(bb) * K + k0) * Qp;
          const uint32_t bytes = uint32_t(rows_valid * Qp * 2);
          asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst),
                       "r"(smem_u32(stg + tid * blk_bytes)), "r"(bytes)
                       : "memory");
        }
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
      }
    }
    if (tid < n_blk) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc<CT_TMEM_COLS>(tmem_base);
  }
}

}  // namespace

int launch_centroid_scores_v2(const fpb_index* ix, const Ws& ws, cudaStream_t st, bool* handled) {
  *handled = false;
  const fpb_layout& L = *ws.L;
  if (ix->dim != 128 || L.Qp > 128 || !ix->has_tmap) return FPB_OK;
  *handled = true;
  // opt in on every launch: the attribute is per device and the call costs about a microsecond
  FPB_CUDA_CHECK(cudaFuncSetAttribute(k1_centroid_v2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, G1Smem::bytes));
  const int n_ttiles = (L.B * L.Qp + 127) / 128;
  const int n_ctiles = L.n_tiles;
  int splits = ix->sm_count / n_ttiles;
  if (splits < 1) splits = 1;
  if (splits > n_ctiles) splits = n_ctiles;
  const int per = (n_ctiles + splits - 1) / splits;
  splits = (n_ctiles + per - 1) / per;
  dim3 grid(n_ttiles, splits);
  CUtensorMap tm;
  memcpy(&tm, ix->tmap_centroids, sizeof(tm));
  k1_centroid_v2_kernel<<<grid, G1_THREADS, G1Smem::bytes, st>>>(tm, int(ix->K), ws.queries(), L.B, L.Qp,
                                                                ws.S(), ws.tmax(), n_ctiles, per);
  FPB_LAUNCH_CHECK("k1_centroid_v2");
  return FPB_OK;
}
