// Index-build encode kernels (SURVEY.md 8(f-1); replaces the per-batch closure of create_index,
// rust/index/create.rs:404-428):
//   * assign : code[t] = argmax_k fp16(<x_t, c_k>)  (compress_into_codes, create.rs:148-170) on
//              tcgen05 -- the centroid-tile ring K1 v2 uses (tc05.cuh: TMA-fed centroid tiles, TMEM
//              accumulators) with an argmax epilogue instead of the S store; ties -> smallest centroid
//              id, which is what ATen's CPU argmax returns
//   * pack   : residual = fp16(x - c[code]); bucket = #cutoffs < residual (bucketize right=false,
//              create.rs:413-414); each index written LSB-first into nbits bits, bits packed
//              big-endian per byte (create.rs:416-427, packbits :176-184)
#include "kernels.h"
#include "tc05.cuh"

namespace {

constexpr int EN_THREADS = 288;

struct EnSmem {
  static constexpr int a_off = 0;
  static constexpr int b_off = CT_TILE;
  static constexpr int bar_off = b_off + CT_STAGES * CT_TILE;
  static constexpr int bytes = bar_off + 256 + 1024;
};

// KMEANS = false: code = argmax_k fp16(<x, c_k>)                      (index-build encode)
// KMEANS = true : code = argmax_k (<x, c_k> + bias[k]) in fp32, bias[k] = -|c_k|^2 / 2, i.e. the nearest centroid
//                 by squared distance (the assignment step of Lloyd's algorithm, kmeans.py:153-160); `best`
//                 (optional) receives that maximum, from which the caller gets min_k |x - c_k|^2 = |x|^2 - 2 best
template <bool KMEANS>
__global__ void __launch_bounds__(EN_THREADS, 1)
encode_assign_kernel(const __grid_constant__ CUtensorMap tmap_c, int K, const __half* __restrict__ X, int64_t n,
                     int32_t* __restrict__ codes, int n_ctiles, const float* __restrict__ bias,
                     float* __restrict__ best_out) {
  __shared__ float s_bias[4][2][128];  // per epilogue warp and accumulator: the tile's biases
  extern __shared__ unsigned char smem_dyn[];
  unsigned char* base = SMEM_ALIGN1024(smem_dyn);
  unsigned char* smA = base + EnSmem::a_off;
  unsigned char* smB = base + EnSmem::b_off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + EnSmem::bar_off);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const CtileBars ring(bars);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) ring.init(4);
  if (warp == 8) tmem_alloc<CT_TMEM_COLS>(smem_u32(tmem_slot));
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int64_t n_ttiles = (n + 127) / 128;
  uint32_t it = 0;  // centroid tiles streamed so far by this CTA (pipeline state persists across token tiles)
  for (int64_t tt = blockIdx.x; tt < n_ttiles; tt += gridDim.x) {
    __syncthreads();  // every role is done with the previous token tile (A tile can be replaced)
    for (int i = tid; i < 128 * 16; i += EN_THREADS) {
      const int r = i >> 4, c = i & 15;
      const int64_t tok = tt * 128 + r;
      uint4 v = make_uint4(0u, 0u, 0u, 0u);
      if (tok < n) v = __ldg(reinterpret_cast<const uint4*>(X + tok * 128) + c);
      *reinterpret_cast<uint4*>(smA + sw128_off(r, c)) = v;
    }
    fence_proxy_async();
    __syncthreads();

    if (warp == 4) {
      if (lane == 0) ctile_produce(&tmap_c, ring, smB, 0, n_ctiles, it);
      __syncwarp();
    } else if (warp == 8) {
      if (lane == 0) ctile_mma(ring, smA, smB, tmem_base, n_ctiles, it);
      __syncwarp();
    } else if (warp < 4) {
      const int64_t tok = tt * 128 + warp * 32 + lane;
      float best = -INFINITY;
      int best_k = 0;
      for (int i = 0; i < n_ctiles; ++i) {
        const uint32_t g = it + i;
        const int acc = g & 1;
        const int k0 = i * 128;
        const int rows_valid = min(128, K - k0);
        if (KMEANS) {
#pragma unroll
          for (int x = 0; x < 4; ++x) {
            const int kk = k0 + x * 32 + lane;
            s_bias[warp][acc][x * 32 + lane] = kk < K ? __ldg(bias + kk) : 0.f;
          }
          __syncwarp();
        }
        mbar_wait(ring.tfull + 8 * acc, (g >> 1) & 1);
        tc_fence_after();
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          float r[32];
          tmem_ld32(tmem_base + (uint32_t(warp * 32) << 16) + acc * 128 + c0, r);
#pragma unroll
          for (int x = 0; x < 32; ++x) {
            // encode: the reference compares fp16 scores (half matmul output); first maximum wins
            const float v = KMEANS ? r[x] + s_bias[warp][acc][c0 + x] : __half2float(__float2half_rn(r[x]));
            if (c0 + x < rows_valid && v > best) {
              best = v;
              best_k = k0 + c0 + x;
            }
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ring.tempty + 8 * acc);
      }
      if (tok < n) {
        codes[tok] = best_k;
        if (KMEANS && best_out) best_out[tok] = best;
      }
    }
    it += uint32_t(n_ctiles);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    tmem_dealloc<CT_TMEM_COLS>(tmem_base);
  }
}

// residual = fp16(x - c[code]) -> bucket index -> packed bits.  One thread per output byte.
template <int NBITS>
__global__ void encode_pack_kernel(const __half* __restrict__ X, const __half* __restrict__ C,
                                   const int32_t* __restrict__ codes, const float* __restrict__ cutoffs, int64_t n,
                                   int dim, uint8_t* __restrict__ out) {
  constexpr int PER = 8 / NBITS;       // elements per byte
  constexpr int NCUT = (1 << NBITS) - 1;
  __shared__ float cut[NCUT];
  if (threadIdx.x < NCUT) cut[threadIdx.x] = cutoffs[threadIdx.x];
  __syncthreads();
  const int pd = dim / PER;
  const int64_t total = n * pd;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < total; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t t = i / pd;
    const int j = int(i % pd);
    const __half* x = X + t * dim + j * PER;
    const __half* c = C + int64_t(codes[t]) * dim + j * PER;
    uint32_t byte = 0;
#pragma unroll
    for (int e = 0; e < PER; ++e) {
      const float r = __half2float(__hsub(x[e], c[e]));  // one fp16 subtraction, like the reference
      int b = 0;
#pragma unroll
      for (int k = 0; k < NCUT; ++k) b += (cut[k] < r) ? 1 : 0;  // bucketize(right=false)
      uint32_t rev = 0;  // LSB-first bit order inside the element's field
#pragma unroll
      for (int k = 0; k < NBITS; ++k) rev |= ((uint32_t(b) >> k) & 1u) << (NBITS - 1 - k);
      byte |= rev << (8 - NBITS * (e + 1));
    }
    out[i] = uint8_t(byte);
  }
}

}  // namespace

// tensor map of the centroid table + launch of the assign kernel (shared by fpb_encode, fpb_kmeans_assign and
// fpb_nearest_centroid; d_best needs d_bias)
static int launch_assign(int device, int64_t n_centroids, const void* d_centroids, const void* d_tokens,
                         int64_t n_tokens, int32_t* d_codes, const float* d_bias, float* d_best, cudaStream_t st,
                         const char* who) {
  CUtensorMap tm;
  if (const char* why = encode_centroid_tmap(&tm, d_centroids, n_centroids)) {
    fpb_set_error("%s: %s", who, why);
    return FPB_ERR_CUDA;
  }
  cudaDeviceProp prop;
  FPB_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
  const int64_t n_ttiles = (n_tokens + 127) / 128;
  const int blocks = int(n_ttiles < prop.multiProcessorCount ? n_ttiles : prop.multiProcessorCount);
  const int n_ctiles = int((n_centroids + 127) / 128);
  // opt in on every launch: the attribute is per device and the call costs about a microsecond
  if (d_bias) {
    FPB_CUDA_CHECK(cudaFuncSetAttribute(encode_assign_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, EnSmem::bytes));
    encode_assign_kernel<true><<<blocks, EN_THREADS, EnSmem::bytes, st>>>(tm, int(n_centroids),
                                                                         static_cast<const __half*>(d_tokens), n_tokens,
                                                                         d_codes, n_ctiles, d_bias, d_best);
  } else {
    FPB_CUDA_CHECK(cudaFuncSetAttribute(encode_assign_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, EnSmem::bytes));
    encode_assign_kernel<false><<<blocks, EN_THREADS, EnSmem::bytes, st>>>(tm, int(n_centroids),
                                                                          static_cast<const __half*>(d_tokens), n_tokens,
                                                                          d_codes, n_ctiles, nullptr, nullptr);
  }
  FPB_LAUNCH_CHECK("encode_assign");
  return FPB_OK;
}

// Centroid update of Lloyd's algorithm as a deterministic segmented mean: `order` lists the point indices sorted by
// assigned centroid, `seg_offsets[k] .. seg_offsets[k+1]` is centroid k's segment.  One warp per centroid, each lane
// sums four dimensions in fp32 in segment order; empty segments leave the output row untouched and count 0.
__global__ void __launch_bounds__(256)
segment_mean_kernel(const __half* __restrict__ X, const int64_t* __restrict__ order,
                    const int64_t* __restrict__ seg_offsets, int64_t K, __half* __restrict__ out,
                    float* __restrict__ shift) {
  const int lane = threadIdx.x & 31;
  const int64_t k = int64_t(blockIdx.x) * 8 + (threadIdx.x >> 5);
  if (k >= K) return;
  const int64_t s0 = seg_offsets[k], s1 = seg_offsets[k + 1];
  if (s1 <= s0) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  for (int64_t i = s0; i < s1; ++i) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(X + order[i] * 128) + lane);
    const float2 f0 = __half22float2(u32_as_half2(v.x)), f1 = __half22float2(u32_as_half2(v.y));
    a0 += f0.x; a1 += f0.y; a2 += f1.x; a3 += f1.y;
  }
  const float inv = 1.0f / float(s1 - s0);
  const __half2 h0 = __floats2half2_rn(a0 * inv, a1 * inv), h1 = __floats2half2_rn(a2 * inv, a3 * inv);
  uint2* dst = reinterpret_cast<uint2*>(out + k * 128) + lane;
  if (shift) {  // |new - old| of this centroid, for the convergence test (kmeans.py:213-218)
    const uint2 old = *dst;
    const float2 o0 = __half22float2(u32_as_half2(old.x)), o1 = __half22float2(u32_as_half2(old.y));
    const float2 n0 = __half22float2(h0), n1 = __half22float2(h1);
    float d = (n0.x - o0.x) * (n0.x - o0.x) + (n0.y - o0.y) * (n0.y - o0.y) + (n1.x - o1.x) * (n1.x - o1.x) +
              (n1.y - o1.y) * (n1.y - o1.y);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) d += __shfl_xor_sync(0xffffffffu, d, off);
    if (lane == 0) shift[k] = sqrtf(d);
  }
  *dst = make_uint2(half2_as_u32(h0), half2_as_u32(h1));
}

extern "C" int fpb_kmeans_assign(int device, int dim, int64_t n_centroids, const void* d_centroids,
                                 const float* d_bias, const void* d_points, int64_t n_points, int32_t* d_assign,
                                 void* stream) {
  if (dim != 128) {
    fpb_set_error("fpb_kmeans_assign: this build handles dim=128 (got %d)", dim);
    return FPB_ERR_UNSUPPORTED;
  }
  if (!d_centroids || !d_bias || !d_points || !d_assign || n_centroids < 1 || n_points < 0) {
    fpb_set_error("fpb_kmeans_assign: bad arguments");
    return FPB_ERR_INVALID;
  }
  if (n_points == 0) return FPB_OK;
  FPB_CUDA_CHECK(cudaSetDevice(device));
  return launch_assign(device, n_centroids, d_centroids, d_points, n_points, d_assign, d_bias, nullptr,
                       static_cast<cudaStream_t>(stream), "fpb_kmeans_assign");
}

extern "C" int fpb_nearest_centroid(int device, int dim, int64_t n_centroids, const void* d_centroids,
                                    const float* d_bias, const void* d_points, int64_t n_points, int32_t* d_assign,
                                    float* d_best, void* stream) {
  if (dim != 128) {
    fpb_set_error("fpb_nearest_centroid: this build handles dim=128 (got %d)", dim);
    return FPB_ERR_UNSUPPORTED;
  }
  if (!d_centroids || !d_bias || !d_points || !d_assign || !d_best || n_centroids < 1 || n_points < 0) {
    fpb_set_error("fpb_nearest_centroid: bad arguments");
    return FPB_ERR_INVALID;
  }
  if (n_points == 0) return FPB_OK;
  FPB_CUDA_CHECK(cudaSetDevice(device));
  return launch_assign(device, n_centroids, d_centroids, d_points, n_points, d_assign, d_bias, d_best,
                       static_cast<cudaStream_t>(stream), "fpb_nearest_centroid");
}

extern "C" int fpb_kmeans_update(int device, int dim, int64_t n_centroids, const void* d_points,
                                 const int64_t* d_order, const int64_t* d_seg_offsets, void* d_centroids,
                                 float* d_shift, void* stream) {
  if (dim != 128) {
    fpb_set_error("fpb_kmeans_update: this build handles dim=128 (got %d)", dim);
    return FPB_ERR_UNSUPPORTED;
  }
  if (!d_points || !d_order || !d_seg_offsets || !d_centroids || n_centroids < 1) {
    fpb_set_error("fpb_kmeans_update: bad arguments");
    return FPB_ERR_INVALID;
  }
  FPB_CUDA_CHECK(cudaSetDevice(device));
  segment_mean_kernel<<<unsigned((n_centroids + 7) / 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      static_cast<const __half*>(d_points), d_order, d_seg_offsets, n_centroids, static_cast<__half*>(d_centroids),
      d_shift);
  FPB_LAUNCH_CHECK("segment_mean");
  return FPB_OK;
}

extern "C" int fpb_encode(int device, int nbits, int dim, int64_t n_centroids, const void* d_centroids,
                          const void* d_tokens, int64_t n_tokens, const float* d_cutoffs, int32_t* d_codes,
                          uint8_t* d_residuals, void* stream) {
  if (dim != 128 || (nbits != 2 && nbits != 4)) {
    fpb_set_error("fpb_encode: this build encodes dim=128 with nbits 2 or 4 (got dim=%d nbits=%d)", dim, nbits);
    return FPB_ERR_UNSUPPORTED;
  }
  if (!d_centroids || !d_tokens || !d_cutoffs || !d_codes || !d_residuals || n_centroids < 1 || n_tokens < 0) {
    fpb_set_error("fpb_encode: bad arguments");
    return FPB_ERR_INVALID;
  }
  if (n_tokens == 0) return FPB_OK;
  FPB_CUDA_CHECK(cudaSetDevice(device));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  {
    const int rc = launch_assign(device, n_centroids, d_centroids, d_tokens, n_tokens, d_codes, nullptr, nullptr, st,
                                 "fpb_encode");
    if (rc != FPB_OK) return rc;
  }
  const int pd = dim * nbits / 8;
  const int64_t total = n_tokens * pd;
  const int pblocks = int(((total + 255) / 256) < 65535 * 16 ? ((total + 255) / 256) : 65535 * 16);
  if (nbits == 4)
    encode_pack_kernel<4><<<pblocks, 256, 0, st>>>(static_cast<const __half*>(d_tokens),
                                                   static_cast<const __half*>(d_centroids), d_codes, d_cutoffs,
                                                   n_tokens, dim, d_residuals);
  else
    encode_pack_kernel<2><<<pblocks, 256, 0, st>>>(static_cast<const __half*>(d_tokens),
                                                   static_cast<const __half*>(d_centroids), d_codes, d_cutoffs,
                                                   n_tokens, dim, d_residuals);
  FPB_LAUNCH_CHECK("encode_pack");
  return FPB_OK;
}
