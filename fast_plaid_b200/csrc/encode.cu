// Index-build encode kernels (SURVEY.md 8(f-1); replaces the per-batch closure of create_index,
// rust/index/create.rs:404-428):
//   * assign : code[t] = argmax_k fp16(<x_t, c_k>)  (compress_into_codes, create.rs:148-170) on
//              tcgen05 -- the K1 v2 pipeline (TMA-fed centroid tiles, TMEM accumulators) with an
//              argmax epilogue instead of the S store; ties -> smallest centroid id, which is what
//              ATen's CPU argmax returns
//   * pack   : residual = fp16(x - c[code]); bucket = #cutoffs < residual (bucketize right=false,
//              create.rs:413-414); each index written LSB-first into nbits bits, bits packed
//              big-endian per byte (create.rs:416-427, packbits :176-184)
#include <cuda.h>
#include <string.h>

#include "kernels.h"

namespace {

constexpr int EN_THREADS = 288;
constexpr int EN_STAGES = 3;
constexpr int EN_KBLOCK = 128 * 128;
constexpr int EN_TILE = 2 * EN_KBLOCK;
constexpr int EN_TMEM_COLS = 256;

struct EnSmem {
  static constexpr int a_off = 0;
  static constexpr int b_off = EN_TILE;
  static constexpr int bar_off = b_off + EN_STAGES * EN_TILE;
  static constexpr int bytes = bar_off + 256 + 1024;
};
__device__ __forceinline__ void en_mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void en_mbar_arrive(uint32_t bar) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void en_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ uint64_t en_desc(uint32_t smem_addr) {
  return uint64_t((smem_addr >> 4) & 0x3FFFu) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
__device__ __forceinline__ void en_umma(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                        uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void en_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void en_tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// 16-byte chunk c (0..15) of row r of a [128 x 128] fp16 operand tile, K-major SWIZZLE_128B
__device__ __forceinline__ uint32_t en_sw_off(int r, int c) {
  return uint32_t((c >> 3) * EN_KBLOCK + (r >> 3) * 1024 + (r & 7) * 128 + (((c & 7) ^ (r & 7)) << 4));
}


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
  const uint32_t dyn_addr = smem_u32(smem_dyn);
  unsigned char* base = smem_dyn + ((1024u - (dyn_addr & 1023u)) & 1023u);
  unsigned char* smA = base + EnSmem::a_off;
  unsigned char* smB = base + EnSmem::b_off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(base + EnSmem::bar_off);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 16);
  const uint32_t bar_full = smem_u32(bars), bar_empty = smem_u32(bars + 3);
  const uint32_t bar_tfull = smem_u32(bars + 6), bar_tempty = smem_u32(bars + 8);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  if (tid == 0) {
    for (int s = 0; s < EN_STAGES; ++s) {
      en_mbar_init(bar_full + 8 * s, 1);
      en_mbar_init(bar_empty + 8 * s, 1);
    }
    for (int t = 0; t < 2; ++t) {
      en_mbar_init(bar_tfull + 8 * t, 1);
      en_mbar_init(bar_tempty + 8 * t, 4);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "n"(EN_TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
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
      *reinterpret_cast<uint4*>(smA + en_sw_off(r, c)) = v;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    if (warp == 4) {
      if (lane == 0) {
        for (int i = 0; i < n_ctiles; ++i) {
          const uint32_t g = it + i;
          const int stage = g % EN_STAGES;
          en_mbar_wait(bar_empty + 8 * stage, ((g / EN_STAGES) & 1) ^ 1);
          const uint32_t dst = smem_u32(smB + stage * EN_TILE);
          const uint32_t bar = bar_full + 8 * stage;
          asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}" ::"r"(bar),
                       "r"(uint32_t(EN_TILE))
                       : "memory");
#pragma unroll
          for (int kb = 0; kb < 2; ++kb) {
            asm volatile(
                "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
                    "r"(dst + kb * EN_KBLOCK),
                "l"(&tmap_c), "r"(kb * 64), "r"(i * 128), "r"(bar)
                : "memory");
          }
        }
      }
      __syncwarp();
    } else if (warp == 8) {
      if (lane == 0) {
        const uint32_t a_addr = smem_u32(smA);
        const uint32_t idesc = (1u << 4) | (uint32_t(128 >> 3) << 17) | (uint32_t(128 >> 4) << 24);
        for (int i = 0; i < n_ctiles; ++i) {
          const uint32_t g = it + i;
          const int stage = g % EN_STAGES, acc = g & 1;
          en_mbar_wait(bar_full + 8 * stage, (g / EN_STAGES) & 1);
          en_mbar_wait(bar_tempty + 8 * acc, ((g >> 1) & 1) ^ 1);
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t b_addr = smem_u32(smB + stage * EN_TILE);
          const uint32_t d_tmem = tmem_base + acc * 128;
#pragma unroll
          for (int ks = 0; ks < 8; ++ks) {
            const uint32_t off = (ks >> 2) * EN_KBLOCK + (ks & 3) * 32;
            en_umma(d_tmem, en_desc(a_addr + off), en_desc(b_addr + off), idesc, ks > 0 ? 1u : 0u);
          }
          en_commit(bar_empty + 8 * stage);
          en_commit(bar_tfull + 8 * acc);
        }
      }
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
        en_mbar_wait(bar_tfull + 8 * acc, (g >> 1) & 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
        for (int c0 = 0; c0 < 128; c0 += 32) {
          uint32_t r[32];
          en_tmem_ld32(tmem_base + (uint32_t(warp * 32) << 16) + acc * 128 + c0, r);
#pragma unroll
          for (int x = 0; x < 32; ++x) {
            // encode: the reference compares fp16 scores (half matmul output); first maximum wins
            const float v = KMEANS ? __uint_as_float(r[x]) + s_bias[warp][acc][c0 + x]
                                   : __half2float(__float2half_rn(__uint_as_float(r[x])));
            if (c0 + x < rows_valid && v > best) {
              best = v;
              best_k = k0 + c0 + x;
            }
          }
        }
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) en_mbar_arrive(bar_tempty + 8 * acc);
      }
      if (tok < n) {
        codes[tok] = best_k;
        if (KMEANS && best_out) best_out[tok] = best;
      }
    }
    it += uint32_t(n_ctiles);
  }

  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 8) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(EN_TMEM_COLS));
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

typedef CUresult (*en_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

// tensor map of the centroid table + launch of the assign kernel (shared by fpb_encode, fpb_kmeans_assign and
// fpb_nearest_centroid; d_best needs d_bias)
static int launch_assign(int device, int64_t n_centroids, const void* d_centroids, const void* d_tokens,
                         int64_t n_tokens, int32_t* d_codes, const float* d_bias, float* d_best, cudaStream_t st,
                         const char* who) {
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn ||
      qres != cudaDriverEntryPointSuccess) {
    fpb_set_error("%s: cuTensorMapEncodeTiled is not available from this driver", who);
    return FPB_ERR_CUDA;
  }
  CUtensorMap tm;
  const cuuint64_t gdim[2] = {128, cuuint64_t(n_centroids)};
  const cuuint64_t gstride[1] = {256};
  const cuuint32_t box[2] = {64, 128};
  const cuuint32_t estr[2] = {1, 1};
  if (reinterpret_cast<en_encode_tiled_fn>(fn)(&tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(d_centroids),
                                               gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                               CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS) {
    fpb_set_error("%s: cuTensorMapEncodeTiled failed", who);
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
