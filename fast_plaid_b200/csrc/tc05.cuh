// The one home of the tcgen05 / mbarrier / TMA PTX used by the kernels on the 5th-generation tensor cores
// (k1_centroid_v2.cu, encode.cu, k5_maxsim_v5.cu), and the centroid-tile ring that K1 v2 and encode_assign share.
#pragma once

#include <cuda.h>

#include "common.cuh"

// ---- PTX wrappers ------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
// makes the mbarrier.init of this thread visible to the async proxy (TMA, tcgen05.commit)
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.shared::cta.b64 st, [%0];\n}" ::"r"(bar) : "memory");
}
// arrive and add `bytes` to the transaction count the phase waits for
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n.reg .b64 st;\nmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n}" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
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
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// 2-D TMA tile load of the box at (x, y) into shared memory; completion is counted on `bar` in bytes
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* tmap, int x, int y, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
          "r"(dst),
      "l"(tmap), "r"(x), "r"(y), "r"(bar)
      : "memory");
}

// TMEM allocation of COLS columns (a power of 2 >= 32), issued by one whole warp; the base address is written to
// shared memory at `slot`.  The permit is relinquished at once: one CTA per SM, nothing else allocates.
template <int COLS>
__device__ __forceinline__ void tmem_alloc(uint32_t slot) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "n"(COLS));
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
}
template <int COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t base) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "n"(COLS));
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address
// and offsets in 16-byte units, LBO = 1 (unused for swizzled K-major), SBO = 1024 B between 8-row
// groups, version = 1 (Blackwell), layout_type = 2 (SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr) {
  return uint64_t((smem_addr >> 4) & 0x3FFFu) | (uint64_t(1) << 16) | (uint64_t(1024 >> 4) << 32) |
         (uint64_t(1) << 46) | (uint64_t(2) << 61);
}
// kind::f16 instruction descriptor: D = F32, A = B = F16, both K-major, M = 128, N = n.
__device__ __forceinline__ uint32_t umma_idesc(int n) {
  return (1u << 4) | (uint32_t(n >> 3) << 17) | (uint32_t(128 >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
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
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
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
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}


__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// ---- shared-memory layout ----------------------------------------------------------------
// The dynamic shared array `p` rounded up to 1024 B, the alignment of a SWIZZLE_128B atom (the kernels reserve
// 1024 B of slack for it).  A macro because the same code in an inline function reorders the kernels' later
// swizzled-address arithmetic and changes their register allocation.
#define SMEM_ALIGN1024(p) ((p) + ((1024u - (smem_u32(p) & 1023u)) & 1023u))
// Byte offset of 16-byte chunk c (0..15) of row r in a [128 x 128] fp16 operand tile, K-major SWIZZLE_128B:
// two K blocks of 128 rows x 128 B, chunk (c % 8) xor (r % 8) inside the row.
__device__ __forceinline__ uint32_t sw128_off(int r, int c) {
  return uint32_t((c >> 3) * (128 * 128) + (r >> 3) * 1024 + (r & 7) * 128 + (((c & 7) ^ (r & 7)) << 4));
}

// ---- centroid-tile ring (K1 v2, encode_assign) -------------------------------------------
// A resident 128-token A tile against 128 x 128 fp16 centroid tiles that a TMA-producer lane streams through a
// 3-stage shared-memory ring; an MMA-issuer lane accumulates each tile into one of two 128-column TMEM
// accumulators, which an epilogue drains.  Ring iteration g (tiles this CTA streamed before) uses stage g % 3 and
// accumulator g % 2.
constexpr int CT_STAGES = 3;
constexpr int CT_KBLOCK = 128 * 128;   // bytes: 128 rows x 128 B, one SWIZZLE_128B K block
constexpr int CT_TILE = 2 * CT_KBLOCK;  // 32 KB operand tile (K = 128)
constexpr int CT_TMEM_COLS = 256;       // two fp32 accumulators of 128 columns

// Shared addresses of the ring's mbarriers, 10 consecutive uint64 from `bars`: full[3] (TMA -> MMA), empty[3]
// (MMA -> TMA), tfull[2] (MMA -> epilogue), tempty[2] (epilogue -> MMA).
struct CtileBars {
  uint32_t full, empty, tfull, tempty;
  __device__ __forceinline__ explicit CtileBars(const uint64_t* bars)
      : full(smem_u32(bars)), empty(smem_u32(bars + 3)), tfull(smem_u32(bars + 6)), tempty(smem_u32(bars + 8)) {}
  // one thread; tempty counts one arrival per epilogue warp
  __device__ __forceinline__ void init(uint32_t epilogue_warps) const {
    for (int s = 0; s < CT_STAGES; ++s) {
      mbar_init(full + 8 * s, 1);
      mbar_init(empty + 8 * s, 1);
    }
    for (int t = 0; t < 2; ++t) {
      mbar_init(tfull + 8 * t, 1);
      mbar_init(tempty + 8 * t, epilogue_warps);
    }
    mbar_fence_init();
  }
};

// TMA producer (one lane): centroid tiles tile0 .. tile0 + n - 1 into ring iterations it .. it + n - 1.  Each
// tile is two 64-column boxes; rows past K are zero-filled by the TMA unit.
__device__ __forceinline__ void ctile_produce(const CUtensorMap* tmap, const CtileBars& bars, const unsigned char* smB,
                                              int tile0, int n, uint32_t it) {
  for (int i = 0; i < n; ++i) {
    const uint32_t g = it + i;
    const int stage = g % CT_STAGES;
    mbar_wait(bars.empty + 8 * stage, ((g / CT_STAGES) & 1) ^ 1);
    const uint32_t dst = smem_u32(smB + stage * CT_TILE);
    const uint32_t bar = bars.full + 8 * stage;
    mbar_arrive_expect_tx(bar, uint32_t(CT_TILE));
#pragma unroll
    for (int kb = 0; kb < 2; ++kb) tma_load_2d(dst + kb * CT_KBLOCK, tmap, kb * 64, (tile0 + i) * 128, bar);
  }
}

// MMA issuer (one lane): ring iterations it .. it + n - 1, D[token][centroid] = A . B^T (M = N = K = 128) into
// accumulator g % 2 at TMEM columns tmem_base + 128 (g % 2).
__device__ __forceinline__ void ctile_mma(const CtileBars& bars, const unsigned char* smA, const unsigned char* smB,
                                          uint32_t tmem_base, int n, uint32_t it) {
  const uint32_t a_addr = smem_u32(smA);
  const uint32_t idesc = umma_idesc(128);
  for (int i = 0; i < n; ++i) {
    const uint32_t g = it + i;
    const int stage = g % CT_STAGES, acc = g & 1;
    mbar_wait(bars.full + 8 * stage, (g / CT_STAGES) & 1);
    mbar_wait(bars.tempty + 8 * acc, ((g >> 1) & 1) ^ 1);
    tc_fence_after();
    const uint32_t b_addr = smem_u32(smB + stage * CT_TILE);
    const uint32_t d_tmem = tmem_base + acc * 128;
#pragma unroll
    for (int ks = 0; ks < 8; ++ks) {
      const uint32_t off = (ks >> 2) * CT_KBLOCK + (ks & 3) * 32;
      umma_f16(d_tmem, umma_desc(a_addr + off), umma_desc(b_addr + off), idesc, ks > 0 ? 1u : 0u);
    }
    umma_commit(bars.empty + 8 * stage);  // stage reusable once these MMAs have read it
    umma_commit(bars.tfull + 8 * acc);    // accumulator ready
  }
}
