// Thin inline-PTX layer over the sm_100a tensor-core path: TMEM allocation, tcgen05.mma
// (A from TMEM or smem, B from smem), tcgen05.ld/st, commit -> mbarrier.
//
// Conventions used by the kernels in this library:
//   * B operand (weights) in shared memory, K-major, SWIZZLE_NONE canonical layout: 8x8-element
//     (8 rows x 16 bytes) core matrices, element (n, k) of a [N, K] fp16 matrix at byte offset
//         (n/8)*SBO + (k/8)*LBO + (n%8)*16 + (k%8)*2,   LBO = 128, SBO = (K/8)*128.
//   * A operand (activations) in TMEM ("TS" form): row m on lane m, two fp16 per 32-bit column,
//     element (m, k) in column k/2, low half = even k.  The thread that owns TMEM lane m (= stream m
//     of the tile) writes its own row with tcgen05.st, so no shared-memory staging or proxy fence.
//   * A operand in shared memory ("SS" form) where it arrives by bulk copy: the row-tiled layout
//     [K/8 chunks][128 rows][8 elements] (kTileChunkBytes = 2048 per chunk), i.e. the same core matrices with
//     LBO = 2048 (K direction), SBO = 128 (M direction).  It is what the layers hand to each other in HBM, so one
//     contiguous copy of (K/8)*2048 bytes is an MMA-ready operand.
//   * D accumulators fp32 in TMEM, row m on lane m, one column per n.
#pragma once

#include <cuda_fp16.h>
#include <stdint.h>

namespace kws {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---- TMEM allocation (one warp, whole-warp collective)
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}

__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// generic-proxy writes to smem -> visible to the async proxy (tcgen05.mma operand fetch)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ bool mbar_try_wait(uint32_t addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(ok)
      : "r"(addr), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a tensor-core op that never completes must trap, not hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  for (uint32_t spins = 0; !mbar_try_wait(addr, parity); ++spins) {
    if (spins > (1u << 24)) __trap();
  }
}

// ---- bulk async copy (TMA without a tensor map): `bytes` contiguous bytes global -> shared through the async proxy,
// completion counted on an mbarrier whose pending transaction count was raised by mbar_arrive_expect_tx.
// Source, destination and size are multiples of 16 bytes.  SASS: UBLKCP.
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// ---- descriptors
// shared-memory matrix descriptor, K-major, SWIZZLE_NONE (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3fffu);             // [0,14)  start address >> 4
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3fffu) << 16;   // [16,30) leading byte offset >> 4
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3fffu) << 32;   // [32,46) stride byte offset >> 4
  d |= static_cast<uint64_t>(1) << 46;                            // [46,48) descriptor version = 1 (Blackwell)
  return d;                                                       // base_offset 0, lbo_mode 0, layout SWIZZLE_NONE
}
// instruction descriptor for kind::f16: fp16 A/B (both K-major), fp32 accumulate (cute::UMMA::InstrDescriptor)
__host__ __device__ constexpr uint32_t idesc_f16(int M, int N) {
  return (1u << 4)                                 // c_format = F32
         | (0u << 7) | (0u << 10)                  // a_format = b_format = F16
         | (0u << 15) | (0u << 16)                 // a_major = b_major = K
         | (static_cast<uint32_t>(N >> 3) << 17)   // n_dim
         | (static_cast<uint32_t>(M >> 4) << 24);  // m_dim
}

// same, B operand MN-major (N contiguous: 8 n-elements per 16-byte row, 8 k-rows per core matrix; in the smem
// descriptor SBO is then the stride between 8-groups of N and LBO the stride between 8-groups of K)
__host__ __device__ constexpr uint32_t idesc_f16_bmn(int M, int N) { return idesc_f16(M, N) | (1u << 16); }

// One lane of a CONVERGED warp (elect.sync).  Guard tcgen05.mma / commit / bulk-copy issue with this, not with
// `lane == 0`: ptxas recognises the elected region as single-threaded and emits the uniform-datapath instruction
// as is, whereas under an ordinary lane predicate it wraps EVERY such instruction in a loop over the active lanes
// (ELECT, two PLOP3, BRA.U.ANY: six instructions and a branch per MMA).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// ---- MMA (issued by ONE thread).  D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(static_cast<uint32_t>(accumulate))
      : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, bool accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(static_cast<uint32_t>(accumulate))
      : "memory");
}
// arrive on an mbarrier once every tcgen05 op issued so far by this thread has completed
__device__ __forceinline__ void commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- TMEM <-> registers: this thread's lane (warp w%4 owns lanes 32*(w%4)..+31), consecutive columns
__device__ __forceinline__ void ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void st8(uint32_t taddr, const uint32_t (&v)[8]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(v[0]),
      "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
      : "memory");
}
__device__ __forceinline__ void st4(uint32_t taddr, const uint32_t (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(v[0]), "r"(v[1]),
               "r"(v[2]), "r"(v[3])
               : "memory");
}

__device__ __forceinline__ void st2(uint32_t taddr, uint32_t a, uint32_t b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(taddr), "r"(a), "r"(b) : "memory");
}

__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);      // .x (low 16 bits) = lo
  return *reinterpret_cast<const uint32_t*>(&h);
}

// 8 fp32 values -> 8 fp16 roundings (hi) and the 8 fp16 roundings of what they lost (lo): x = hi + lo to 2^-22 relative
__device__ __forceinline__ void split_half8(const float (&v)[8], uint4* hi, uint4* lo) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const __half2 hh = __floats2half2_rn(v[2 * i], v[2 * i + 1]);
    const float2 b = __half22float2(hh);
    h[i] = *reinterpret_cast<const uint32_t*>(&hh);
    l[i] = pack_half2(v[2 * i] - b.x, v[2 * i + 1] - b.y);
  }
  *hi = make_uint4(h[0], h[1], h[2], h[3]);
  *lo = make_uint4(l[0], l[1], l[2], l[3]);
}

// byte offset of element (n, k) of a [N, K] fp16 matrix in the canonical K-major SWIZZLE_NONE layout
__host__ __device__ constexpr size_t canon_offset(int n, int k, int K) {
  return static_cast<size_t>(n / 8) * (static_cast<size_t>(K / 8) * 128) + static_cast<size_t>(k / 8) * 128 +
         static_cast<size_t>(n % 8) * 16 + static_cast<size_t>(k % 8) * 2;
}

// row-tiled A operand (see the conventions above): byte offset of element (m, k) of a [128, K] fp16 tile
constexpr uint32_t kTileChunkBytes = 2048;
__host__ __device__ constexpr size_t tile_offset(int m, int k) {
  return static_cast<size_t>(k / 8) * kTileChunkBytes + static_cast<size_t>(m) * 16 + static_cast<size_t>(k % 8) * 2;
}

// byte offset of element (n, k) of a [N, K] fp16 matrix in the canonical MN-major SWIZZLE_NONE layout
// (LBO = 128 between 8-groups of K, SBO = (K/8)*128 between 8-groups of N)
__host__ __device__ constexpr size_t canon_offset_mn(int n, int k, int K) {
  return static_cast<size_t>(n / 8) * (static_cast<size_t>(K / 8) * 128) + static_cast<size_t>(k / 8) * 128 +
         static_cast<size_t>(k % 8) * 16 + static_cast<size_t>(n % 8) * 2;
}

}  // namespace tc
}  // namespace kws
