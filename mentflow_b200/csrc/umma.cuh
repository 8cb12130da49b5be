// Minimal tcgen05 / TMEM helpers (sm_100a): shared-memory matrix descriptors for K-major
// SWIZZLE_128B tiles, the kind::f16 instruction descriptor, MMA issue, commit, TMEM
// alloc/load.  Bit layouts follow cute/arch/mma_sm100_desc.hpp (SmemDescriptor /
// InstrDescriptor) of the CUTLASS tree vendored with flashinfer; written out by hand here.
#pragma once
#include <cuda_fp16.h>

#include "common.cuh"

namespace mfb {
namespace umma {

// K-major operand tile: rows of 64 fp16 (128 bytes), 8-row swizzle atoms of 1024 bytes, atoms
// stacked along M/N.  Byte offset of element (row r, 16-byte chunk c in [0,8)):
__device__ __forceinline__ uint32_t sw128_offset(int r, int c) {
  return (uint32_t)((r >> 3) * 1024 + (r & 7) * 128 + ((c ^ (r & 7)) << 4));
}

// SmemDescriptor: start_address[0,14) | LBO[16,30) | SBO[32,46) | version[46,48)=1 | layout[61,64)=2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc_sw128(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;             // leading byte offset (unused for swizzled K-major), 16-B units
  d |= (uint64_t)(1024 >> 4) << 32;   // stride byte offset: 8 rows * 128 B between swizzle atoms
  d |= (uint64_t)1 << 46;             // descriptor version for sm_100
  d |= (uint64_t)2 << 61;             // SWIZZLE_128B
  return d;
}
// advance along K by one UMMA_K (=16 fp16 = 32 bytes) inside the 128-byte swizzle span
__device__ __forceinline__ uint64_t desc_advance_k(uint64_t desc, int kstep) { return desc + (uint64_t)(kstep * 2); }

// K-major tile with 32-byte rows (16 fp16 = ONE MMA K step), SWIZZLE_32B: rows stored back to back,
// swizzle atoms of 8 rows x 32 B = 256 bytes; the swizzle XORs address bit 4 with bit 7, i.e. the
// 16-byte chunk c in {0,1} of row r lands at chunk c ^ ((r >> 2) & 1).
__device__ __forceinline__ uint32_t sw32_offset(int r, int c) {
  return (uint32_t)(r * 32 + ((c ^ ((r >> 2) & 1)) << 4));
}
__device__ __forceinline__ uint64_t make_desc_sw32(uint32_t smem_addr) {
  uint64_t d = (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;            // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(256 >> 4) << 32;   // stride byte offset: 8 rows * 32 B between swizzle atoms
  d |= (uint64_t)1 << 46;            // descriptor version for sm_100
  d |= (uint64_t)6 << 61;            // SWIZZLE_32B
  return d;
}

// InstrDescriptor for kind::f16: fp16 A/B (K-major), fp32 accumulate, shape M x N x 16
__host__ __device__ constexpr uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_f16_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with the A operand in TMEM (lane = row m, one 32-bit column = two consecutive K elements, the even one in
// the low half): written there by the thread that owns the row with tcgen05.st, so A costs no shared-memory traffic
__device__ __forceinline__ void mma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// warp-collective: 32 consecutive 32-bit columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
      "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
// eight consecutive 32-bit columns
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
// four consecutive 32-bit columns
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3])
               : "memory");
}
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// all previously issued MMAs of this thread arrive on the mbarrier when they complete
__device__ __forceinline__ void commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// one warp allocates `cols` (power of two >= 32) TMEM columns; base address lands in *dst (smem)
__device__ __forceinline__ void tmem_alloc(uint32_t* dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

// ---- CTA pairs (cta_group::2): one MMA of M = 256 over the tensor cores of two SMs of a cluster.  Each CTA of the
// pair holds its 128 rows of A and HALF of B (rows [N/2 r, N/2 r + N/2) for cluster rank r) at the same shared-memory
// offsets; D row 128 r + m lands in TMEM lane m of CTA r.  As in CUTLASS's 2-SM kernels, the even CTA issues the MMAs
// and commits, one warp of EACH CTA (the same warp index) allocates and frees the columns, and both CTAs stay
// resident until the last MMA of the pair has completed.
__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
// all threads of both CTAs; orders the shared-memory writes (mbarrier init included) before it cluster-wide
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\nbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// address of the same shared-memory object in the CTA of cluster rank `rank`
__device__ __forceinline__ uint32_t cluster_addr(const void* p, uint32_t rank) {
  uint32_t a;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(p)), "r"(rank));
  return a;
}
// arrive on an mbarrier of any CTA of the cluster (address from cluster_addr); releases this thread's prior writes
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar) : "memory");
}
// wait side of such arrivals: acquires what the arriving threads of either CTA released
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mma_f16_ss_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs arrives on the mbarrier at this offset in both CTAs
__device__ __forceinline__ void commit_pair(uint64_t* bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

// warp-collective: this thread's TMEM lane (= accumulator row), 32 consecutive fp32 columns
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// fp32 -> (hi, lo) fp16 pair with hi + lo = x to ~2^-22 relative (lo may be subnormal)
__device__ __forceinline__ void split_f16(float x, __half& hi, __half& lo) {
  hi = __float2half_rn(x);
  lo = __float2half_rn(x - __half2float(hi));
}

}  // namespace umma
}  // namespace mfb
