// Building blocks shared by the tcgen05 flow kernels (forward: nsf_tc.cu, data gradient: nsf_tc_bwd.cu):
// CTA shape, mbarrier helpers, the warpgroup -> issuer hand-off, TMEM loads, split-fp16 MMA issue.
#pragma once
#include "nsf_common.cuh"
#include "umma.cuh"

namespace mfb {
namespace tc {

constexpr int kWG = 3;
constexpr int kThreads = (kWG + 1) * 128;   // 3 compute warpgroups + the warpgroup of the MMA-issuer warp
constexpr int kRegsCompute = 160, kRegsIssuer = 32;   // setmaxnreg: 3*128*160 + 128*32 = 64 K registers
constexpr int kTileBytes = 8192;     // 64 rows x 128 B (one fp16 operand tile, K = 64)
constexpr int kABytes = 32768;       // 128 rows x 128 B, hi then lo
// Backward workspace of the tensor-core kernels (tile-major: a row = the 128 particles of a tile).  dL/dphi of a
// feature is stored COMPACT: rows [0, 2 NB) widths and heights (dense), then the only two non-zero entries of the
// derivative block (knots k-1 and k of the particle's bin k) and k itself -- 2 NB + 3 rows instead of 64; the
// consumers rebuild the 64-row operand.  ReLU masks of the hidden layers travel as two 32-bit words per layer.
constexpr int kGRowsOf(int nb) { return 2 * nb + 4; }   // + one row of padding: blocks stay 16-byte multiples
constexpr int kGRows = kGRowsOf(20);

// Tiles are dealt to the (CTA, warpgroup) slots warpgroup-major: slot = wg * gridDim.x + cta, so the slots that get one
// tile more than the others (n / 128 is not a multiple of 3 x grid) are spread over all SMs -- the warpgroups of an SM
// share its issue slots, so what matters is the tile count per SM (1e6 particles on 148 SMs: 53 / 52 instead of 54 / 51).
#ifndef MFB_TC_DEAL_BY_WG
#define MFB_TC_DEAL_BY_WG 1
#endif
__device__ __forceinline__ int64_t first_tile_of(int wg) {
#if MFB_TC_DEAL_BY_WG
  return (int64_t)wg * gridDim.x + blockIdx.x;
#else
  return (int64_t)blockIdx.x * kWG + wg;
#endif
}

__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity);

// mbarrier wait that traps instead of hanging the device if an MMA / TMA never arrives
// mbarrier wait that traps instead of hanging the device if an MMA / TMA never arrives.  Plain
// try_wait polling: the suspend-time-hint form sleeps in coarse quanta (measured: 2-4 thousand
// cycles from arrival to wake-up), which is longer than the MMAs being waited for.
__device__ __forceinline__ void mbar_wait_bounded(uint64_t* bar, uint32_t parity) {
  for (int spins = 0; !mbar_try_wait(bar, parity); ++spins)
    if (spins > (1 << 24)) __trap();
}
// issuer side: poll without occupying the issue port of the compute warps on the same scheduler
__device__ __forceinline__ void mbar_wait_polite(uint64_t* bar, uint32_t parity) {
#ifndef MFB_POLL_NS
#define MFB_POLL_NS 40
#endif
#if defined(MFB_ISSUER_TRYWAIT)
  while (!mbar_try_wait(bar, parity)) {
  }
#else
  while (!mbar_test_wait(bar, parity)) __nanosleep(MFB_POLL_NS);
#endif
}

// Warpgroup -> issuer hand-off: every compute warp arrives (lane 0, after __syncwarp) on a request
// mbarrier of count 4 when its part is done (A rows written / TMEM buffer read) and carries on; the
// issuer warp sees the phase complete and issues the MMAs.  Nobody in the warpgroup waits, and the
// issue work does not land on one of the four compute warps (a warp that issues falls behind the
// others, arrives last again and keeps the duty: measured as 20 % of warp time lost).
// one lane of a fully converged warp (the idiom ptxas recognises: MMAs issued under it take their
// operands from uniform registers without a per-instruction election loop)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void request_arrive(uint64_t* bar) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0)
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

__device__ __forceinline__ void tmem_ld64(uint32_t taddr, float (&v)[64]) {
  uint32_t r[64];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x64.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, "
      "%32, %33, %34, %35, %36, %37, %38, %39, %40, %41, %42, %43, %44, %45, %46, %47, "
      "%48, %49, %50, %51, %52, %53, %54, %55, %56, %57, %58, %59, %60, %61, %62, %63}, [%64];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]), "=r"(r[32]),
        "=r"(r[33]), "=r"(r[34]), "=r"(r[35]), "=r"(r[36]), "=r"(r[37]), "=r"(r[38]), "=r"(r[39]), "=r"(r[40]),
        "=r"(r[41]), "=r"(r[42]), "=r"(r[43]), "=r"(r[44]), "=r"(r[45]), "=r"(r[46]), "=r"(r[47]), "=r"(r[48]),
        "=r"(r[49]), "=r"(r[50]), "=r"(r[51]), "=r"(r[52]), "=r"(r[53]), "=r"(r[54]), "=r"(r[55]), "=r"(r[56]),
        "=r"(r[57]), "=r"(r[58]), "=r"(r[59]), "=r"(r[60]), "=r"(r[61]), "=r"(r[62]), "=r"(r[63])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 64; ++i) v[i] = __uint_as_float(r[i]);
}

// N (a multiple of 4) consecutive columns of this thread's TMEM lane with ONE wait: the spline and the hidden
// steps read their accumulator in pieces, so that no more of it is live in registers than the step works on.
template <int W>
__device__ __forceinline__ void tmem_ld_issue(uint32_t taddr, uint32_t* r) {
  static_assert(W == 4 || W == 8 || W == 16 || W == 32, "tcgen05.ld widths used here");
  if constexpr (W == 4) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
  } else if constexpr (W == 8) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
  } else if constexpr (W == 16) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
  } else {
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
  }
}
template <int N>
__device__ __forceinline__ void tmem_ld_cols(uint32_t taddr, float (&v)[N]) {
  static_assert(N % 4 == 0 && N <= 64, "pieces of 4 to 64 columns");
  uint32_t r[N];
  int c = 0;
#pragma unroll
  for (; c + 32 <= N; c += 32) tmem_ld_issue<32>(taddr + c, r + c);
  if constexpr ((N & 16) != 0) { tmem_ld_issue<16>(taddr + c, r + c); c += 16; }
  if constexpr ((N & 8) != 0) { tmem_ld_issue<8>(taddr + c, r + c); c += 8; }
  if constexpr ((N & 4) != 0) { tmem_ld_issue<4>(taddr + c, r + c); }
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; ++i) v[i] = __uint_as_float(r[i]);
}

// Split MMAs of one K step.  The cross terms (hi*lo + lo*hi, 2^-11 of the result) of ALL K steps
// are accumulated first, the hi*hi terms last: the tensor core rounds the fp32 accumulator once per
// MMA, so only the last few MMAs round at the full magnitude of the result.
__device__ __forceinline__ void mma_cross(uint32_t tmem_d, uint64_t a_hi, uint64_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                          int kstep, uint32_t idesc, uint32_t accumulate) {
  umma::mma_f16_ss(tmem_d, umma::desc_advance_k(a_hi, kstep), umma::desc_advance_k(b_lo, kstep), idesc, accumulate);
  umma::mma_f16_ss(tmem_d, umma::desc_advance_k(a_lo, kstep), umma::desc_advance_k(b_hi, kstep), idesc, 1);
}
__device__ __forceinline__ void mma_main(uint32_t tmem_d, uint64_t a_hi, uint64_t b_hi, int kstep, uint32_t idesc) {
  umma::mma_f16_ss(tmem_d, umma::desc_advance_k(a_hi, kstep), umma::desc_advance_k(b_hi, kstep), idesc, 1);
}
// eight fp32 values -> (hi, lo) fp16 chunks of a 64-wide SWIZZLE_128B tile
__device__ __forceinline__ void store_split8(unsigned char* hi_tile, unsigned char* lo_tile, int row, int chunk,
                                             const float (&x)[8]) {
  __align__(16) __half hi[8], lo[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) umma::split_f16(x[e], hi[e], lo[e]);
  const uint32_t off = umma::sw128_offset(row, chunk);
  *reinterpret_cast<uint4*>(hi_tile + off) = *reinterpret_cast<const uint4*>(hi);
  *reinterpret_cast<uint4*>(lo_tile + off) = *reinterpret_cast<const uint4*>(lo);
}
// hidden unit h has autoregressive class 1 + h % (d-1); perm lists the units sorted by class
static void hidden_classes(int d, int* cls, int* perm) {
  for (int h = 0; h < kH; ++h) cls[h] = 1 + h % (d - 1);
  int p = 0;
  for (int c = 1; c <= d - 1; ++c)
    for (int h = 0; h < kH; ++h)
      if (cls[h] == c) perm[p++] = h;
}

}  // namespace tc

// The tcgen05 layer kernels of nsf_tc.cu, run from one layer's operand image (mfb_nsf_tc_prepare); the C entry points
// of nsf.cu, nsf_inv.cu and nsf_bwd.cu call them when they are given an image.  order: HOST array of d ints.
// nsf_tc_check: MFB_E_UNSUPPORTED for a shape the kernels are not compiled for (mfb_nsf_tc_supported), MFB_E_BADARG
// for an order that is not a permutation, or for an image or particle rows that are not 16-byte aligned (both are
// loaded with bulk copies).  rows: the layer input the kernel bulk-copies (v of the forward and the backward), or
// NULL where the kernel reads its rows with ordinary loads (y of the inverse).
int nsf_tc_check(int d, int hidden_layers, int bins, const void* image, const int32_t* order, const void* rows);
// the layer forward and inverse; each runs nsf_tc_check first
int nsf_tc_fwd(const float* v, int64_t n, int d, int hidden_layers, int bins, const void* image,
               const int32_t* order, const float* logq_in, int first_layer, float* y, float* logq_out,
               cudaStream_t st);
int nsf_tc_inv(const float* y, int64_t n, int d, int hidden_layers, int bins, const void* image,
               const int32_t* order, const float* ladj_in, int last_layer, float* v, float* ladj_out,
               cudaStream_t st);
// first stage of the layer backward: recompute + spline forward/backward into the tile-major workspace matrices of
// nsf_bwd.cu.  The caller has run nsf_tc_check.
int nsf_tc_spline_bwd(const float* v, const float* gy, const float* glogq, int64_t n, int d, const void* image,
                      const int32_t* order, int first_layer, float* acts, float* gphi, uint32_t* masks, float* gvd,
                      float* gmax, int* gmaxes, cudaStream_t st);

}  // namespace mfb
