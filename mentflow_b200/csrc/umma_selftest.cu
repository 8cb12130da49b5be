// Self-test of the tcgen05 building blocks used by the tensor-core conditioner:
// D[128 x N] = A[128 x 64] * B[N x 64]^T with fp32 inputs split into fp16 (hi, lo) pairs and
// three kind::f16 MMAs per K step (hi*hi + hi*lo + lo*hi), accumulators in TMEM.
#include "umma.cuh"

namespace mfb {

constexpr int kSelfWaitLimit = 1 << 22;

__global__ void __launch_bounds__(128, 1)
umma_selftest_kernel(const float* __restrict__ A, const float* __restrict__ B, int N, float* __restrict__ D,
                     int* __restrict__ err) {
  extern __shared__ __align__(1024) unsigned char smem[];
  // [A_hi 16K][A_lo 16K][B_hi N*128][B_lo N*128]
  unsigned char* a_hi = smem;
  unsigned char* a_lo = smem + 16384;
  unsigned char* b_hi = smem + 32768;
  unsigned char* b_lo = b_hi + (size_t)N * 128;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  const int tid = threadIdx.x;

  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  if (tid < 32) umma::tmem_alloc(&tmem_base, 256);
  // operands: thread r handles row r of A; rows r (and r+128 for N = 256...) of B
  for (int r = tid; r < 128 + N; r += 128) {
    const bool isA = r < 128;
    const int row = isA ? r : r - 128;
    const float* src = isA ? A + (size_t)row * 64 : B + (size_t)row * 64;
    unsigned char* dhi = isA ? a_hi : b_hi;
    unsigned char* dlo = isA ? a_lo : b_lo;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      __align__(16) __half hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) umma::split_f16(src[c * 8 + e], hi[e], lo[e]);
      const uint32_t off = umma::sw128_offset(row, c);
      *reinterpret_cast<uint4*>(dhi + off) = *reinterpret_cast<const uint4*>(hi);
      *reinterpret_cast<uint4*>(dlo + off) = *reinterpret_cast<const uint4*>(lo);
    }
  }
  fence_proxy_async();   // generic-proxy smem writes -> visible to the tensor core (async proxy)
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tbase = tmem_base;

  if (tid == 0) {
    const uint32_t idesc = umma::make_idesc_f16(128, N);
    const uint64_t da_hi = umma::make_desc_sw128(smem_u32(a_hi)), da_lo = umma::make_desc_sw128(smem_u32(a_lo));
    const uint64_t db_hi = umma::make_desc_sw128(smem_u32(b_hi)), db_lo = umma::make_desc_sw128(smem_u32(b_lo));
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      umma::mma_f16_ss(tbase, umma::desc_advance_k(da_hi, k), umma::desc_advance_k(db_hi, k), idesc, acc);
      acc = 1;
      umma::mma_f16_ss(tbase, umma::desc_advance_k(da_hi, k), umma::desc_advance_k(db_lo, k), idesc, 1);
      umma::mma_f16_ss(tbase, umma::desc_advance_k(da_lo, k), umma::desc_advance_k(db_hi, k), idesc, 1);
    }
    umma::commit(&bar);
  }
  // everyone waits for the accumulator
  int spins = 0;
  while (!mbar_try_wait(&bar, 0)) {
    if (++spins > kSelfWaitLimit) {
      if (tid == 0) *err = 1;
      break;
    }
  }
  umma::fence_after_sync();
  const int warp = tid >> 5;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    umma::tmem_ld32(tbase + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) D[(size_t)tid * N + c0 + i] = v[i];
  }
  umma::fence_before_sync();
  __syncthreads();
  if (tid < 32) umma::tmem_dealloc(tbase, 256);
}

// Second self-test: one K step (K = 16) with 32-byte-row SWIZZLE_32B operand tiles (the packed
// weight / bias tiles of the flow kernel) against a SWIZZLE_128B A operand, as issued there:
//   mode 0: A sw32 x B sw32      mode 1: A sw128 (K step `kstep` of a 64-wide tile) x B sw32
__global__ void __launch_bounds__(128, 1)
umma_selftest_sw32_kernel(const float* __restrict__ A, const float* __restrict__ B, int N, int mode, int kstep,
                          float* __restrict__ D, int* __restrict__ err) {
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* a32 = smem;               // 128 x 32 B
  unsigned char* a128 = smem + 4096;       // 128 x 128 B (1024-aligned)
  unsigned char* b32 = smem + 4096 + 16384;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  if (tid < 32) umma::tmem_alloc(&tmem_base, 256);
  for (int i = tid; i < 16384 / 16; i += 128) reinterpret_cast<uint4*>(a128)[i] = make_uint4(0, 0, 0, 0);
  __syncthreads();
  for (int r = tid; r < 128 + N; r += 128) {
    const bool isA = r < 128;
    const int row = isA ? r : r - 128;
    const float* src = isA ? A + (size_t)row * 16 : B + (size_t)row * 16;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      __align__(16) __half h[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) h[e] = __float2half_rn(src[c * 8 + e]);
      if (isA) {
        *reinterpret_cast<uint4*>(a32 + umma::sw32_offset(row, c)) = *reinterpret_cast<const uint4*>(h);
        *reinterpret_cast<uint4*>(a128 + umma::sw128_offset(row, 2 * kstep + c)) = *reinterpret_cast<const uint4*>(h);
      } else {
        *reinterpret_cast<uint4*>(b32 + umma::sw32_offset(row, c)) = *reinterpret_cast<const uint4*>(h);
      }
    }
  }
  fence_proxy_async();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tbase = tmem_base;
  if (tid == 0) {
    const uint32_t idesc = umma::make_idesc_f16(128, N);
    const uint64_t da = mode == 0 ? umma::make_desc_sw32(smem_u32(a32))
                                  : umma::desc_advance_k(umma::make_desc_sw128(smem_u32(a128)), kstep);
    umma::mma_f16_ss(tbase, da, umma::make_desc_sw32(smem_u32(b32)), idesc, 0);
    umma::commit(&bar);
  }
  int spins = 0;
  while (!mbar_try_wait(&bar, 0)) {
    if (++spins > kSelfWaitLimit) {
      if (tid == 0) *err = 1;
      break;
    }
  }
  umma::fence_after_sync();
  const int warp = tid >> 5;
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    umma::tmem_ld32(tbase + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) D[(size_t)tid * N + c0 + i] = v[i];
  }
  umma::fence_before_sync();
  __syncthreads();
  if (tid < 32) umma::tmem_dealloc(tbase, 256);
}

// Third self-test: the split GEMM of the first test with the A operand in TENSOR MEMORY (tcgen05.st by the thread
// that owns the row, tcgen05.mma with a TMEM A address): the form the KDE-2D kernel uses to keep its kernel rows out
// of shared memory.  D at columns [0, N), A hi at [128, 160), A lo at [160, 192)  (N <= 128).
__global__ void __launch_bounds__(128, 1)
umma_selftest_ts_kernel(const float* __restrict__ A, const float* __restrict__ B, int N, float* __restrict__ D,
                        int* __restrict__ err) {
  extern __shared__ __align__(1024) unsigned char smem[];
  unsigned char* b_hi = smem;
  unsigned char* b_lo = b_hi + (size_t)N * 128;
  __shared__ uint64_t bar;
  __shared__ uint32_t tmem_base;
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) {
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  if (tid < 32) umma::tmem_alloc(&tmem_base, 256);
  for (int row = tid; row < N; row += 128) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      __align__(16) __half hi[8], lo[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) umma::split_f16(B[(size_t)row * 64 + c * 8 + e], hi[e], lo[e]);
      const uint32_t off = umma::sw128_offset(row, c);
      *reinterpret_cast<uint4*>(b_hi + off) = *reinterpret_cast<const uint4*>(hi);
      *reinterpret_cast<uint4*>(b_lo + off) = *reinterpret_cast<const uint4*>(lo);
    }
  }
  fence_proxy_async();
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  const uint32_t tbase = tmem_base;
  {   // row tid of A -> TMEM lane tid
    uint32_t hi[32], lo[32];
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      __half h0, l0, h1, l1;
      umma::split_f16(A[(size_t)tid * 64 + 2 * c], h0, l0);
      umma::split_f16(A[(size_t)tid * 64 + 2 * c + 1], h1, l1);
      hi[c] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
      lo[c] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
    }
    const uint32_t lane_base = tbase + ((uint32_t)(warp * 32) << 16);
    umma::tmem_st32(lane_base + 128, hi);
    umma::tmem_st32(lane_base + 160, lo);
    umma::tmem_wait_st();
  }
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  if (tid == 0) {
    const uint32_t idesc = umma::make_idesc_f16(128, N);
    const uint64_t db_hi = umma::make_desc_sw128(smem_u32(b_hi)), db_lo = umma::make_desc_sw128(smem_u32(b_lo));
    uint32_t acc = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {   // one K step = 16 elements = 8 packed columns
      umma::mma_f16_ts(tbase, tbase + 128 + 8 * k, umma::desc_advance_k(db_hi, k), idesc, acc);
      acc = 1;
      umma::mma_f16_ts(tbase, tbase + 128 + 8 * k, umma::desc_advance_k(db_lo, k), idesc, 1);
      umma::mma_f16_ts(tbase, tbase + 160 + 8 * k, umma::desc_advance_k(db_hi, k), idesc, 1);
    }
    umma::commit(&bar);
  }
  int spins = 0;
  while (!mbar_try_wait(&bar, 0)) {
    if (++spins > kSelfWaitLimit) {
      if (tid == 0) *err = 1;
      break;
    }
  }
  umma::fence_after_sync();
  for (int c0 = 0; c0 < N; c0 += 32) {
    float v[32];
    umma::tmem_ld32(tbase + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) D[(size_t)tid * N + c0 + i] = v[i];
  }
  umma::fence_before_sync();
  __syncthreads();
  if (tid < 32) umma::tmem_dealloc(tbase, 256);
}

// Fourth self-test: the 2-SM MMA of a CTA pair (cluster of 2, cta_group::2), as the pair kernel of the flow layer
// issues it: D[256 x 64] = A[256 x K] * B[64 x K]^T, CTA r holding rows [128 r, 128 r + 128) of A and rows
// [32 r, 32 r + 32) of B -- the first or second contiguous half of a 64-row operand tile.
//   mode 0: K = 16, SWIZZLE_32B tiles (one K step)      mode 1: K = 64, SWIZZLE_128B tiles (four K steps)
// Both CTAs signal "operands written" to the even CTA's mbarrier (count 2) by a remote arrive; the even CTA issues
// and commits to the mbarriers of both.
__global__ void __launch_bounds__(128, 1)
umma_selftest_pair_kernel(const float* __restrict__ A, const float* __restrict__ B, int mode, float* __restrict__ D,
                          int* __restrict__ err) {
  extern __shared__ unsigned char smem_raw[];
  // same offsets in both CTAs: the MMA addresses the operands of the peer with the issuer's descriptors
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* a_t = smem;            // 128 rows: 4 KB (mode 0) / 16 KB (mode 1)
  unsigned char* b_t = smem + 16384;    // 32 rows: 1 KB / 4 KB
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 16384 + 4096);   // [0] MMA done (count 1), [1] request (count 2)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
  const int tid = threadIdx.x, K = mode == 0 ? 16 : 64;
  const uint32_t rank = umma::cluster_rank();
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 2);
    fence_mbar_init();
  }
  if (tid < 32) umma::tmem_alloc_pair(tmem_slot, 64);
  for (int r = tid; r < 128 + 32; r += 128) {
    const bool isA = r < 128;
    const int row = isA ? r : r - 128;
    const float* src = isA ? A + (size_t)(128 * rank + row) * K : B + (size_t)(32 * rank + row) * K;
    for (int c = 0; c < K / 8; ++c) {
      __align__(16) __half h[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) h[e] = __float2half_rn(src[c * 8 + e]);
      const uint32_t off = mode == 0 ? umma::sw32_offset(row, c) : umma::sw128_offset(row, c);
      *reinterpret_cast<uint4*>((isA ? a_t : b_t) + off) = *reinterpret_cast<const uint4*>(h);
    }
  }
  fence_proxy_async();
  umma::fence_before_sync();
  umma::cluster_sync();   // mbarriers of both CTAs initialised, operands of both written
  umma::fence_after_sync();
  const uint32_t tbase = *tmem_slot;
  if (tid == 0) umma::mbar_arrive_cluster(umma::cluster_addr(&bars[1], 0));
  if (rank == 0 && tid == 0) {
    int spins = 0;
    while (!umma::mbar_try_wait_cluster(&bars[1], 0)) {
      if (++spins > kSelfWaitLimit) {
        *err = 2;
        break;
      }
    }
    umma::fence_after_sync();
    const uint32_t idesc = umma::make_idesc_f16(256, 64);
    if (mode == 0) {
      umma::mma_f16_ss_pair(tbase, umma::make_desc_sw32(smem_u32(a_t)), umma::make_desc_sw32(smem_u32(b_t)), idesc, 0);
    } else {
      const uint64_t da = umma::make_desc_sw128(smem_u32(a_t)), db = umma::make_desc_sw128(smem_u32(b_t));
      for (int k = 0; k < 4; ++k)
        umma::mma_f16_ss_pair(tbase, umma::desc_advance_k(da, k), umma::desc_advance_k(db, k), idesc, k > 0);
    }
    umma::commit_pair(&bars[0]);
  }
  int spins = 0;
  while (!mbar_try_wait(&bars[0], 0)) {
    if (++spins > kSelfWaitLimit) {
      if (tid == 0) *err = 1;
      break;
    }
  }
  umma::fence_after_sync();
  const int warp = tid >> 5;
  for (int c0 = 0; c0 < 64; c0 += 32) {
    float v[32];
    umma::tmem_ld32(tbase + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll
    for (int i = 0; i < 32; ++i) D[(size_t)(128 * rank + tid) * 64 + c0 + i] = v[i];
  }
  umma::fence_before_sync();
  umma::cluster_sync();   // no CTA frees its columns or exits while the pair's MMA may still use them
  if (tid < 32) umma::tmem_dealloc_pair(tbase, 64);
}

}  // namespace mfb

extern "C" int mfb_selftest_umma_pair(const float* a, const float* b, int mode, float* d, int* err, void* stream) {
  MFB_CHECK_ARG(a && b && d && err && (mode == 0 || mode == 1));
  const size_t smem = 16384 + 4096 + 64 + 1024;
  MFB_CUDA(cudaFuncSetAttribute(mfb::umma_selftest_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2);
  cfg.blockDim = dim3(128);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MFB_CUDA(cudaLaunchKernelEx(&cfg, mfb::umma_selftest_pair_kernel, a, b, mode, d, err));
  return mfb::launch_status();
}

extern "C" int mfb_selftest_umma_ts(const float* a, const float* b, int n, float* d, int* err, void* stream) {
  MFB_CHECK_ARG(a && b && d && err && (n == 64 || n == 96 || n == 128));
  const size_t smem = (size_t)n * 256 + 1024;
  MFB_CUDA(cudaFuncSetAttribute(mfb::umma_selftest_ts_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mfb::umma_selftest_ts_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(a, b, n, d, err);
  return mfb::launch_status();
}

extern "C" int mfb_selftest_umma_sw32(const float* a, const float* b, int n, int mode, int kstep, float* d, int* err,
                                      void* stream) {
  MFB_CHECK_ARG(a && b && d && err && (n == 64 || n == 128) && (mode == 0 || mode == 1) && kstep >= 0 && kstep < 4);
  const size_t smem = 4096 + 16384 + (size_t)n * 32 + 1024;
  MFB_CUDA(cudaFuncSetAttribute(mfb::umma_selftest_sw32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mfb::umma_selftest_sw32_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(a, b, n, mode, kstep, d, err);
  return mfb::launch_status();
}

extern "C" int mfb_selftest_umma(const float* a, const float* b, int n, float* d, int* err, void* stream) {
  MFB_CHECK_ARG(a && b && d && err && (n == 64 || n == 128 || n == 256));
  const size_t smem = 32768 + (size_t)n * 256 + 1024;
  MFB_CUDA(cudaFuncSetAttribute(mfb::umma_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mfb::umma_selftest_kernel<<<1, 128, smem, (cudaStream_t)stream>>>(a, b, n, d, err);
  return mfb::launch_status();
}
