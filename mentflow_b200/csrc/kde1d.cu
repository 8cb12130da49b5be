// Fused linear projection + 1-D binning (Gaussian KDE deposit or exact histogram).
//
// Replaces, for all K measurements in ONE pass over the particles (reference file:line,
// relative to mentflow/):
//   simulate/simulate.py:29-33, simulate/transform.py:67-68   u = x.clone() @ M_k^T  (K SGEMMs + K clones)
//   diagnostics/diagnostics.py:116-131                       project, then KDE or torch.histogram
//   diagnostics/histogram.py:37-39                           dense (N,B) kernel matrix + mean
//
// Design (B200): the particle block streams HBM -> smem through the TMA engine
// (cp.async.bulk + mbarrier, double buffered).  Thread t of a CTA owns projection
// k = t % Kc and particle slice t / Kc, and a PRIVATE column of bins in shared memory
// (pairs of rows as float2, blocked per warp: [warp][pair][lane] -- a warp touches 256
// contiguous bytes whatever bins its lanes hit, conflict free), so deposits are plain 8-byte
// LDS/FADD/STS -- no atomics, and the accumulation order is fixed => run-to-run deterministic.
// Each particle touches only the pair-aligned window of 2R+2 bins around its projection
// (everything beyond ~8.9 sigma is below 1e-17 of a central tap), instead of all B; the taps
// come from recurrences whose factors are all <= 1 (4 MUFU, packed-fp32 multiplies, no overflow at
// any bandwidth).  Per-CTA partials are merged in a fixed order by a second tiny kernel
// (kde1d_finish_kernel), which also normalises and evaluates the KL term.  The kernel sits at its shared-memory floor (80 B read + written
// per particle-projection); the backward kernel uses the same taps on a zero-padded table.
#include <type_traits>

#include "common.cuh"
#include "multipole.cuh"

namespace mfb {

constexpr int kTile = 1024;        // particles per TMA stage
constexpr int kBinThreads = 256;   // upper bound on threads per CTA of the deposit kernels

struct ProjLaunch {
  int kc;        // projections handled per CTA (<= kBinThreads)
  int slices;    // particle slices per CTA
  int threads;   // kc * slices
  int kchunks;   // gridDim.y
  int grid_x;    // particle-tile CTAs
  int tile;      // particles per stage (multiple of 4, <= kTile)
  size_t smem;   // dynamic shared memory bytes
};

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Window radius in bins.  Dropped taps are further than (R+0.5) bins = 8.85 sigma from the
// particle, i.e. below exp(-0.5*8.85^2) ~ 1e-17 of a central tap.  That is far below fp32
// resolution of the *profile*, but the KL gradient divides by (p_b + 1e-12): a bin reached
// only by tails must still see them, or dL/dx is off by 1e-4 (measured) -- hence 1e-17, not 1e-9.
static inline int window_radius(double sigma_over_delta) {
  double r = 8.85 * sigma_over_delta - 0.5;
  int ri = (int)r;
  if ((double)ri < r) ++ri;
  return ri < 1 ? 1 : ri;
}

static ProjLaunch plan_launch(int64_t n, int d, int k, int b, int bytes_per_bin, size_t extra_smem) {
  ProjLaunch L;
  L.kchunks = (k + kBinThreads - 1) / kBinThreads;
  L.kc = (k + L.kchunks - 1) / L.kchunks;
  // private bins must fit: b * threads * bytes_per_bin + 2 stages of x
  size_t budget = 200 * 1024 - extra_smem;
  int max_threads = kBinThreads;
  while (max_threads > L.kc && (size_t)b * max_threads * bytes_per_bin + 2ull * kTile * d * 4 > budget)
    max_threads -= 32;
  L.slices = max_threads / L.kc;
  if (L.slices < 1) L.slices = 1;
  L.threads = L.kc * L.slices;
  int sms = sm_count();
  // small batches: shrink the tile so that every SM gets work
  int tile = kTile;
  while (tile > 128 && ceil_div64(n, tile) < 2 * sms) tile >>= 1;
  L.tile = tile;
  int64_t tiles = ceil_div64(n, tile);
  // bins are stored with a row stride of threads rounded up to 32: bank = thread % 32 for any bin
  size_t smem = 2ull * tile * d * 4 + 64 + (size_t)b * ((L.threads + 31) & ~31) * bytes_per_bin + extra_smem;
  int ctas_per_sm = (int)((220 * 1024) / (smem + 1024));
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  if (ctas_per_sm > 4) ctas_per_sm = 4;
  int64_t gx = (int64_t)sms * ctas_per_sm;
  if (gx > tiles) gx = tiles;
  if (gx < 1) gx = 1;
  L.grid_x = (int)gx;
  L.smem = smem;
  return L;
}

// ---- TMA tile pipeline ---------------------------------------------------------------------
struct TilePipe {
  float* buf[2];
  uint64_t* bar;  // 2 barriers
};

__device__ __forceinline__ void issue_tile(const TilePipe& tp, int stage, const float* __restrict__ x,
                                           int64_t n, int d, int tile, int64_t tile_idx) {
  // called by thread 0 only
  int64_t first = tile_idx * tile;
  int64_t rows = n - first;
  if (rows > tile) rows = tile;
  uint32_t bytes = (uint32_t)(rows * d * 4);
  uint32_t bulk = bytes & ~15u;
  const float* src = x + first * d;
  // ragged tail (< 16 B): plain stores, ordered before the arrive below
  for (uint32_t i = bulk / 4; i < bytes / 4; ++i) tp.buf[stage][i] = src[i];
  mbar_expect_tx(&tp.bar[stage], bulk);
  if (bulk) tma_load_1d(tp.buf[stage], src, bulk, &tp.bar[stage]);
}

template <int D>
__device__ __forceinline__ float project_row(const float* __restrict__ xr, const float (&w)[kMaxDim], int d) {
  float u = 0.f;
  if (D > 0) {
#pragma unroll
    for (int i = 0; i < D; ++i) u = fmaf(w[i], xr[i], u);
  } else {
    for (int i = 0; i < d; ++i) u = fmaf(w[i], xr[i], u);
  }
  return u;
}

// ---- forward: KDE deposit --------------------------------------------------------------------
// Launch plan of the deposit kernel: up to 512 threads (= projections x particle slices) per CTA,
// one private column of B + 2G bins per thread (G = 2R+2 guard rows on either side, so that no tap
// needs a bounds check: particles beyond the screen are clamped to a position whose whole window
// lies in the guard rows).
constexpr int kDepThreads = 512;
struct KdePlan {
  int kc, slices, threads, ld, kchunks, grid_x, tile, rows, guard;   // ld = row stride of the bins (threads rounded up to 32)
  size_t smem;
};
static KdePlan plan_kde(int64_t n, int d, int k, int b, int r) {
  KdePlan P;
  P.guard = 2 * r + 2;                    // even, so that rows pair up as (2i, 2i+1) from row 0
  P.rows = (b + 2 * P.guard + 1) & ~1;
  P.kchunks = (k + kDepThreads - 1) / kDepThreads;
  P.kc = (k + P.kchunks - 1) / P.kchunks;
  int sms = sm_count();
  int tile = 512;
  while (tile > 128 && ceil_div64(n, tile) < 2 * sms) tile >>= 1;
  P.tile = tile;
  const size_t budget = 222 * 1024;
  int slices = kDepThreads / P.kc;
  while (slices > 1 && (size_t)P.rows * ((slices * P.kc + 31) & ~31) * 4 + 2ull * tile * d * 4 + 64 > budget) --slices;
  if (slices < 1) slices = 1;
  P.slices = slices;
  P.threads = slices * P.kc;
  P.ld = (P.threads + 31) & ~31;   // bank = thread % 32 whatever bin a lane hits: conflict free
  P.smem = (size_t)P.rows * P.ld * 4 + 2ull * tile * d * 4 + 64;
  int ctas_per_sm = (int)((226 * 1024) / (P.smem + 1024));
  if (ctas_per_sm < 1) ctas_per_sm = 1;
  if (ctas_per_sm * P.threads > 1024) ctas_per_sm = 1024 / P.threads > 0 ? 1024 / P.threads : 1;
  int64_t gx = (int64_t)sms * ctas_per_sm;
  const int64_t tiles = ceil_div64(n, tile);
  if (gx > tiles) gx = tiles;
  if (gx < 1) gx = 1;
  P.grid_x = (int)gx;
  return P;
}

// two fp32 products for one issue slot (Blackwell FMUL2; lanes are IEEE round-to-nearest like the scalar multiply)
__device__ __forceinline__ void mul_pair(float a0, float a1, float b0, float b1, float& c0, float& c1) {
  unsigned long long a, b, c;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(c) : "l"(a), "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(c0), "=f"(c1) : "l"(c));
}

// Gaussian taps of one particle for a window ALIGNED to row pairs: 2R+2 slots starting at an even row, slot i at offset
// o_i = i - (R + 1/2) from the window's centre, t in [-1, 1] = particle position relative to that centre:
//   tap[i] = 2^(alpha (t - o_i)^2),  alpha = -log2(e) / (2 (sigma / delta)^2) < 0.
// The two centre taps (o = -1/2, +1/2) are evaluated directly; one slot further out multiplies by the ratio
//   up (slot R+1+j from R+j):     2^(alpha (2j - 2t)) = su * rr[j-2],
//   down (slot R-j from R-j+1):   2^(alpha (2j + 2t)) = sd * rr[j-2],
// with su = 2^(alpha (2 - 2t)), sd = 2^(alpha (2 + 2t)) and rr[i] = 2^(2 alpha (i + 1)) per projection.  Every factor is
// <= 1, so no intermediate overflows however narrow the kernel is; a tap below the fp32 range underflows to zero, which is
// its correctly rounded value.  Four MUFU instead of 2R+2.  The nine taps of the unaligned window [fb-R, fb+R] are all
// inside (plus one more, 1e-18 of the centre) and land in their pair slots without shift-by-parity selects.
template <int R>
__device__ __forceinline__ void gauss_taps_pairs(float t, float alpha, const float (&rr)[R - 1], float (&tap)[2 * R + 2]) {
  static_assert(R >= 2, "window radius");
  float qu, qd;
  mul_pair(t - 0.5f, t + 0.5f, t - 0.5f, t + 0.5f, qu, qd);
  mul_pair(qu, qd, alpha, alpha, qu, qd);
  float up = fast_exp2(qu), dn = fast_exp2(qd);
  const float a2 = 2.0f * alpha;
  const float su = fast_exp2(fmaf(-a2, t, a2)), sd = fast_exp2(fmaf(a2, t, a2));
  tap[R + 1] = up;
  tap[R] = dn;
  mul_pair(up, dn, su, sd, up, dn);
  tap[R + 2] = up;
  tap[R - 1] = dn;
#pragma unroll
  for (int j = 2; j <= R; ++j) {
    float ru, rd;
    mul_pair(su, sd, rr[j - 2], rr[j - 2], ru, rd);
    mul_pair(up, dn, ru, rd, up, dn);
    tap[R + 1 + j] = up;
    tap[R - j] = dn;
  }
}

// particle row of an even-dimensional tile from shared memory with 8-byte loads (a generic pointer into the
// staging buffers compiles to six generic 4-byte loads per row)
template <int D>
__device__ __forceinline__ void load_row_shared(uint32_t saddr, float (&xr)[kMaxDim]) {
  static_assert(D % 2 == 0 && D >= 2, "even dimension");
#pragma unroll
  for (int i = 0; i < D; i += 2)
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(xr[i]), "=f"(xr[i + 1]) : "r"(saddr + 4u * i));
}

template <int D, int R, bool kMP = false>
__global__ void __launch_bounds__(kDepThreads)
kde1d_deposit_kernel(const float* __restrict__ x, int64_t n, int d_rt, const float* __restrict__ proj,
                     const float* __restrict__ geom, int K, int B, int kc, int tile, int guard, int ld,
                     float* __restrict__ partial /* [gridDim.x][K][B] */, const float* __restrict__ mp = nullptr) {
  const int d = D > 0 ? D : d_rt;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  TilePipe tp;
  tp.buf[0] = reinterpret_cast<float*>(smem_raw);
  tp.buf[1] = tp.buf[0] + (size_t)tile * d;
  tp.bar = reinterpret_cast<uint64_t*>(tp.buf[1] + (size_t)tile * d);
  float* bins = reinterpret_cast<float*>(tp.bar + 8);

  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int rows_total = (B + 2 * guard + 1) & ~1;
  const int kbase = blockIdx.y * kc;
  const int kloc = tid % kc;
  const int slice = tid / kc;
  const int slices = nthreads / kc;
  const int k = kbase + kloc;
  const bool active = k < K;

  for (int i = tid; i < rows_total * ld; i += nthreads) bins[i] = 0.f;
  if (tid == 0) {
    mbar_init(&tp.bar[0], 1);
    mbar_init(&tp.bar[1], 1);
    fence_mbar_init();
  }
  pdl_enter();   // the 170 KB of private bins were cleared under the previous kernel's tail; global memory from here on
  __syncthreads();

  float w[kMaxDim];
  float c0s = 0.f, inv_delta = 0.f, alpha = 0.f;
  float rr[R - 1];
#pragma unroll
  for (int j = 0; j < R - 1; ++j) rr[j] = 0.f;
  if (active) {
#pragma unroll
    for (int i = 0; i < kMaxDim; ++i) w[i] = i < d ? proj[(size_t)k * d + i] : 0.f;
    const float* g = geom + (size_t)k * MFB_GEOM_STRIDE;
    inv_delta = 1.0f / g[1];
    c0s = g[0] * inv_delta;
    float r = g[1] / g[2];
    alpha = -0.5f * r * r * kLog2e;
#pragma unroll
    for (int j = 0; j < R - 1; ++j) rr[j] = exp2f(alpha * (float)(2 * j + 2));
  }
  MpTerms mpt;
  if constexpr (kMP) {
    if (active) load_mp(mpt, mp + (size_t)k * MFB_MP_STRIDE(d), d);
  }

  const int64_t ntiles = (n + tile - 1) / tile;
  if ((int64_t)blockIdx.x < ntiles && tid == 0) issue_tile(tp, 0, x, n, d, tile, blockIdx.x);
  // The column of a thread is stored as pairs of rows, float2 (row 2i, row 2i+1) at pair index i, in blocks of one
  // WARP: [warp][pair][lane].  A warp touches 256 contiguous bytes whatever pairs its lanes hit (conflict free), and
  // consecutive pairs of a thread are a compile-time 256 bytes apart, so the R+1 pairs of a window are immediate
  // offsets from ONE address, itself one multiply-add of the rounding constant's mantissa bits (see below).
  // 8-byte accesses halve the shared-memory INSTRUCTION count (the LSU pipe issues one per two cycles).
  const int npairs = rows_total >> 1;
  const uint32_t mybase = smem_u32(bins) + (uint32_t)(((tid >> 5) * npairs * 32 + (tid & 31)) * 8);
  const uint32_t cthread = mybase - 0x4B400000u * 256u;   // address = mantissa bits * 256 + cthread (mod 2^32)
  const float lo = -(float)(R + 1), hi = (float)(B + R);
  constexpr int kPairs = R + 1;
  const float centre = (float)guard - ((float)R + 0.5f);

  // kPer particles of this thread's slice from row p on: their taps are independent (ILP for the MUFU / FMA work),
  // only the deposits into the private bins are ordered.  No bounds checks: the callers pass rows that exist.
  auto deposit = [&](auto per, const float* xs, uint32_t xs_shared, int p, int stride) {
    constexpr int kPer = decltype(per)::value;
    float taps[kPer][2 * R + 2];
    uint32_t dst[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
      const int pq = p + q * stride;
      float u;
      if constexpr (kMP) {
        u = project_row_mp(xs + (size_t)pq * d, w, mpt, d);
      } else if constexpr (D > 0 && D % 2 == 0) {
        float xr[kMaxDim];
        load_row_shared<D>(xs_shared + (uint32_t)(pq * (D * 4)), xr);
        u = 0.f;
#pragma unroll
        for (int i = 0; i < D; ++i) u = fmaf(w[i], xr[i], u);     // ascending FMA chain from zero (= the reference's sgemm bits)
      } else {
        u = project_row<D>(xs + (size_t)pq * d, w, d);
      }
      const float a = fminf(fmaxf(fmaf(u, inv_delta, -c0s), lo), hi);   // beyond the screen (or NaN): guard rows
      // window of 2R+2 rows starting at the even row 2 fp that holds the taps fb-R .. fb+R; t = position of the
      // particle relative to the window's centre, |t| <= 1
      const float ar = a + centre;
      // round-to-nearest of ar / 2 through the 1.5 * 2^23 constant (0 <= ar / 2 < 2^22): the integer is in the low
      // mantissa bits, no FRND / F2I
      const float shifted = fmaf(0.5f, ar, 12582912.0f);
      const float fp = shifted - 12582912.0f;
      gauss_taps_pairs<R>(fmaf(-2.0f, fp, ar), alpha, rr, taps[q]);
      dst[q] = __float_as_uint(shifted) * 256u + cthread;
    }
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
#pragma unroll
      for (int j = 0; j < kPairs; ++j) {
        float vx, vy;
        asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(vx), "=f"(vy) : "r"(dst[q] + 256u * j));
        vx += taps[q][2 * j];
        vy += taps[q][2 * j + 1];
        asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(dst[q] + 256u * j), "f"(vx), "f"(vy) : "memory");
      }
    }
  };

  int it = 0;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
    const int stage = it & 1;
    const int64_t nxt = t + gridDim.x;
    if (nxt < ntiles && tid == 0) issue_tile(tp, stage ^ 1, x, n, d, tile, nxt);
    mbar_wait(&tp.bar[stage], (it >> 1) & 1);
    int64_t rows64 = n - t * tile;
    const int rows = rows64 > tile ? tile : (int)rows64;
    const float* xs = tp.buf[stage];
    const uint32_t xs_shared = smem_u32(xs);
    if (active) {
      int p = slice;
      for (; p + 3 * slices < rows; p += 4 * slices) deposit(std::integral_constant<int, 4>{}, xs, xs_shared, p, slices);
      for (; p < rows; p += slices) deposit(std::integral_constant<int, 1>{}, xs, xs_shared, p, slices);
    }
    __syncthreads();  // everyone is done with buf[stage] before it is refilled
  }

  // fixed-order merge of the private columns -> per-CTA partial
  float* out = partial + (size_t)blockIdx.x * K * B;
  for (int idx = tid; idx < kc * B; idx += nthreads) {
    const int kk = idx % kc, b = idx / kc;
    if (kbase + kk < K) {
      float s = 0.f;
      const int row = b + guard;
      for (int sl = 0; sl < slices; ++sl) {
        const int tt = sl * kc + kk;   // the thread that owns this column
        s += bins[((size_t)((tt >> 5) * npairs + (row >> 1)) * 32 + (tt & 31)) * 2 + (row & 1)];
      }
      out[(size_t)(kbase + kk) * B + b] = s;
    }
  }
}

// ---- merge, normalisation and KL, forward and backward: one CTA per projection ---------------
__device__ __forceinline__ float block_sum_256(float v, float* red) {
  // deterministic: warp shuffle tree, then thread 0 adds the 8 warp sums in order
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float t = 0.f;
  if (threadIdx.x == 0) {
    for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += red[i];
    red[32] = t;
  }
  __syncthreads();
  t = red[32];
  __syncthreads();
  return t;
}

// ---- fused tail of the forward pass: merge per-CTA partials, normalise, KL against the measurement ----
// One CTA per projection.  Replaces the merge, the normalisation of histogram.py:39-43 and the ~8
// elementwise/reduce kernels of loss.py:15-17 evaluated on (K, B) tensors.  Sum order is fixed
// (partials c = g, g+G, ... per group g, groups combined in order), so the result is run-to-run deterministic.
constexpr int kFinishThreads = 256;

__device__ __forceinline__ void merge_partials_to_smem(const float* __restrict__ partial, int nparts, int64_t len,
                                                       int k, int B, float* __restrict__ part /*[G][B]*/,
                                                       float* __restrict__ s /*[B]*/) {
  const int tid = threadIdx.x;
  const int lanes = B < kFinishThreads ? B : kFinishThreads;
  const int G = kFinishThreads / lanes;
  const int g = tid / lanes, l = tid % lanes;
  if (g < G) {
    for (int b = l; b < B; b += lanes) {
      const float* src = partial + (size_t)k * B + b;
      float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
      int c = g;
      for (; c + 3 * G < nparts; c += 4 * G) {
        a0 += src[(size_t)c * len];
        a1 += src[(size_t)(c + G) * len];
        a2 += src[(size_t)(c + 2 * G) * len];
        a3 += src[(size_t)(c + 3 * G) * len];
      }
      for (; c < nparts; c += G) a0 += src[(size_t)c * len];
      part[(size_t)g * B + b] = (a0 + a1) + (a2 + a3);
    }
  }
  __syncthreads();
  for (int b = tid; b < B; b += kFinishThreads) {
    float t = 0.f;
    for (int gg = 0; gg < G; ++gg) t += part[(size_t)gg * B + b];
    s[b] = t;
  }
  __syncthreads();
}

// xlogy(t, t) - t log(p + pad): the summand of F.kl_div(log(p + pad), t) with 0 log 0 = 0
__device__ __forceinline__ float kl_term(float t, float p, float pad) {
  const float tl = t == 0.f ? 0.f : t * logf(t);
  return tl - t * logf(p + pad);
}

__global__ void __launch_bounds__(kFinishThreads)
kde1d_finish_kernel(const float* __restrict__ partial, int nparts, int64_t len, float inv_n,
                    const float* __restrict__ geom, int B, const float* __restrict__ meas, float pad,
                    float* __restrict__ sums_out, float* __restrict__ prof, float* __restrict__ kl) {
  extern __shared__ float fsm[];
  __shared__ float red[33];
  pdl_enter();
  const int k = blockIdx.x;
  float* s = fsm;
  float* part = fsm + B;
  merge_partials_to_smem(partial, nparts, len, k, B, part, s);
  const float delta = geom[(size_t)k * MFB_GEOM_STRIDE + 3];  // the reference's c[1]-c[0]
  float acc = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float v = s[b];
    if (sums_out) sums_out[(size_t)k * B + b] = v;
    acc += v * inv_n * delta;
  }
  const float z = block_sum_256(acc, red) + 1.0e-10f;
  if (prof == nullptr) return;   // merge only (the all-reduce across ranks comes next)
  float term = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float p = s[b] * inv_n / z;
    prof[(size_t)k * B + b] = p;
    if (meas) term += kl_term(meas[(size_t)k * B + b], p, pad);
  }
  if (kl) {
    const float tot = block_sum_256(term, red);
    if (threadIdx.x == 0) kl[k] = tot / (float)B;
  }
}

// ---- the same tail with the cross-rank sum inside: all-reduce over NVLink peer memory + normalise + KL ------------
// Multi-GPU forward step (particles sharded over ranks, SURVEY.md 8e): the unnormalised sums S[K][B] of every
// rank (25.6 KB at K = 100, B = 64) have to be added before the non-linear tail.  Through NCCL that is a
// latency-bound collective of its own on the critical path (+40..70 us per step at 2..8 GPUs); here the ranks
// exchange the rows through peer-mapped ("symmetric") buffers inside the finish kernel:
//   1. CTA k copies row k of the local sums (CTA 0 also the double tail: the entropy's moment sums) into this
//      rank's symmetric buffer of the current parity; the last CTA to finish publishes the step's epoch in every
//      peer's signal row (st.release.sys after __threadfence_system);
//   2. every CTA waits until all ranks have published this epoch (ld.acquire.sys on the local signal row);
//   3. CTA k adds row k of ALL ranks' buffers in rank order (plain loads over NVLink, bypassing L1), so every
//      rank forms bit-identical sums, and carries on with the normalisation and the KL of kde1d_finish_kernel.
// Buffers are double-buffered by epoch parity: a rank publishes epoch e only after its finish kernel of epoch
// e-1 (which read the peers' buffers of parity (e-1)&1) is complete in stream order, so passing the barrier of
// epoch e means every peer is done with parity (e+1)&1 -- the one the next step overwrites.  The epoch lives in
// device memory and is advanced by the last CTA to leave, so a captured CUDA graph can be replayed as is.
constexpr int kMaxRanks = 8;
struct PeerSet {
  float* buf[kMaxRanks];        // base of every rank's symmetric block: [signals 32 x u32][parity 0][parity 1]
};
constexpr int kP2PSignalFloats = 32;

__device__ __forceinline__ void st_release_sys_u32(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float ld_peer_f32(const float* p) {
  float v;
  asm volatile("ld.relaxed.sys.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ double ld_peer_f64(const double* p) {
  double v;
  asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory");
  return v;
}

__global__ void __launch_bounds__(kFinishThreads)
kde1d_finish_p2p_kernel(const __grid_constant__ PeerSet peers, int rank, int world, uint32_t* __restrict__ state,
                        int64_t parity_floats /* floats per parity block (sums + tail, 8-byte multiple) */,
                        const float* __restrict__ local_sums /* [K][B], or the deposit's per-CTA partials */,
                        int nparts /* 0: local_sums is merged already */, const double* __restrict__ local_tail,
                        int tail_n, float inv_n, const float* __restrict__ geom, int K, int B,
                        const float* __restrict__ meas, float pad, float* __restrict__ sums_out,
                        float* __restrict__ prof, float* __restrict__ kl, double* __restrict__ tail_out) {
  extern __shared__ float fsm[];
  __shared__ float red[33];
  float* s = fsm;
  const int k = blockIdx.x, tid = threadIdx.x;
  if (nparts > 0) merge_partials_to_smem(local_sums, nparts, (int64_t)K * B, k, B, fsm + B, s);   // fixed order
  // state[0] = epoch of the last completed step, state[1] / state[2] = arrival counters of this launch
  const uint32_t epoch = state[0] + 1u;
  const int64_t off = kP2PSignalFloats + (int64_t)(epoch & 1u) * parity_floats;
  float* mine = peers.buf[rank] + off;
  for (int b = tid; b < B; b += kFinishThreads) mine[(size_t)k * B + b] = nparts > 0 ? s[b] : local_sums[(size_t)k * B + b];
  if (k == 0 && tid < tail_n) reinterpret_cast<double*>(mine + (size_t)K * B)[tid] = local_tail[tid];
  __threadfence_system();
  __syncthreads();
  if (tid == 0) {
    const unsigned int arrived = atomicAdd(&state[1], 1u);
    if (arrived == (unsigned int)K - 1u) {           // every row of this rank is in place: publish the epoch
      __threadfence_system();
      for (int r = 0; r < world; ++r) st_release_sys_u32(reinterpret_cast<uint32_t*>(peers.buf[r]) + rank, epoch);
    }
  }
  if (tid < world) {
    const uint32_t* sig = reinterpret_cast<const uint32_t*>(peers.buf[rank]) + tid;
    long long spins = 0;
    while ((int32_t)(ld_acquire_sys_u32(sig) - epoch) < 0) {
      if (++spins > (1ll << 28)) __trap();             // a peer never arrived: fail loudly instead of hanging
      __nanosleep(20);
    }
  }
  __syncthreads();
  // rank-ordered sum: bit-identical on every rank
  for (int b = tid; b < B; b += kFinishThreads) {
    float v = 0.f;
    for (int r = 0; r < world; ++r) v += ld_peer_f32(peers.buf[r] + off + (size_t)k * B + b);
    s[b] = v;
  }
  if (k == 0 && tid < tail_n) {
    double v = 0.0;
    for (int r = 0; r < world; ++r)
      v += ld_peer_f64(reinterpret_cast<const double*>(peers.buf[r] + off + (size_t)K * B) + tid);
    tail_out[tid] = v;
  }
  __syncthreads();
  const float delta = geom[(size_t)k * MFB_GEOM_STRIDE + 3];
  float acc = 0.f;
  for (int b = tid; b < B; b += kFinishThreads) {
    const float v = s[b];
    sums_out[(size_t)k * B + b] = v;
    acc += v * inv_n * delta;
  }
  const float z = block_sum_256(acc, red) + 1.0e-10f;
  float term = 0.f;
  for (int b = tid; b < B; b += kFinishThreads) {
    const float p = s[b] * inv_n / z;
    prof[(size_t)k * B + b] = p;
    if (meas) term += kl_term(meas[(size_t)k * B + b], p, pad);
  }
  if (kl) {
    const float tot = block_sum_256(term, red);
    if (tid == 0) kl[k] = tot / (float)B;
  }
  // the last CTA to leave closes the step
  __syncthreads();
  if (tid == 0) {
    const unsigned int left = atomicAdd(&state[2], 1u);
    if (left == (unsigned int)K - 1u) {
      state[1] = 0u;
      state[2] = 0u;
      __threadfence();
      state[0] = epoch;
    }
  }
}

// gradient of (profiles, KL) w.r.t. the unnormalised sums:  gp_b = gprof_b - gkl * t_b / (p_b + pad) / B,
// then the normalisation backward  gsums_b = (gp_b / z - delta sum_j gp_j p_j / z) / N
__global__ void __launch_bounds__(kFinishThreads)
kde1d_finish_bwd_kernel(const float* __restrict__ sums, float inv_n, const float* __restrict__ geom, int B,
                        const float* __restrict__ meas, float pad, const float* __restrict__ gprof,
                        const float* __restrict__ gkl, float* __restrict__ gsums) {
  __shared__ float red[33];
  const int k = blockIdx.x;
  const float delta = geom[(size_t)k * MFB_GEOM_STRIDE + 3];
  float acc = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) acc += sums[(size_t)k * B + b] * inv_n * delta;
  const float z = block_sum_256(acc, red) + 1.0e-10f;
  const float gk = gkl ? gkl[k] / (float)B : 0.f;
  float dot = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const size_t i = (size_t)k * B + b;
    const float p = sums[i] * inv_n / z;
    float gp = gprof ? gprof[i] : 0.f;
    if (gkl) gp -= gk * meas[i] / (p + pad);
    dot += gp * p;
  }
  const float g = block_sum_256(dot, red);
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const size_t i = (size_t)k * B + b;
    const float p = sums[i] * inv_n / z;
    float gp = gprof ? gprof[i] : 0.f;
    if (gkl) gp -= gk * meas[i] / (p + pad);
    gsums[i] = (gp / z - delta * g / z) * inv_n;
  }
}

static inline size_t finish_smem(int b) {
  const int lanes = b < kFinishThreads ? b : kFinishThreads;
  return ((size_t)b + (size_t)(kFinishThreads / lanes) * b) * 4;
}

// ---- backward w.r.t. the particles: thread per particle ---------------------------------------
template <int D, int R, bool kMP = false>
__global__ void __launch_bounds__(256)
kde1d_bwd_kernel(const float* __restrict__ x, int64_t n, int d_rt, const float* __restrict__ proj,
                 const float* __restrict__ geom, int K, int B, const float* __restrict__ gsums,
                 float* __restrict__ gx, int accumulate, const float* __restrict__ mp = nullptr) {
  const int d = D > 0 ? D : d_rt;
  extern __shared__ __align__(16) float sm[];
  // gradient table with kPad zero bins on either side of every row: the 2R+1 taps of a (clamped) particle never need a
  // bounds check
  constexpr int kPad = 2 * R + 2;
  const int BP = B + 2 * kPad;
  float* s_g = sm;                          // [K][BP]
  float* s_w = s_g + (((size_t)K * BP + 3) & ~(size_t)3);   // [K][d]; 16-byte aligned so that s_q is
  float4* s_q = reinterpret_cast<float4*>(s_w + (((size_t)K * d + 3) & ~(size_t)3));  // [K] c0, inv_delta, alpha, beta
  float* s_rr = reinterpret_cast<float*>(s_q + K);   // [K][R]: 2^(2 alpha j), steps of the tap ratios
  float* s_mp = s_rr + (size_t)K * R;                // [K][2d + 4] (multipole variant only)
  for (int i = threadIdx.x; i < K * BP; i += blockDim.x) {
    const int kk = i / BP, b = i % BP - kPad;
    s_g[i] = (b >= 0 && b < B) ? gsums[(size_t)kk * B + b] : 0.f;
  }
  for (int i = threadIdx.x; i < K * d; i += blockDim.x) s_w[i] = proj[i];
  if constexpr (kMP) {
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(d); i += blockDim.x) s_mp[i] = mp[i];
  }
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    const float* g = geom + (size_t)k * MFB_GEOM_STRIDE;
    const float r = g[1] / g[2];
    const float alpha = -0.5f * r * r * kLog2e;
    s_q[k] = make_float4(g[0], 1.0f / g[1], alpha, -g[1] / (g[2] * g[2]));
    for (int j = 0; j < R; ++j) s_rr[(size_t)k * R + j] = exp2f(alpha * (float)(2 * j));
  }
  __syncthreads();
  const float lo = -(float)(R + 2), hi = (float)(B + R + 1);
  for (int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
    float xr[kMaxDim], g[kMaxDim];
#pragma unroll
    for (int i = 0; i < kMaxDim; ++i) {
      xr[i] = (i < d) ? x[p * d + i] : 0.f;
      g[i] = 0.f;
    }
    for (int k = 0; k < K; ++k) {
      const float* wk = s_w + (size_t)k * d;
      float u = 0.f;
#pragma unroll
      for (int i = 0; i < kMaxDim; ++i)
        if (i < d) u = fmaf(wk[i], xr[i], u);
      float cx = 0.f, cy = 0.f;   // du/d(xm), du/d(ym) of the multipole terms
      if constexpr (kMP) {
        const float* mk = s_mp + (size_t)k * MFB_MP_STRIDE(d);
        float xm = 0.f, ym = 0.f;
#pragma unroll
        for (int i = 0; i < kMaxDim; ++i)
          if (i < d) {
            xm = fmaf(mk[i], xr[i], xm);
            ym = fmaf(mk[d + i], xr[i], ym);
          }
        const float a = mk[2 * d], bq = mk[2 * d + 1];
        const int m = (int)mk[2 * d + 2] - 1;
        float zr, zi, pr, pi;
        zpow(xm, ym, m, zr, zi, pr, pi);
        u = fmaf(bq, zi, fmaf(a, zr, u));
        // d z^m / d xm = m z^(m-1),  d z^m / d ym = i m z^(m-1)
        cx = (float)m * (a * pr + bq * pi);
        cy = (float)m * (bq * pr - a * pi);
      }
      const float4 q = s_q[k];
      float a = (u - q.x) * q.y;
      a = fminf(fmaxf(a, lo), hi);
      // nearest bin through the 1.5 * 2^23 rounding constant (no FRND / F2I), taps by recurrences as in the forward
      // kernel: the value at offset 0 is 2^(alpha f^2), the ratio from offset j to j+1 is 2^(alpha (2j + 1 - 2f)) =
      // su rr[j] (up) and from -j to -(j+1) 2^(alpha (2j + 1 + 2f)) = sd rr[j] (down), su = 2^(alpha (1 - 2f)),
      // sd = 2^(alpha (1 + 2f)).  |f| <= 1/2 keeps every factor <= 1 (no overflow at any bandwidth); three MUFU per
      // particle-projection instead of 2R+1, the up / down recurrences as packed multiplies
      const float shifted = a + 12582912.0f;
      const float fb = shifted - 12582912.0f;
      const float f = a - fb;
      const float* grow = s_g + (size_t)k * BP + ((__float_as_int(shifted) - 0x4B400000) + kPad);
      const float af = q.z * f;
      const float e0 = fast_exp2(af * f);
      const float su = fast_exp2(fmaf(-2.0f, af, q.z)), sd = fast_exp2(fmaf(2.0f, af, q.z));
      const float* rr = s_rr + (size_t)k * R;
      float acc = grow[0] * (e0 * f);
      float up = e0, dn = e0;
#pragma unroll
      for (int j = 0; j < R; ++j) {
        float ru = su, rd = sd;
        if (j > 0) mul_pair(su, sd, rr[j], rr[j], ru, rd);
        mul_pair(up, dn, ru, rd, up, dn);
        float wu, wd;
        mul_pair(up, dn, f - (float)(j + 1), f + (float)(j + 1), wu, wd);
        acc = fmaf(grow[j + 1], wu, acc);
        acc = fmaf(grow[-(j + 1)], wd, acc);
      }
      const float gu = q.w * acc;
#pragma unroll
      for (int i = 0; i < kMaxDim; ++i)
        if (i < d) {
          float wi = wk[i];
          if constexpr (kMP) {
            const float* mk = s_mp + (size_t)k * MFB_MP_STRIDE(d);
            wi = fmaf(cx, mk[i], fmaf(cy, mk[d + i], wi));
          }
          g[i] = fmaf(wi, gu, g[i]);
        }
    }
#pragma unroll
    for (int i = 0; i < kMaxDim; ++i)
      if (i < d) {
        if (accumulate) gx[p * d + i] += g[i];
        else gx[p * d + i] = g[i];
      }
  }
}

// ---- exact histogram deposit ----------------------------------------------------------------------
template <int D, bool kMP = false>
__global__ void __launch_bounds__(kBinThreads)
hist1d_deposit_kernel(const float* __restrict__ x, int64_t n, int d_rt, const float* __restrict__ proj,
                      const float* __restrict__ edges, int K, int B, int kc, int tile,
                      unsigned long long* __restrict__ counts /* [K][B] */, const float* __restrict__ mp = nullptr) {
  const int d = D > 0 ? D : d_rt;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  TilePipe tp;
  tp.buf[0] = reinterpret_cast<float*>(smem_raw);
  tp.buf[1] = tp.buf[0] + (size_t)tile * d;
  tp.bar = reinterpret_cast<uint64_t*>(tp.buf[1] + (size_t)tile * d);
  unsigned int* bins = reinterpret_cast<unsigned int*>(tp.bar + 8);

  const int tid = threadIdx.x, nthreads = blockDim.x;
  const int ld = (nthreads + 31) & ~31;   // row stride of the private bins: conflict free for any bin pattern
  float* s_edges = reinterpret_cast<float*>(bins + (size_t)B * ld);  // [kc][B+1]
  const int kbase = blockIdx.y * kc;
  const int kloc = tid % kc;
  const int slice = tid / kc;
  const int slices = nthreads / kc;
  const int k = kbase + kloc;
  const bool active = k < K;

  for (int i = tid; i < B * ld; i += nthreads) bins[i] = 0u;
  for (int i = tid; i < kc * (B + 1); i += nthreads) {
    const int kk = kbase + i / (B + 1);
    s_edges[i] = kk < K ? edges[(size_t)kk * (B + 1) + i % (B + 1)] : 0.f;
  }
  if (tid == 0) {
    mbar_init(&tp.bar[0], 1);
    mbar_init(&tp.bar[1], 1);
    fence_mbar_init();
  }
  __syncthreads();

  float w[kMaxDim];
  const float* E = s_edges + (size_t)kloc * (B + 1);
  float e0 = 0.f, eB = 0.f, inv_w = 0.f;
  if (active) {
#pragma unroll
    for (int i = 0; i < kMaxDim; ++i) w[i] = i < d ? proj[(size_t)k * d + i] : 0.f;
    e0 = E[0];
    eB = E[B];
    inv_w = (float)B / (eB - e0);
  }
  MpTerms mpt;
  if constexpr (kMP) {
    if (active) load_mp(mpt, mp + (size_t)k * MFB_MP_STRIDE(d), d);
  }

  const int64_t ntiles = (n + tile - 1) / tile;
  if ((int64_t)blockIdx.x < ntiles && tid == 0) issue_tile(tp, 0, x, n, d, tile, blockIdx.x);
  unsigned int* mybins = bins + tid;

  int it = 0;
  for (int64_t t = blockIdx.x; t < ntiles; t += gridDim.x, ++it) {
    const int stage = it & 1;
    const int64_t nxt = t + gridDim.x;
    if (nxt < ntiles && tid == 0) issue_tile(tp, stage ^ 1, x, n, d, tile, nxt);
    mbar_wait(&tp.bar[stage], (it >> 1) & 1);
    int64_t rows64 = n - t * tile;
    const int rows = rows64 > tile ? tile : (int)rows64;
    const float* xs = tp.buf[stage];
    if (active) {
      for (int p = slice; p < rows; p += slices) {
        float u;
        if constexpr (kMP) u = project_row_mp(xs + (size_t)p * d, w, mpt, d);
        else u = project_row<D>(xs + (size_t)p * d, w, d);
        if (u >= e0 && u <= eB) {  // NaN fails both
          int b = (int)((u - e0) * inv_w);
          b = min(max(b, 0), B - 1);
          while (b > 0 && u < E[b]) --b;
          while (b < B - 1 && u >= E[b + 1]) ++b;
          mybins[(size_t)b * ld] += 1u;
        }
      }
    }
    __syncthreads();
  }

  for (int idx = tid; idx < kc * B; idx += nthreads) {
    const int kk = idx % kc, b = idx / kc;
    if (kbase + kk < K) {
      unsigned long long s = 0ull;
      for (int sl = 0; sl < slices; ++sl) s += bins[(size_t)b * ld + sl * kc + kk];
      if (s) atomicAdd(&counts[(size_t)(kbase + kk) * B + b], s);
    }
  }
}

// ---- host-side dispatch -----------------------------------------------------------------------------
template <int D, bool kMP = false>
static int launch_kde1d_deposit(int r, const KdePlan& L, const float* x, int64_t n, int d, const float* proj,
                                const float* geom, int k, int b, float* partial, cudaStream_t st,
                                const float* mp = nullptr) {
  dim3 grid(L.grid_x, L.kchunks), block(L.threads);
#define MFB_LAUNCH_R(RR)                                                                                   \
  {                                                                                                        \
    MFB_CUDA(cudaFuncSetAttribute(kde1d_deposit_kernel<D, RR, kMP>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                  (int)L.smem));                                                           \
    MFB_CUDA(launch_pdl(kde1d_deposit_kernel<D, RR, kMP>, grid, block, L.smem, st, x, n, d, proj, geom, k, b, L.kc, L.tile, L.guard, L.ld, partial, mp)); \
  }
  if (r <= 4) MFB_LAUNCH_R(4)
  else if (r <= 9) MFB_LAUNCH_R(9)
  else if (r <= 13) MFB_LAUNCH_R(13)
  else return MFB_E_UNSUPPORTED;
#undef MFB_LAUNCH_R
  return launch_status();
}

template <int D, bool kMP = false>
static int launch_kde1d_bwd(int r, int grid, size_t smem, const float* x, int64_t n, int d, const float* proj,
                            const float* geom, int k, int b, const float* gsums, float* gx, int acc,
                            cudaStream_t st, const float* mp = nullptr) {
#define MFB_LAUNCH_R(RR)                                                                                \
  {                                                                                                     \
    MFB_CUDA(cudaFuncSetAttribute(kde1d_bwd_kernel<D, RR, kMP>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                  (int)smem));                                                          \
    kde1d_bwd_kernel<D, RR, kMP><<<grid, 256, smem, st>>>(x, n, d, proj, geom, k, b, gsums, gx, acc, mp);    \
  }
  if (r <= 4) MFB_LAUNCH_R(4)
  else if (r <= 9) MFB_LAUNCH_R(9)
  else if (r <= 13) MFB_LAUNCH_R(13)
  else return MFB_E_UNSUPPORTED;
#undef MFB_LAUNCH_R
  return launch_status();
}

}  // namespace mfb

using namespace mfb;

// The window radius must be known on the host while geom lives on the device, so the caller
// passes the largest sigma/delta ratio of the launch (<= 0 means the default bandwidth 0.5).
static int radius_from_hint(float hint) { return window_radius(hint > 0.f ? hint : 0.5); }

// the window radius of the kernel template that serves radius r (launches refuse r > 13)
static int compiled_radius(int r) { return r <= 4 ? 4 : (r <= 9 ? 9 : 13); }

// deposit of all projections (n >= 1) into the per-CTA partials [nparts][k][b] in the workspace; mp != nullptr
// selects the multipole variant (runtime dimension: the non-linear configurations are low-dimensional)
static int kde1d_deposit(const float* x, int64_t n, int d, const float* proj, const float* mp, const float* geom,
                         int k, int b, float max_sigma_over_delta, void* workspace, int64_t workspace_bytes,
                         cudaStream_t st, int* nparts) {
  const int r = radius_from_hint(max_sigma_over_delta);
  KdePlan L = plan_kde(n, d, k, b, compiled_radius(r));
  if (L.smem > 227 * 1024) return MFB_E_UNSUPPORTED;
  if (workspace_bytes < (int64_t)L.grid_x * k * b * 4) return MFB_E_WORKSPACE;
  *nparts = L.grid_x;
  float* partial = (float*)workspace;
  if (mp) return launch_kde1d_deposit<0, true>(r, L, x, n, d, proj, geom, k, b, partial, st, mp);
  switch (d) {
    case 2: return launch_kde1d_deposit<2>(r, L, x, n, d, proj, geom, k, b, partial, st);
    case 4: return launch_kde1d_deposit<4>(r, L, x, n, d, proj, geom, k, b, partial, st);
    case 6: return launch_kde1d_deposit<6>(r, L, x, n, d, proj, geom, k, b, partial, st);
    default: return launch_kde1d_deposit<0>(r, L, x, n, d, proj, geom, k, b, partial, st);
  }
}

extern "C" {

int64_t mfb_kde1d_workspace_bytes(int64_t n, int d, int k, int b) {
  if (n < 0 || d < 1 || d > kMaxDim || k < 1 || b < 1) return 0;
  // upper bound over every deposit plan (the window radius is not known here)
  const int64_t tiles = ceil_div64(n > 0 ? n : 1, 128);
  int64_t gx = (int64_t)sm_count() * 4;
  if (gx > tiles) gx = tiles;
  return gx * k * b * 4;
}

int mfb_project_kde1d_fwd(const float* x, int64_t n, int d, const float* proj, const float* mp, const float* geom,
                          int k, int b, float max_sigma_over_delta, double n_total, const float* meas, float pad,
                          float* sums, float* profiles, float* kl, void* workspace, int64_t workspace_bytes,
                          void* stream) {
  MFB_CHECK_ARG(x && proj && geom && sums && workspace);
  MFB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim && k >= 1 && b >= 2);
  MFB_CHECK_ARG((meas != nullptr) == (kl != nullptr));
  MFB_CHECK_ARG(profiles ? n >= 1 && n_total > 0 : meas == nullptr);
  cudaStream_t st = (cudaStream_t)stream;
  if (n == 0) return (int)cudaMemsetAsync(sums, 0, (size_t)k * b * 4, st);
  if (finish_smem(b) > 48 * 1024) return MFB_E_UNSUPPORTED;
  int nparts = 0;
  int rc = kde1d_deposit(x, n, d, proj, mp, geom, k, b, max_sigma_over_delta, workspace, workspace_bytes, st, &nparts);
  if (rc) return rc;
  const float inv_n = profiles ? (float)(1.0 / n_total) : 1.f;   // without profiles the kernel stops after the merge
  MFB_CUDA(launch_pdl(kde1d_finish_kernel, dim3(k), dim3(kFinishThreads), finish_smem(b), st, workspace, nparts,
                      (int64_t)k * b, inv_n, geom, b, meas, pad, sums, profiles, kl));
  return launch_status();
}

int64_t mfb_kde1d_p2p_block_floats(int k, int b, int tail_doubles) {
  if (k < 1 || b < 2 || tail_doubles < 0) return 0;
  const int64_t parity = (((int64_t)k * b + 1) & ~(int64_t)1) + 2 * (int64_t)tail_doubles;
  return kP2PSignalFloats + 2 * parity;
}

int mfb_kde1d_finish_p2p(const uint64_t* peer_blocks_host, int rank, int world, uint32_t* state,
                         const float* local_sums, const double* local_tail, int tail_doubles, double n_total,
                         const float* geom, int k, int b, const float* meas, float pad, float* sums, float* profiles,
                         float* kl, double* tail_out, void* stream) {
  MFB_CHECK_ARG(peer_blocks_host && state && local_sums && geom && sums && profiles && k >= 1 && b >= 2 && n_total > 0);
  MFB_CHECK_ARG(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world);
  MFB_CHECK_ARG((meas != nullptr) == (kl != nullptr));
  MFB_CHECK_ARG(tail_doubles >= 0 && tail_doubles <= 32 && (tail_doubles == 0 || (local_tail && tail_out)));
  MFB_CHECK_ARG(((int64_t)k * b) % 2 == 0);           // keeps the double tail 8-byte aligned
  if (k > 1024 || (size_t)b * 4 > 48 * 1024) return MFB_E_UNSUPPORTED;   // every CTA of the grid must be resident
  PeerSet ps;
  for (int r = 0; r < kMaxRanks; ++r) ps.buf[r] = r < world ? reinterpret_cast<float*>(peer_blocks_host[r]) : nullptr;
  const int64_t parity = (int64_t)k * b + 2 * (int64_t)tail_doubles;
  kde1d_finish_p2p_kernel<<<k, kFinishThreads, (size_t)b * 4, (cudaStream_t)stream>>>(
      ps, rank, world, state, parity, local_sums, 0, local_tail, tail_doubles, (float)(1.0 / n_total), geom, k, b, meas,
      pad, sums, profiles, kl, tail_out);
  return launch_status();
}

/* deposit + (merge, cross-rank sum, normalise, KL) in two launches: the sharded counterpart of
 * mfb_project_kde1d_fwd with profiles */
int mfb_project_kde1d_loss_fwd_p2p(const float* x, int64_t n, int d, const float* proj, const float* geom, int k, int b,
                                   float max_sigma_over_delta, double n_total, const float* meas, float pad,
                                   const uint64_t* peer_blocks_host, int rank, int world, uint32_t* state,
                                   const double* local_tail, int tail_doubles, float* sums, float* profiles, float* kl,
                                   double* tail_out, void* workspace, int64_t workspace_bytes, void* stream) {
  MFB_CHECK_ARG(x && proj && geom && sums && profiles && workspace && peer_blocks_host && state);
  MFB_CHECK_ARG((meas != nullptr) == (kl != nullptr));
  MFB_CHECK_ARG(n >= 1 && d >= 1 && d <= kMaxDim && k >= 1 && b >= 2 && n_total > 0);
  MFB_CHECK_ARG(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world && ((int64_t)k * b) % 2 == 0);
  MFB_CHECK_ARG(tail_doubles >= 0 && tail_doubles <= 32 && (tail_doubles == 0 || (local_tail && tail_out)));
  if (finish_smem(b) > 48 * 1024 || k > 1024) return MFB_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  int nparts = 0;
  int rc = kde1d_deposit(x, n, d, proj, nullptr, geom, k, b, max_sigma_over_delta, workspace, workspace_bytes, st,
                         &nparts);
  if (rc) return rc;
  PeerSet ps;
  for (int i = 0; i < kMaxRanks; ++i) ps.buf[i] = i < world ? reinterpret_cast<float*>(peer_blocks_host[i]) : nullptr;
  const int64_t parity = (int64_t)k * b + 2 * (int64_t)tail_doubles;
  kde1d_finish_p2p_kernel<<<k, kFinishThreads, finish_smem(b), st>>>(
      ps, rank, world, state, parity, (const float*)workspace, nparts, local_tail, tail_doubles,
      (float)(1.0 / n_total), geom, k, b, meas, pad, sums, profiles, kl, tail_out);
  return launch_status();
}

int mfb_kde1d_finish(const float* sums, double n_total, const float* geom, int k, int b, const float* meas,
                     float pad, float* profiles, float* kl, void* stream) {
  MFB_CHECK_ARG(sums && geom && profiles && k >= 1 && b >= 2 && n_total > 0);
  MFB_CHECK_ARG((meas != nullptr) == (kl != nullptr));
  if (finish_smem(b) > 48 * 1024) return MFB_E_UNSUPPORTED;
  MFB_CUDA(launch_pdl(kde1d_finish_kernel, dim3(k), dim3(kFinishThreads), finish_smem(b), (cudaStream_t)stream, sums, 1, (int64_t)k * b, (float)(1.0 / n_total), geom, b, meas, pad, nullptr, profiles, kl));
  return launch_status();
}

int mfb_kde1d_finish_bwd(const float* sums, double n_total, const float* geom, int k, int b, const float* meas,
                         float pad, const float* gprof, const float* gkl, float* gsums, void* stream) {
  MFB_CHECK_ARG(sums && geom && gsums && k >= 1 && b >= 2 && n_total > 0);
  MFB_CHECK_ARG(gprof || gkl);
  MFB_CHECK_ARG(!gkl || meas);
  kde1d_finish_bwd_kernel<<<k, kFinishThreads, 0, (cudaStream_t)stream>>>(sums, (float)(1.0 / n_total), geom, b, meas,
                                                                          pad, gprof, gkl, gsums);
  return launch_status();
}

int mfb_project_kde1d_bwd(const float* x, int64_t n, int d, const float* proj, const float* mp, const float* geom,
                          int k, int b, float max_sigma_over_delta, const float* gsums, float* gx, int accumulate,
                          void* stream) {
  MFB_CHECK_ARG(x && proj && geom && gsums && gx);
  MFB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim && k >= 1 && b >= 2);
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int r = radius_from_hint(max_sigma_over_delta);
  // projections are processed in chunks whose gradient table fits in shared memory
  const int rt = compiled_radius(r);
  const size_t bp = (size_t)b + 2 * (2 * rt + 2);                       // padded gradient row
  const size_t per_k = bp * 4 + (size_t)d * 4 + 16 + (size_t)rt * 4 + (mp ? (size_t)MFB_MP_STRIDE(d) * 4 : 0);
  int kchunk = (int)((160 * 1024) / per_k);
  if (kchunk < 1) return MFB_E_UNSUPPORTED;
  if (kchunk > k) kchunk = k;
  const int sms = sm_count();
  int64_t blocks = (n + 255) / 256;
  for (int k0 = 0; k0 < k; k0 += kchunk) {
    const int kk = (k - k0 < kchunk) ? (k - k0) : kchunk;
    const size_t smem = (((size_t)kk * bp + 3) & ~(size_t)3) * 4 + (((size_t)kk * d + 3) & ~(size_t)3) * 4 + (size_t)kk * 16 + 16 +
                        (size_t)kk * rt * 4 + (mp ? (size_t)kk * MFB_MP_STRIDE(d) * 4 : 0);
    int per_sm = (int)((200 * 1024) / (smem + 1024));
    if (per_sm < 1) per_sm = 1;
    if (per_sm > 8) per_sm = 8;
    int64_t grid = (int64_t)sms * per_sm;
    if (grid > blocks) grid = blocks;
    const int acc = (accumulate || k0 > 0) ? 1 : 0;
    int rc;
    const float* pj = proj + (size_t)k0 * d;
    const float* gm = geom + (size_t)k0 * MFB_GEOM_STRIDE;
    const float* gs = gsums + (size_t)k0 * b;
    if (mp) {
      rc = launch_kde1d_bwd<0, true>(r, (int)grid, smem, x, n, d, pj, gm, kk, b, gs, gx, acc, st,
                                     mp + (size_t)k0 * MFB_MP_STRIDE(d));
      if (rc) return rc;
      continue;
    }
    switch (d) {
      case 2: rc = launch_kde1d_bwd<2>(r, (int)grid, smem, x, n, d, pj, gm, kk, b, gs, gx, acc, st); break;
      case 4: rc = launch_kde1d_bwd<4>(r, (int)grid, smem, x, n, d, pj, gm, kk, b, gs, gx, acc, st); break;
      case 6: rc = launch_kde1d_bwd<6>(r, (int)grid, smem, x, n, d, pj, gm, kk, b, gs, gx, acc, st); break;
      default: rc = launch_kde1d_bwd<0>(r, (int)grid, smem, x, n, d, pj, gm, kk, b, gs, gx, acc, st); break;
    }
    if (rc) return rc;
  }
  return 0;
}

int mfb_project_hist1d(const float* x, int64_t n, int d, const float* proj, const float* mp, const float* edges, int k,
                       int b, int64_t* counts, void* stream) {
  MFB_CHECK_ARG(x && proj && edges && counts);
  MFB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim && k >= 1 && b >= 1);
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  // edges of the CTA's projections live in smem next to the private bins
  int kc_guess = k < kBinThreads ? k : kBinThreads;
  ProjLaunch L = plan_launch(n, d, k, b, 4, (size_t)kc_guess * (b + 1) * 4 + 16);
  if (L.smem > 227 * 1024) return MFB_E_UNSUPPORTED;
  dim3 grid(L.grid_x, L.kchunks), block(L.threads);
  unsigned long long* c = reinterpret_cast<unsigned long long*>(counts);
#define MFB_LAUNCH_D(DD)                                                                                  \
  {                                                                                                       \
    MFB_CUDA(cudaFuncSetAttribute(hist1d_deposit_kernel<DD>, cudaFuncAttributeMaxDynamicSharedMemorySize,  \
                                  (int)L.smem));                                                          \
    hist1d_deposit_kernel<DD><<<grid, block, L.smem, st>>>(x, n, d, proj, edges, k, b, L.kc, L.tile, c);   \
  }
  if (mp) {
    MFB_CUDA(cudaFuncSetAttribute(hist1d_deposit_kernel<0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)L.smem));
    hist1d_deposit_kernel<0, true><<<grid, block, L.smem, st>>>(x, n, d, proj, edges, k, b, L.kc, L.tile, c, mp);
    return launch_status();
  }
  switch (d) {
    case 2: MFB_LAUNCH_D(2) break;
    case 4: MFB_LAUNCH_D(4) break;
    case 6: MFB_LAUNCH_D(6) break;
    default: MFB_LAUNCH_D(0) break;
  }
#undef MFB_LAUNCH_D
  return launch_status();
}

}  // extern "C"
