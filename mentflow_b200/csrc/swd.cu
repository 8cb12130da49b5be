// Sliced p-Wasserstein distance (loss.py sliced_wasserstein_distance / SlicedWassersteinDistance): P projections
// u_k = x theta_k of the model samples, a stable sort of every projection, and the 1-D quantile integral
//   W_p^p(k) = int_0^1 |F_u^-1(q) - F_v^-1(q)|^p dq
// against the already sorted projections v_k of the reference set.
//
// Projections are fp32 fused multiply-add chains from zero in ascending coordinate order.  Each becomes an
// order-preserving uint32 key (-0 and +0 share a key, every NaN gets 0xffffffff and sorts last) and is sorted with
// its particle index by four stable 8-bit LSD digit passes; the segments are the directions.  Per chunk of directions:
//   1. swd_keys_kernel: a tile of rows is read once for a group of directions; keys of every (direction, particle)
//      pair, all four digit histograms of each direction (integer atomics), and the tile's digit counts of pass 0;
//   2. per pass q: swd_count_kernel (tile digit counts, q > 0), swd_scan_kernel (exclusive scan over
//      [direction][digit][tile], offset by the direction's histogram of the smaller digits: reduce-then-scan, no CTA
//      waits on another) and swd_scatter_kernel: each 2048-key tile is ranked in shared memory (warp match/ballot
//      ranks in index order, then a stable CTA-local reorder by digit) and written at its scanned offsets.  The index
//      payload of pass 0 is the position itself and is not read;
//   3. the last pass does not store keys.  swd_sort writes the sorted projections (recomputed from x, so -0.0 and NaN
//      payloads keep their bits) and the permutation.  swd_wpp instead lets every lane, which holds consecutive global
//      ranks i after the reorder, add rank i's share of W_p^p from the sorted v at ranks j(i) (coalesced reads), and
//      write dW_p^p/du at the particle's index when a gradient is wanted.  Per-CTA double partials are added per
//      direction in a fixed order by swd_reduce_kernel.
// Rank i of N covers [i/N, (i+1)/N), rank j of M covers [j/M, (j+1)/M); in units of 1/(N M) these are the integer
// intervals [i M, (i+1) M) and [j N, (j+1) N), so the overlaps are exact int64 and rank i reads j = floor(i M / N) ..
// floor(((i+1) M - 1) / N): at most M/N + 2 values.
// Backward (swd_bwd_kernel): gx[n] = sum_k gw[k] theta_k dW_p^p(k)/du_{k,n}, k ascending.  No floating-point atomics:
// every output is bitwise reproducible and independent of the chunking of the directions.
#include <math.h>

#include "common.cuh"

namespace mfb {

constexpr int kSwdThreads = 256;
constexpr int kSwdWarps = kSwdThreads / 32;
constexpr int kSwdItems = 8;
constexpr int kSwdTile = kSwdThreads * kSwdItems;   // keys per tile (a CTA of every pass)
constexpr int kSwdDigits = 256;
constexpr int kSwdMaxChunk = 65535;                 // directions per chunk: gridDim.y

enum { kSwdMid = 0, kSwdSorted = 1, kSwdWpp = 2 };

__device__ __forceinline__ uint32_t swd_key(float u) {
  if (u != u) return 0xffffffffu;
  uint32_t b = __float_as_uint(u);
  if (b == 0x80000000u) b = 0u;
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float swd_value(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

template <int D>
__device__ __forceinline__ float swd_project(const float* __restrict__ row, const float* __restrict__ th) {
  float u = 0.f;
#pragma unroll
  for (int c = 0; c < D; ++c) u = fmaf(row[c], th[c], u);
  return u;
}

__device__ __forceinline__ uint32_t lanemask_lt() {
  uint32_t m;
  asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
  return m;
}

// ---- 1. keys + histograms ---------------------------------------------------------------------------------------
// grid (ntiles, groups): CTA = one tile of rows x directions [y * per, (y + 1) * per).  The rows stay in registers
// across the group; groups exist only to fill the GPU when the tiles are few.
template <int D>
__global__ void __launch_bounds__(kSwdThreads)
swd_keys_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ theta, int nproj, int per,
                int ntiles, uint32_t* __restrict__ keys, uint32_t* __restrict__ tcount, uint32_t* __restrict__ hist) {
  __shared__ uint32_t h[4 * kSwdDigits];
  pdl_enter();
  const int tid = threadIdx.x, tile = blockIdx.x;
  const int64_t t0 = (int64_t)tile * kSwdTile;
  float xr[kSwdItems][D];
#pragma unroll
  for (int j = 0; j < kSwdItems; ++j) {
    const int64_t r = t0 + tid + j * kSwdThreads;
#pragma unroll
    for (int c = 0; c < D; ++c) xr[j][c] = r < n ? x[r * D + c] : 0.f;
  }
  const int k_end = min(nproj, (int)(blockIdx.y + 1) * per);
  for (int k = blockIdx.y * per; k < k_end; ++k) {
    for (int i = tid; i < 4 * kSwdDigits; i += kSwdThreads) h[i] = 0;
    __syncthreads();
    float th[D];
#pragma unroll
    for (int c = 0; c < D; ++c) th[c] = theta[k * D + c];
#pragma unroll
    for (int j = 0; j < kSwdItems; ++j) {
      const int64_t r = t0 + tid + j * kSwdThreads;
      if (r < n) {
        const uint32_t key = swd_key(swd_project<D>(xr[j], th));
        keys[(int64_t)k * n + r] = key;
#pragma unroll
        for (int q = 0; q < 4; ++q) atomicAdd(&h[q * kSwdDigits + ((key >> (8 * q)) & 255u)], 1u);
      }
    }
    __syncthreads();
    for (int i = tid; i < 4 * kSwdDigits; i += kSwdThreads) {
      const uint32_t c = h[i];
      if (i < kSwdDigits) tcount[((int64_t)k * kSwdDigits + i) * ntiles + tile] = c;
      if (c) atomicAdd(&hist[k * 4 * kSwdDigits + i], c);
    }
    __syncthreads();
  }
}

// ---- 2. per pass: tile counts, scan, ranked scatter ------------------------------------------------------------
// grid (ntiles, nproj): digit counts of one tile of one direction; lanes of a warp with equal digits add once
__global__ void __launch_bounds__(kSwdThreads)
swd_count_kernel(const uint32_t* __restrict__ keys, int64_t n, int shift, int ntiles, uint32_t* __restrict__ tcount) {
  __shared__ uint32_t h[kSwdDigits + 1];
  const int tid = threadIdx.x;
  h[tid] = 0;
  if (tid == 0) h[kSwdDigits] = 0;
  pdl_enter();
  __syncthreads();
  const int tile = blockIdx.x, k = blockIdx.y;
  const int64_t t0 = (int64_t)tile * kSwdTile;
  const uint32_t* kk = keys + (int64_t)k * n;
#pragma unroll
  for (int j = 0; j < kSwdItems; ++j) {
    const int64_t r = t0 + tid + j * kSwdThreads;
    const uint32_t dg = r < n ? (kk[r] >> shift) & 255u : (uint32_t)kSwdDigits;
    const uint32_t peers = __match_any_sync(0xffffffffu, dg);
    if ((threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&h[dg], (uint32_t)__popc(peers));
  }
  __syncthreads();
  tcount[((int64_t)k * kSwdDigits + tid) * ntiles + tile] = h[tid];
}

// one warp per (direction, digit) row, in place: base = (keys of the direction with a smaller digit) + (keys with this
// digit in earlier tiles)
__global__ void __launch_bounds__(kSwdThreads)
swd_scan_kernel(uint32_t* __restrict__ tcount, const uint32_t* __restrict__ hist, int pass, int nproj, int ntiles) {
  pdl_enter();
  const int row = (int)((blockIdx.x * (unsigned)kSwdThreads + threadIdx.x) >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nproj * kSwdDigits) return;
  const int k = row / kSwdDigits, dg = row % kSwdDigits;
  const uint32_t* hk = hist + (k * 4 + pass) * kSwdDigits;
  uint32_t s = 0;
  for (int i = lane; i < dg; i += 32) s += hk[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  uint32_t* r = tcount + (int64_t)row * ntiles;
  for (int t0 = 0; t0 < ntiles; t0 += 32) {
    const int t = t0 + lane;
    const uint32_t c = t < ntiles ? r[t] : 0u;
    uint32_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += v;
    }
    if (t < ntiles) r[t] = s + inc - c;
    s += __shfl_sync(0xffffffffu, inc, 31);
  }
}

struct SwdPass {
  const uint32_t* keys_in;
  const int32_t* idx_in;     // unused in pass 0 (the payload is the position)
  uint32_t* keys_out;
  int32_t* idx_out;
  const uint32_t* base;      // scanned [direction][digit][tile]
  int64_t n;
  int ntiles, shift;
  // kSwdSorted
  const float* x;
  const float* theta;        // [direction][D] of this chunk
  float* sorted;             // [direction][n] of this chunk
  int32_t* perm;             // may be NULL
  // kSwdWpp
  const float* v;            // sorted reference projections [direction][m] of this chunk
  int64_t m;
  double p;
  float* grad;               // [direction][n] of this chunk, may be NULL
  double* partial;           // [direction][tile]
};

// p-th power of |d| and p |d|^(p-1) sign(d) / p (the factor p is applied once per element)
template <int PM>
__device__ __forceinline__ double swd_pow(double d, double p) {
  const double a = fabs(d);
  if (PM == 1) return a;
  if (PM == 2) return d * d;
  return pow(a, p);
}
template <int PM>
__device__ __forceinline__ double swd_dpow(double d, double p) {
  const double s = (double)((d > 0.0) - (d < 0.0));
  if (PM == 1) return s;
  if (PM == 2) return d;
  return pow(fabs(d), p - 1.0) * s;
}

// rank i's share of W_p^p (returned) and of dW_p^p/du (in g)
template <int PM>
__device__ __forceinline__ double swd_rank_term(float u, int64_t i, const SwdPass& a, const float* __restrict__ v,
                                                bool want_grad, double& g) {
  const int64_t n = a.n, m = a.m;
  const int64_t lo = i * m, hi = lo + m;
  const int64_t jend = (hi - 1) / n;
  double w = 0.0, gs = 0.0;
  for (int64_t j = lo / n; j <= jend; ++j) {
    const int64_t len = min(hi, (j + 1) * n) - max(lo, j * n);
    const double d = (double)u - (double)v[j];
    w += (double)len * swd_pow<PM>(d, a.p);
    if (want_grad) gs += (double)len * swd_dpow<PM>(d, a.p);
  }
  const double inv = 1.0 / ((double)n * (double)m);
  g = a.p * gs * inv;
  return w * inv;
}

// grid (ntiles, nproj)
template <int kOut, bool kFirst, int D, int PM>
__global__ void __launch_bounds__(kSwdThreads)
swd_scatter_kernel(const SwdPass a) {
  __shared__ uint32_t skey[kSwdTile];
  __shared__ int32_t sidx[kSwdTile];
  __shared__ uint32_t wcnt[kSwdWarps][kSwdDigits + 1];   // slot 256 collects the lanes past the end of the tile
  __shared__ uint32_t dstart[kSwdDigits], gbase[kSwdDigits], wsum[kSwdWarps];
  __shared__ double red[kSwdWarps];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < kSwdWarps * (kSwdDigits + 1); i += kSwdThreads) (&wcnt[0][0])[i] = 0;
  pdl_enter();
  const int tile = blockIdx.x, k = blockIdx.y;
  const int64_t n = a.n, t0 = (int64_t)tile * kSwdTile;
  const int cnt = (int)min((int64_t)kSwdTile, n - t0);
  const int64_t dir = (int64_t)k * n;
  gbase[tid] = a.base[((int64_t)k * kSwdDigits + tid) * a.ntiles + tile];
  __syncthreads();

  // ranks within (warp, digit) in index order: warp w owns keys [256 w, 256 w + 256) of the tile, 32 per round
  uint32_t key[kSwdItems], rank[kSwdItems];
  int32_t id[kSwdItems];
#pragma unroll
  for (int r = 0; r < kSwdItems; ++r) {
    const int e = warp * (32 * kSwdItems) + r * 32 + lane;
    const bool live = e < cnt;
    key[r] = live ? a.keys_in[dir + t0 + e] : 0u;
    id[r] = kFirst ? (int32_t)(t0 + e) : (live ? a.idx_in[dir + t0 + e] : 0);
  }
#pragma unroll
  for (int r = 0; r < kSwdItems; ++r) {
    const int e = warp * (32 * kSwdItems) + r * 32 + lane;
    const uint32_t dg = e < cnt ? (key[r] >> a.shift) & 255u : (uint32_t)kSwdDigits;
    const uint32_t peers = __match_any_sync(0xffffffffu, dg);
    const uint32_t before = wcnt[warp][dg];
    __syncwarp();
    if (lane == __ffs(peers) - 1) wcnt[warp][dg] = before + __popc(peers);
    __syncwarp();
    rank[r] = before + __popc(peers & lanemask_lt());
  }
  __syncthreads();

  // thread tid = digit tid: offsets of the warps within the digit, then the digit's start in the tile
  uint32_t tot = 0;
#pragma unroll
  for (int w = 0; w < kSwdWarps; ++w) {
    const uint32_t c = wcnt[w][tid];
    wcnt[w][tid] = tot;
    tot += c;
  }
  uint32_t inc = tot;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += v;
  }
  if (lane == 31) wsum[warp] = inc;
  __syncthreads();
  uint32_t woff = 0;
  for (int w = 0; w < warp; ++w) woff += wsum[w];
  dstart[tid] = woff + inc - tot;
  __syncthreads();

  // stable reorder by digit inside the tile
#pragma unroll
  for (int r = 0; r < kSwdItems; ++r) {
    const int e = warp * (32 * kSwdItems) + r * 32 + lane;
    if (e < cnt) {
      const uint32_t dg = (key[r] >> a.shift) & 255u;
      const uint32_t lp = dstart[dg] + wcnt[warp][dg] + rank[r];
      skey[lp] = key[r];
      sidx[lp] = id[r];
    }
  }
  __syncthreads();

  // consecutive threads hold consecutive positions of a digit's run, i.e. consecutive global ranks
  double acc = 0.0;
  const bool want_grad = kOut == kSwdWpp && a.grad != nullptr;
#pragma unroll
  for (int j = 0; j < kSwdItems; ++j) {
    const int s = tid + j * kSwdThreads;
    if (s < cnt) {
      const uint32_t kk = skey[s];
      const uint32_t dg = (kk >> a.shift) & 255u;
      const int64_t pos = (int64_t)gbase[dg] + (s - (int)dstart[dg]);
      const int32_t idx = sidx[s];
      if (kOut == kSwdMid) {
        a.keys_out[dir + pos] = kk;
        a.idx_out[dir + pos] = idx;
      } else if (kOut == kSwdSorted) {
        a.sorted[dir + pos] = swd_project<D>(a.x + (int64_t)idx * D, a.theta + k * D);
        if (a.perm) a.perm[dir + pos] = idx;
      } else {
        double g;
        acc += swd_rank_term<PM>(swd_value(kk), pos, a, a.v + (int64_t)k * a.m, want_grad, g);
        if (want_grad) a.grad[dir + idx] = (float)g;
      }
    }
  }
  if (kOut == kSwdWpp) {
    acc = warp_sum(acc);
    if (lane == 0) red[warp] = acc;
    __syncthreads();
    if (tid == 0) {
      double s = 0.0;
      for (int w = 0; w < kSwdWarps; ++w) s += red[w];
      a.partial[(int64_t)k * a.ntiles + tile] = s;
    }
  }
}

// one CTA per direction: its tile partials in a fixed order
__global__ void __launch_bounds__(kSwdThreads)
swd_reduce_kernel(const double* __restrict__ partial, int ntiles, double* __restrict__ wpp) {
  pdl_enter();
  const double* pk = partial + (int64_t)blockIdx.x * ntiles;
  double s = 0.0;
  for (int t = threadIdx.x; t < ntiles; t += kSwdThreads) s += pk[t];
  __shared__ double red[kSwdWarps];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kSwdWarps; ++w) t += red[w];
    wpp[blockIdx.x] = t;
  }
}

// ---- backward ---------------------------------------------------------------------------------------------------
template <int D>
__global__ void __launch_bounds__(kSwdThreads)
swd_bwd_kernel(const float* __restrict__ gcoef, int64_t n, const float* __restrict__ theta, int nproj,
               const double* __restrict__ gw, float* __restrict__ gx) {
  __shared__ float w[kSwdThreads][D];
  pdl_enter();
  const int tid = threadIdx.x;
  const int64_t i = (int64_t)blockIdx.x * kSwdThreads + tid;
  float acc[D];
#pragma unroll
  for (int c = 0; c < D; ++c) acc[c] = 0.f;
  for (int k0 = 0; k0 < nproj; k0 += kSwdThreads) {
    __syncthreads();
    const int kk = k0 + tid;
    if (kk < nproj) {
#pragma unroll
      for (int c = 0; c < D; ++c) w[tid][c] = (float)(gw[kk] * (double)theta[kk * D + c]);
    }
    __syncthreads();
    const int kn = min(kSwdThreads, nproj - k0);
    if (i < n) {
      for (int k = 0; k < kn; ++k) {
        const float g = gcoef[(int64_t)(k0 + k) * n + i];
#pragma unroll
        for (int c = 0; c < D; ++c) acc[c] = fmaf(w[k][c], g, acc[c]);
      }
    }
  }
  if (i < n) {
#pragma unroll
    for (int c = 0; c < D; ++c) gx[i * D + c] = acc[c];
  }
}

// ---- launch plan ------------------------------------------------------------------------------------------------
typedef void (*SwdKeysFn)(const float*, int64_t, const float*, int, int, int, uint32_t*, uint32_t*, uint32_t*);
typedef void (*SwdScatterFn)(const SwdPass);
typedef void (*SwdBwdFn)(const float*, int64_t, const float*, int, const double*, float*);

#define MFB_SWD_BY_D(K) {K<1>, K<2>, K<3>, K<4>, K<5>, K<6>, K<7>, K<8>}
static SwdKeysFn swd_keys_for(int d) {
  static const SwdKeysFn t[kMaxDim] = MFB_SWD_BY_D(swd_keys_kernel);
  return t[d - 1];
}
static SwdBwdFn swd_bwd_for(int d) {
  static const SwdBwdFn t[kMaxDim] = MFB_SWD_BY_D(swd_bwd_kernel);
  return t[d - 1];
}
#undef MFB_SWD_BY_D
static SwdScatterFn swd_sorted_for(int d) {
  static const SwdScatterFn t[kMaxDim] = {
      swd_scatter_kernel<kSwdSorted, false, 1, 0>, swd_scatter_kernel<kSwdSorted, false, 2, 0>,
      swd_scatter_kernel<kSwdSorted, false, 3, 0>, swd_scatter_kernel<kSwdSorted, false, 4, 0>,
      swd_scatter_kernel<kSwdSorted, false, 5, 0>, swd_scatter_kernel<kSwdSorted, false, 6, 0>,
      swd_scatter_kernel<kSwdSorted, false, 7, 0>, swd_scatter_kernel<kSwdSorted, false, 8, 0>};
  return t[d - 1];
}
static SwdScatterFn swd_wpp_for(double p) {
  return p == 1.0 ? swd_scatter_kernel<kSwdWpp, false, 1, 1>
                  : (p == 2.0 ? swd_scatter_kernel<kSwdWpp, false, 1, 2> : swd_scatter_kernel<kSwdWpp, false, 1, 0>);
}

static size_t swd_round16(size_t b) { return (b + 15) & ~(size_t)15; }

struct SwdPlan {
  int ntiles;
  size_t keys, idx, tcount, hist, partial;   // bytes of each buffer for `chunk` directions
  size_t bytes;
};

static SwdPlan swd_plan(int64_t n, int64_t chunk) {
  SwdPlan p;
  p.ntiles = (int)((n + kSwdTile - 1) / kSwdTile);
  p.keys = swd_round16((size_t)chunk * n * 4);
  p.idx = p.keys;
  p.tcount = swd_round16((size_t)chunk * kSwdDigits * p.ntiles * 4);
  p.hist = swd_round16((size_t)chunk * 4 * kSwdDigits * 4);
  p.partial = swd_round16((size_t)chunk * p.ntiles * 8);
  p.bytes = 2 * p.keys + 2 * p.idx + p.tcount + p.hist + p.partial;
  return p;
}

// directions per chunk: as many as the workspace holds (swd_plan(n, c).bytes <= c * swd_plan(n, 1).bytes)
static int swd_chunk(int64_t n, int nproj, int64_t workspace_bytes) {
  const int64_t one = (int64_t)swd_plan(n, 1).bytes;
  int64_t c = workspace_bytes / one;
  if (c > nproj) c = nproj;
  if (c > kSwdMaxChunk) c = kSwdMaxChunk;
  return (int)c;
}

static int swd_check(const float* x, int64_t n, int d, const float* theta, int nproj) {
  if (!x || !theta || n < 1 || n > INT32_MAX || d < 1 || nproj < 1) return MFB_E_BADARG;
  if (d > kMaxDim) return MFB_E_UNSUPPORTED;
  return 0;
}

// Sorts the projections of directions [0, nproj) chunk by chunk; the last pass of a chunk starting at k0 runs `last`
// with the fields `fin(k0, pass)` fills in.  With wpp, swd_reduce_kernel then writes the chunk's W_p^p at wpp + k0.
template <typename Fin>
static int swd_run(const float* x, int64_t n, int d, const float* theta, int nproj, SwdScatterFn last, double* wpp,
                   void* workspace, int64_t workspace_bytes, cudaStream_t st, Fin fin) {
  const int chunk = swd_chunk(n, nproj, workspace_bytes);
  if (chunk < 1) return MFB_E_WORKSPACE;
  const SwdPlan pl = swd_plan(n, chunk);
  char* ws = (char*)workspace;
  uint32_t* keys[2] = {(uint32_t*)ws, (uint32_t*)(ws + pl.keys)};
  int32_t* idx[2] = {(int32_t*)(ws + 2 * pl.keys), (int32_t*)(ws + 2 * pl.keys + pl.idx)};
  uint32_t* tcount = (uint32_t*)(ws + 2 * pl.keys + 2 * pl.idx);
  uint32_t* hist = (uint32_t*)((char*)tcount + pl.tcount);
  double* partial = (double*)((char*)hist + pl.hist);
  const int ntiles = pl.ntiles;
  const int sms = sm_count();
  for (int k0 = 0; k0 < nproj; k0 += chunk) {
    const int pc = min(chunk, nproj - k0);
    MFB_CUDA(cudaMemsetAsync(hist, 0, (size_t)pc * 4 * kSwdDigits * 4, st));
    // groups of directions per tile of rows: enough CTAs for four per SM
    int groups = (int)min((int64_t)pc, (4 * (int64_t)sms + ntiles - 1) / ntiles);
    const int per = (pc + groups - 1) / groups;
    groups = (pc + per - 1) / per;
    MFB_CUDA(launch_pdl(swd_keys_for(d), dim3(ntiles, groups), dim3(kSwdThreads), 0, st, x, n,
                        theta + (int64_t)k0 * d, pc, per, ntiles, keys[0], tcount, hist));
    for (int q = 0; q < 4; ++q) {
      const int src = q & 1;
      if (q > 0)
        MFB_CUDA(launch_pdl(swd_count_kernel, dim3(ntiles, pc), dim3(kSwdThreads), 0, st, (const uint32_t*)keys[src],
                            n, 8 * q, ntiles, tcount));
      const int64_t rows = (int64_t)pc * kSwdDigits;
      MFB_CUDA(launch_pdl(swd_scan_kernel, dim3((unsigned)((rows + kSwdWarps - 1) / kSwdWarps)), dim3(kSwdThreads), 0,
                          st, tcount, (const uint32_t*)hist, q, pc, ntiles));
      SwdPass a = {};
      a.keys_in = keys[src];
      a.idx_in = idx[src];
      a.keys_out = keys[src ^ 1];
      a.idx_out = idx[src ^ 1];
      a.base = tcount;
      a.n = n;
      a.ntiles = ntiles;
      a.shift = 8 * q;
      a.partial = partial;
      SwdScatterFn fn = q == 0 ? swd_scatter_kernel<kSwdMid, true, 1, 0> : swd_scatter_kernel<kSwdMid, false, 1, 0>;
      if (q == 3) {
        fin(k0, a);
        fn = last;
      }
      MFB_CUDA(launch_pdl(fn, dim3(ntiles, pc), dim3(kSwdThreads), 0, st, (const SwdPass)a));
    }
    if (wpp)
      MFB_CUDA(launch_pdl(swd_reduce_kernel, dim3(pc), dim3(kSwdThreads), 0, st, (const double*)partial, ntiles,
                          wpp + k0));
  }
  return launch_status();
}

}  // namespace mfb

using namespace mfb;

extern "C" {

int64_t mfb_swd_workspace_bytes(int64_t n, int nproj_chunk) {
  if (n < 1 || n > INT32_MAX || nproj_chunk < 1 || nproj_chunk > kSwdMaxChunk) return 0;
  return (int64_t)swd_plan(n, nproj_chunk).bytes;
}

int mfb_swd_sort(const float* x, int64_t n, int d, const float* theta, int nproj, float* sorted, int32_t* perm,
                 void* workspace, int64_t workspace_bytes, void* stream) {
  const int rc = swd_check(x, n, d, theta, nproj);
  if (rc) return rc;
  MFB_CHECK_ARG(sorted && workspace);
  return swd_run(x, n, d, theta, nproj, swd_sorted_for(d), nullptr, workspace, workspace_bytes, (cudaStream_t)stream,
                 [&](int k0, SwdPass& a) {
                   a.x = x;
                   a.theta = theta + (int64_t)k0 * d;
                   a.sorted = sorted + (int64_t)k0 * n;
                   a.perm = perm ? perm + (int64_t)k0 * n : nullptr;
                 });
}

int mfb_swd_wpp(const float* x, int64_t n, int d, const float* theta, int nproj, const float* y_sorted, int64_t m,
                double p, double* wpp, float* grad_coef, void* workspace, int64_t workspace_bytes, void* stream) {
  const int rc = swd_check(x, n, d, theta, nproj);
  if (rc) return rc;
  MFB_CHECK_ARG(y_sorted && wpp && workspace && m >= 1 && m <= INT32_MAX && p >= 1.0 && isfinite(p));
  return swd_run(x, n, d, theta, nproj, swd_wpp_for(p), wpp, workspace, workspace_bytes, (cudaStream_t)stream,
                 [&](int k0, SwdPass& a) {
                   a.v = y_sorted + (int64_t)k0 * m;
                   a.m = m;
                   a.p = p;
                   a.grad = grad_coef ? grad_coef + (int64_t)k0 * n : nullptr;
                 });
}

int mfb_swd_bwd(const float* grad_coef, int64_t n, int d, const float* theta, int nproj, const double* gwpp,
                float* gx, void* stream) {
  MFB_CHECK_ARG(grad_coef && theta && gwpp && gx && n >= 1 && n <= INT32_MAX && d >= 1 && nproj >= 1);
  if (d > kMaxDim) return MFB_E_UNSUPPORTED;
  MFB_CUDA(launch_pdl(swd_bwd_for(d), dim3((unsigned)((n + kSwdThreads - 1) / kSwdThreads)), dim3(kSwdThreads), 0,
                      (cudaStream_t)stream, grad_coef, n, theta, nproj, gwpp, gx));
  return launch_status();
}

}  // extern "C"
