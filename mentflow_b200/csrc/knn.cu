// k-th nearest neighbour of every particle among the batch, for the k-NN entropy estimator (entropy.py
// KNNEntropyEstimator):  r_i = |x_i - x_n(i)|, n(i) the k-th nearest OTHER particle under the key (r^2, j), and
// logsum = sum_i log(r_i + pad) in double.  All pairs, O(N^2 d): the forward is bound by the issue slots of the
// distance arithmetic (DESIGN.md §4.2).
//
// Forward, four launches:
//   1. knn_transpose_kernel: x[N][D] -> xt[D][Npad] (columns padded to whole tiles with +inf, which is never a
//      neighbour: (x - inf)^2 = inf fails every strict compare);
//   2. knn_partial_kernel: one CTA = 512 queries (two per thread, rows in registers) x one contiguous range of
//      candidate tiles (a "split"); candidate tiles stream through a two-stage bulk-copy / mbarrier ring.  Each thread
//      keeps its queries' k best (r^2, j) in sorted register lists and writes them per split;
//   3. knn_merge_kernel: merges the splits' lists in split order, writes r, n and one double partial of the log sum
//      per CTA (a query without k neighbours at a finite distance gets r = inf, n = itself);
//   4. knn_logsum_kernel: adds the partials in a fixed order.
// Candidates reach a list in ascending j (within a tile, tile by tile, split by split), and a list admits a candidate
// only with a STRICTLY smaller r^2 than its current k-th, so ties go to the smaller index and the result does not
// depend on the split.  Distances are direct differences in fp32 (not the Gram form |x|^2 + |y|^2 - 2 x.y, whose
// cancellation costs ~1e-2 of r^2 at |x| ~ 3, r ~ 1e-2: the estimator's logs weigh exactly those short distances).
// No floating-point atomics: every output is bitwise reproducible.
//
// Backward of logsum (neighbour identities held fixed, as autograd through cdist + topk):
//   d logsum / dx_i = w_i (x_i - x_n(i)) + sum_{j : n(j) = i} w_j (x_i - x_j),  w_j = 1 / (r_j (r_j + pad)), 0 at r_j = 0.
// The caller passes n(.) stably sorted with its permutation; particle i sums its segment in ascending j.
//
// Row ranges (particles sharded over ranks): the search and the backward run for the queries [row0, row0 + nrows) of
// a batch of n candidates.  A pair's r^2 and the k-th neighbour depend only on the pair and on the candidate set, so
// the rows of a range are bit for bit those of the whole batch; knn_logpart_kernel then adds log(r + pad) of the
// gathered r with the merge kernel's own block partials (knn_block_logpart), so the log sum is the whole batch's too.
#include "common.cuh"

namespace mfb {

constexpr int kKnnThreads = 256;
constexpr int kKnnRows = 2 * kKnnThreads;   // queries per CTA (two per thread)
constexpr int kKnnTile = 256;               // candidates per tile
constexpr int kKnnMaxK = 16;
constexpr int kKnnMaxSplits = 16;
constexpr int kKnnMinTilesPerSplit = 4;     // keeps the merge's traffic small against the pair work

// ---- packed fp32 pairs: one issue slot for two lanes (FADD2 / FMUL2 / FFMA2, IEEE round-to-nearest) -------------
__device__ __forceinline__ uint64_t pack2(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) {
  uint64_t c;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(c) : "l"(a), "l"(b));
  return c;
}
__device__ __forceinline__ uint64_t mul2(uint64_t a, uint64_t b) {
  uint64_t c;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(c) : "l"(a), "l"(b));
  return c;
}
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}

// ---- sorted register list of the k best (r^2, j) ----------------------------------------------------------------
// KB >= k slots in ascending order; the first KB - k hold the sentinel -1, which nothing displaces, so the k-th best
// is always key[KB - 1] and no slot is indexed at run time.
template <int KB>
struct TopK {
  float key[KB];
  int id[KB];
  __device__ __forceinline__ void init(int k) {
#pragma unroll
    for (int s = 0; s < KB; ++s) {
      key[s] = s < KB - k ? -1.0f : __int_as_float(0x7f800000);
      id[s] = -1;
    }
  }
  __device__ __forceinline__ float worst() const { return key[KB - 1]; }
  // the candidate replaces the k-th and bubbles up past every STRICTLY larger key: it lands after equal keys, which
  // belong to smaller indices
  __device__ __forceinline__ void insert(float d, int j) {
    key[KB - 1] = d;
    id[KB - 1] = j;
#pragma unroll
    for (int s = KB - 1; s > 0; --s) {
      if (key[s] < key[s - 1]) {
        const float tk = key[s];
        key[s] = key[s - 1];
        key[s - 1] = tk;
        const int ti = id[s];
        id[s] = id[s - 1];
        id[s - 1] = ti;
      }
    }
  }
};

__global__ void knn_transpose_kernel(const float* __restrict__ x, int64_t n, int d, int64_t npad,
                                     float* __restrict__ xt) {
  pdl_enter();
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npad * d) return;
  const int c = (int)(i / npad);
  const int64_t j = i - (int64_t)c * npad;
  xt[i] = j < n ? x[j * d + c] : __int_as_float(0x7f800000);
}

// squared distances of two queries (nq = -x, each coordinate twice) to the four candidates jj..jj+3 of a tile
template <int D>
__device__ __forceinline__ void dist_2x4(const float* __restrict__ ts, int jj, const uint64_t (&nq)[2][D],
                                         float (&d2)[2][4]) {
  uint64_t s[2][2];
#pragma unroll
  for (int c = 0; c < D; ++c) {
    const float4 y = *reinterpret_cast<const float4*>(ts + c * kKnnTile + jj);
    const uint64_t y01 = pack2(y.x, y.y), y23 = pack2(y.z, y.w);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      const uint64_t e01 = add2(y01, nq[q][c]), e23 = add2(y23, nq[q][c]);
      if (c == 0) {
        s[q][0] = mul2(e01, e01);
        s[q][1] = mul2(e23, e23);
      } else {
        s[q][0] = fma2(e01, e01, s[q][0]);
        s[q][1] = fma2(e23, e23, s[q][1]);
      }
    }
  }
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    unpack2(s[q][0], d2[q][0], d2[q][1]);
    unpack2(s[q][1], d2[q][2], d2[q][3]);
  }
}

// one tile against the thread's two lists; kSelf: the tile may hold one of the queries (excluded by index)
template <int D, int KB, bool kSelf>
__device__ __forceinline__ void scan_tile(const float* __restrict__ ts, int j0, const int (&qi)[2],
                                          const uint64_t (&nq)[2][D], TopK<KB> (&top)[2]) {
#pragma unroll 2
  for (int jj = 0; jj < kKnnTile; jj += 4) {
    float d2[2][4];
    dist_2x4<D>(ts, jj, nq, d2);
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      if (kSelf) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (j0 + jj + e == qi[q]) d2[q][e] = __int_as_float(0x7f800000);
      }
      // common path: one compare of the four against the current k-th
      const float m = fminf(fminf(d2[q][0], d2[q][1]), fminf(d2[q][2], d2[q][3]));
      if (m < top[q].worst()) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
          if (d2[q][e] < top[q].worst()) top[q].insert(d2[q][e], j0 + jj + e);
      }
    }
  }
}

template <int D, int KB>
__global__ void __launch_bounds__(kKnnThreads, 2)
knn_partial_kernel(const float* __restrict__ x, const float* __restrict__ xt, int64_t npad, int row0, int nrows, int k,
                   int ntiles, int splits, float* __restrict__ pd2, int32_t* __restrict__ pidx) {
  __shared__ __align__(128) float tile[2][D * kKnnTile];
  __shared__ __align__(8) uint64_t bar[2];
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(&bar[0], 1);
    mbar_init(&bar[1], 1);
    fence_mbar_init();
  }
  pdl_enter();
  __syncthreads();

  const int split = blockIdx.y;
  const int t_begin = (int)((int64_t)split * ntiles / splits);
  const int t_end = (int)((int64_t)(split + 1) * ntiles / splits);
  auto issue = [&](int stage, int t) {   // thread 0 only
    mbar_expect_tx(&bar[stage], D * kKnnTile * 4);
#pragma unroll
    for (int c = 0; c < D; ++c)
      tma_load_1d(&tile[stage][c * kKnnTile], xt + c * npad + (int64_t)t * kKnnTile, kKnnTile * 4, &bar[stage]);
  };
  if (tid == 0 && t_begin < t_end) issue(0, t_begin);

  const int q0 = row0 + blockIdx.x * kKnnRows;   // global index of the CTA's first query
  const int qend = row0 + nrows;
  int qi[2];
  uint64_t nq[2][D];
  TopK<KB> top[2];
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    qi[q] = q0 + q * kKnnThreads + tid;
    const bool live = qi[q] < qend;
#pragma unroll
    for (int c = 0; c < D; ++c) {
      const float v = live ? -x[(int64_t)qi[q] * D + c] : 0.f;
      nq[q][c] = pack2(v, v);
    }
    top[q].init(k);
  }

  int it = 0;
  for (int t = t_begin; t < t_end; ++t, ++it) {
    const int stage = it & 1;
    if (tid == 0 && t + 1 < t_end) issue(stage ^ 1, t + 1);   // stage^1 was released by the barrier below
    mbar_wait(&bar[stage], (it >> 1) & 1);
    const int j0 = t * kKnnTile;
    if (j0 < q0 + kKnnRows && q0 < j0 + kKnnTile) scan_tile<D, KB, true>(tile[stage], j0, qi, nq, top);
    else scan_tile<D, KB, false>(tile[stage], j0, qi, nq, top);
    __syncthreads();   // everyone is done with tile[stage] before it is refilled
  }

  // the k real entries, ascending, at [split][rank][local query]
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    if (qi[q] >= qend) continue;
#pragma unroll
    for (int s = 0; s < KB; ++s) {
      const int rank = s - (KB - k);
      if (rank >= 0) {
        const int64_t o = ((int64_t)split * k + rank) * nrows + (qi[q] - row0);
        pd2[o] = top[q].key[s];
        pidx[o] = top[q].id[s];
      }
    }
  }
}

__device__ __forceinline__ double knn_logterm(float rv, double pad) { return log((double)rv + pad); }

// one double partial of the log sum per block of kKnnThreads queries: warp sums, then the warps in order.  The merge
// kernel and knn_logpart_kernel both call it, so a log sum of gathered rows adds exactly as one whole-batch search.
__device__ __forceinline__ void knn_block_logpart(double lg, double* __restrict__ logpart) {
  __shared__ double red[kKnnThreads / 32];
  lg = warp_sum(lg);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = lg;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < kKnnThreads / 32; ++w) s += red[w];
    logpart[blockIdx.x] = s;
  }
}

// local queries q in [0, nrows), global index row0 + q; logpart NULL: no log sum (a row range of a sharded batch)
template <int KB>
__global__ void __launch_bounds__(kKnnThreads)
knn_merge_kernel(const float* __restrict__ pd2, const int32_t* __restrict__ pidx, int64_t row0, int64_t nrows, int k,
                 int splits, double pad, float* __restrict__ r, int32_t* __restrict__ idx, double* __restrict__ logpart) {
  pdl_enter();
  const int64_t q = (int64_t)blockIdx.x * kKnnThreads + threadIdx.x;
  double lg = 0.0;
  if (q < nrows) {
    TopK<KB> top;
    top.init(k);
    for (int s = 0; s < splits; ++s) {
      for (int rank = 0; rank < k; ++rank) {   // a split's list is ascending: the first miss ends it
        const int64_t o = ((int64_t)s * k + rank) * nrows + q;
        const float d = pd2[o];
        if (!(d < top.worst())) break;
        top.insert(d, pidx[o]);
      }
    }
    // fewer than k others at a finite distance (a NaN or inf coordinate, or every r^2 overflowing): r = inf and the
    // query itself as its neighbour, so the index stays in range and the backward gives the pair weight 0
    const int nb = top.id[KB - 1];
    const float rv = nb < 0 ? __int_as_float(0x7f800000) : sqrtf(top.worst());
    r[q] = rv;
    idx[q] = nb < 0 ? (int32_t)(row0 + q) : nb;
    lg = knn_logterm(rv, pad);
  }
  if (logpart) knn_block_logpart(lg, logpart);
}

// the merge kernel's log partials from r of the whole batch (gathered from row ranges)
__global__ void __launch_bounds__(kKnnThreads)
knn_logpart_kernel(const float* __restrict__ r, int64_t n, double pad, double* __restrict__ logpart) {
  pdl_enter();
  const int64_t q = (int64_t)blockIdx.x * kKnnThreads + threadIdx.x;
  knn_block_logpart(q < n ? knn_logterm(r[q], pad) : 0.0, logpart);
}

// one block: threads stride over the partials, fixed shuffle tree, fixed warp order => deterministic
__global__ void knn_logsum_kernel(const double* __restrict__ logpart, int nparts, double* __restrict__ logsum) {
  pdl_enter();
  double s = 0.0;
  for (int c = threadIdx.x; c < nparts; c += blockDim.x) s += logpart[c];
  __shared__ double red[kKnnThreads / 32];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    logsum[0] = t;
  }
}

__device__ __forceinline__ float knn_weight(float rv, double pad, double g) {
  return rv > 0.f ? (float)(g / ((double)rv * ((double)rv + pad))) : 0.f;
}

template <int D>
__global__ void __launch_bounds__(kKnnThreads)
knn_bwd_kernel(const float* __restrict__ x, int64_t n, const float* __restrict__ r, const int32_t* __restrict__ idx,
               const int32_t* __restrict__ sorted_idx, const int64_t* __restrict__ perm, int64_t row0, int64_t nrows,
               double pad, const double* __restrict__ glogsum, float* __restrict__ gx) {
  pdl_enter();
  const int64_t li = (int64_t)blockIdx.x * kKnnThreads + threadIdx.x;   // row of gx; i is its particle in the batch
  if (li >= nrows) return;
  const int64_t i = row0 + li;
  const double g = glogsum[0];
  float xi[D], acc[D];
  const float wi = knn_weight(r[i], pad, g);
  const int64_t ni = idx[i];
#pragma unroll
  for (int c = 0; c < D; ++c) {
    xi[c] = x[i * D + c];
    acc[c] = wi * (xi[c] - x[ni * D + c]);
  }
  // segment of i in the sorted neighbour indices: [lower_bound(i), lower_bound(i + 1))
  int64_t lo = 0, hi = n;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (sorted_idx[mid] < i) lo = mid + 1;
    else hi = mid;
  }
  for (int64_t p = lo; p < n && sorted_idx[p] == i; ++p) {
    const int64_t j = perm[p];
    const float wj = knn_weight(r[j], pad, g);
#pragma unroll
    for (int c = 0; c < D; ++c) acc[c] = fmaf(wj, xi[c] - x[j * D + c], acc[c]);
  }
#pragma unroll
  for (int c = 0; c < D; ++c) gx[li * D + c] = acc[c];
}

// ---- launch plan -----------------------------------------------------------------------------------------------
typedef void (*KnnPartialFn)(const float*, const float*, int64_t, int, int, int, int, int, float*, int32_t*);
typedef void (*KnnMergeFn)(const float*, const int32_t*, int64_t, int64_t, int, int, double, float*, int32_t*,
                           double*);
typedef void (*KnnBwdFn)(const float*, int64_t, const float*, const int32_t*, const int32_t*, const int64_t*, int64_t,
                         int64_t, double, const double*, float*);

static int knn_list_slots(int k) { return k <= 4 ? 4 : (k <= 8 ? 8 : 16); }

#define MFB_KNN_ROW(D) {knn_partial_kernel<D, 4>, knn_partial_kernel<D, 8>, knn_partial_kernel<D, 16>}
static KnnPartialFn knn_partial_for(int d, int k) {
  static const KnnPartialFn table[kMaxDim][3] = {MFB_KNN_ROW(1), MFB_KNN_ROW(2), MFB_KNN_ROW(3), MFB_KNN_ROW(4),
                                                 MFB_KNN_ROW(5), MFB_KNN_ROW(6), MFB_KNN_ROW(7), MFB_KNN_ROW(8)};
  const int kb = knn_list_slots(k);
  return table[d - 1][kb == 4 ? 0 : (kb == 8 ? 1 : 2)];
}
#undef MFB_KNN_ROW

static KnnMergeFn knn_merge_for(int k) {
  const int kb = knn_list_slots(k);
  return kb == 4 ? knn_merge_kernel<4> : (kb == 8 ? knn_merge_kernel<8> : knn_merge_kernel<16>);
}

static KnnBwdFn knn_bwd_for(int d) {
  static const KnnBwdFn table[kMaxDim] = {knn_bwd_kernel<1>, knn_bwd_kernel<2>, knn_bwd_kernel<3>, knn_bwd_kernel<4>,
                                          knn_bwd_kernel<5>, knn_bwd_kernel<6>, knn_bwd_kernel<7>, knn_bwd_kernel<8>};
  return table[d - 1];
}

struct KnnPlan {
  int ntiles, qblocks, splits, mblocks;
  int64_t npad;
  size_t off_pd2, off_pidx, off_logpart, bytes;
};

static size_t round16(size_t b) { return (b + 15) & ~(size_t)15; }
static int64_t knn_logparts(int64_t n) { return (n + kKnnThreads - 1) / kKnnThreads; }

// Queries [row0, row0 + nrows) against n candidates: the candidate tiles follow n, the query blocks and the split
// choice follow nrows.  Splits of the candidate axis: with few queries (25,000 fill 49 CTAs of 512) the grid would
// leave most SMs idle, so the candidate tiles are cut into `splits` ranges.  The choice rounds the CTA count up to
// whole waves of resident CTAs (preferring fewer splits unless more are 2 % better), at least kKnnMinTilesPerSplit
// tiles each.
static int knn_plan(int64_t n, int64_t nrows, int d, int k, KnnPlan& p) {
  p.ntiles = (int)((n + kKnnTile - 1) / kKnnTile);
  p.npad = (int64_t)p.ntiles * kKnnTile;
  p.qblocks = (int)((nrows + kKnnRows - 1) / kKnnRows);
  p.mblocks = (int)knn_logparts(nrows);
  int per_sm = 0;
  MFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, knn_partial_for(d, k), kKnnThreads, 0));
  const int64_t slots = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 1);
  int smax = p.ntiles / kKnnMinTilesPerSplit;
  smax = smax < 1 ? 1 : (smax > kKnnMaxSplits ? kKnnMaxSplits : smax);
  int best = 1;
  double best_eff = 0.0;
  for (int s = 1; s <= smax; ++s) {
    const int64_t ctas = (int64_t)p.qblocks * s;
    const double eff = (double)ctas / (double)(slots * ((ctas + slots - 1) / slots));
    if (eff > best_eff + 0.02) {
      best = s;
      best_eff = eff;
    }
  }
  p.splits = best;
  const size_t list = round16((size_t)p.splits * k * nrows * 4);
  p.off_pd2 = (size_t)d * p.npad * 4;
  p.off_pidx = p.off_pd2 + list;
  p.off_logpart = p.off_pidx + list;
  p.bytes = p.off_logpart + (size_t)p.mblocks * 8;
  return 0;
}

static int knn_check(const float* x, int64_t n, int d, int k) {
  if (!x || n < 2 || n > INT32_MAX || d < 1 || k < 1) return MFB_E_BADARG;
  if (d > kMaxDim || k > kKnnMaxK) return MFB_E_UNSUPPORTED;
  if (k >= n) return MFB_E_BADARG;
  return 0;
}

static bool knn_range_ok(int64_t n, int64_t row0, int64_t nrows) {
  return row0 >= 0 && nrows >= 0 && row0 <= n && nrows <= n - row0;
}

}  // namespace mfb

using namespace mfb;

extern "C" {

int64_t mfb_knn_workspace_bytes(int64_t n, int64_t nrows, int d, int k) {
  if (knn_check((const float*)1, n, d, k) || !knn_range_ok(n, 0, nrows) || nrows == 0) return 0;
  KnnPlan p;
  if (knn_plan(n, nrows, d, k, p)) return 0;
  return (int64_t)p.bytes;
}

// transpose, pair search and merge for the queries [row0, row0 + nrows); with logsum (whole batch only) the merge's
// log partials and their fixed-order sum
int mfb_knn_kth(const float* x, int64_t n, int d, int k, int64_t row0, int64_t nrows, double pad, float* r,
                int32_t* idx, double* logsum, void* workspace, int64_t workspace_bytes, void* stream) {
  int rc = knn_check(x, n, d, k);
  if (rc) return rc;
  MFB_CHECK_ARG(knn_range_ok(n, row0, nrows));
  MFB_CHECK_ARG(!logsum || (row0 == 0 && nrows == n));
  if (nrows == 0) return 0;
  MFB_CHECK_ARG(r && idx && workspace);
  KnnPlan p;
  rc = knn_plan(n, nrows, d, k, p);
  if (rc) return rc;
  if (workspace_bytes < (int64_t)p.bytes) return MFB_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  float* xt = (float*)ws;
  float* pd2 = (float*)(ws + p.off_pd2);
  int32_t* pidx = (int32_t*)(ws + p.off_pidx);
  double* logpart = logsum ? (double*)(ws + p.off_logpart) : nullptr;

  const int64_t tn = p.npad * d;
  MFB_CUDA(launch_pdl(knn_transpose_kernel, dim3((unsigned)((tn + 255) / 256)), dim3(256), 0, st, x, n, d, p.npad, xt));
  MFB_CUDA(launch_pdl(knn_partial_for(d, k), dim3(p.qblocks, p.splits), dim3(kKnnThreads), 0, st, x,
                      (const float*)xt, p.npad, (int)row0, (int)nrows, k, p.ntiles, p.splits, pd2, pidx));
  MFB_CUDA(launch_pdl(knn_merge_for(k), dim3(p.mblocks), dim3(kKnnThreads), 0, st, (const float*)pd2,
                      (const int32_t*)pidx, row0, nrows, k, p.splits, pad, r, idx, logpart));
  if (logsum)
    MFB_CUDA(launch_pdl(knn_logsum_kernel, dim3(1), dim3(kKnnThreads), 0, st, (const double*)logpart, p.mblocks,
                        logsum));
  return launch_status();
}

int mfb_knn_logsum(const float* r, int64_t n, double pad, double* logsum, void* workspace, int64_t workspace_bytes,
                   void* stream) {
  MFB_CHECK_ARG(r && logsum && workspace && n >= 1 && n <= INT32_MAX);
  const int64_t parts = knn_logparts(n);
  if (workspace_bytes < parts * 8) return MFB_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  double* logpart = (double*)workspace;
  MFB_CUDA(launch_pdl(knn_logpart_kernel, dim3((unsigned)parts), dim3(kKnnThreads), 0, st, r, n, pad, logpart));
  MFB_CUDA(launch_pdl(knn_logsum_kernel, dim3(1), dim3(kKnnThreads), 0, st, (const double*)logpart, (int)parts,
                      logsum));
  return launch_status();
}

int mfb_knn_kth_bwd(const float* x, int64_t n, int d, const float* r, const int32_t* idx, const int32_t* sorted_idx,
                    const int64_t* perm, int64_t row0, int64_t nrows, double pad, const double* glogsum, float* gx,
                    void* stream) {
  MFB_CHECK_ARG(x && r && idx && sorted_idx && perm && glogsum && n >= 2 && n <= INT32_MAX && d >= 1);
  if (d > kMaxDim) return MFB_E_UNSUPPORTED;
  MFB_CHECK_ARG(knn_range_ok(n, row0, nrows));
  if (nrows == 0) return 0;
  MFB_CHECK_ARG(gx);
  MFB_CUDA(launch_pdl(knn_bwd_for(d), dim3((unsigned)((nrows + kKnnThreads - 1) / kKnnThreads)), dim3(kKnnThreads), 0,
                      (cudaStream_t)stream, x, n, r, idx, sorted_idx, perm, row0, nrows, pad, glogsum, gx));
  return launch_status();
}

}  // extern "C"
