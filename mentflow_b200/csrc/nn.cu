// Plain tanh-MLP generator (generate/nn.py NNGenerator): x = W_out tanh(... tanh(W_1 z + b_1) ...) + b_out, with
// hidden_layers tanh layers of 64 units, z and x of 1..8 features.  fp32 on the CUDA cores (DESIGN.md §4.2).
//
// Shared-memory weight image (floats, every block a multiple of 4):
//   Wt_in [Din][64] (transposed: the first layer runs over outputs) | b_in [64] | W_hid [L-1][64][64] ([out][in], as
//   nn.Linear) | b_hid [L-1][64] | W_out [Dout][64] | b_out [Dout] (padded to 4)
// Every hidden and output row is read as float4 broadcasts along its inputs; the first layer's columns along its
// outputs.  tanh is the accurate tanhf (2 ulp), not tanh.approx.f32 (relative error ~2^-11).
//
// Forward: persistent CTAs, one thread per particle, the 64 activations in registers; z is read once and x written
// once.
//
// Backward: persistent CTAs over tiles of T particles (T = blockDim, one thread per particle).  A tile recomputes its
// forward on chip, keeping every layer's activations in shared memory ([layer][unit][T + 4]: a thread writes its own
// column, the cooperative products below read float4 runs along the particles without bank conflicts), then walks the
// delta chain down: delta_L = (W_out^T gx) * (1 - t_L^2), delta_{l-1} = (W_l^T delta_l) * (1 - t_{l-1}^2), each delta
// overwriting the activations it was made from once they have been used.  The tile's parameter gradients
// (sum over its particles of delta_l t_{l-1}^T) are added to the CTA's own accumulator, in shared memory when it fits
// and otherwise in the CTA's slot of the workspace; nn_reduce_kernel adds the CTAs' partials in CTA order.  Nothing
// per particle besides z, dL/dx and dL/dz touches global memory, there are no floating-point atomics, and repeated
// calls are bitwise equal.  Gradients come out in nn.Linear layout.
#include "common.cuh"

namespace mfb {

constexpr int kNnH = 64;
constexpr int kNnMaxLayers = 8;
constexpr int kNnFwdThreads = 128;
constexpr size_t kNnMaxSmem = 227 * 1024;

struct NnDims {
  int din, dout, layers;
};

__host__ __device__ inline int nn_pad4(int v) { return (v + 3) & ~3; }

// offsets of the weight image (floats)
struct NnImage {
  int w_in, b_in, w_hid, b_hid, w_out, b_out, floats;
};
__host__ __device__ inline NnImage nn_image(const NnDims& d) {
  NnImage m;
  m.w_in = 0;
  m.b_in = d.din * kNnH;
  m.w_hid = m.b_in + kNnH;
  m.b_hid = m.w_hid + (d.layers - 1) * kNnH * kNnH;
  m.w_out = m.b_hid + (d.layers - 1) * kNnH;
  m.b_out = m.w_out + d.dout * kNnH;
  m.floats = m.b_out + nn_pad4(d.dout);
  return m;
}

// gradient accumulators and partials, in the order of the parameters
struct NnGrads {
  int w_in, b_in, w_hid, b_hid, w_out, b_out, floats;
};
__host__ __device__ inline NnGrads nn_grads(const NnDims& d) {
  NnGrads g;
  g.w_in = 0;
  g.b_in = kNnH * d.din;
  g.w_hid = g.b_in + kNnH;
  g.b_hid = g.w_hid + (d.layers - 1) * kNnH * kNnH;
  g.w_out = g.b_hid + (d.layers - 1) * kNnH;
  g.b_out = g.w_out + d.dout * kNnH;
  g.floats = g.b_out + d.dout;
  return g;
}

struct NnParams {
  const float *w_in, *b_in, *w_hid, *b_hid, *w_out, *b_out;
};

__device__ __forceinline__ void nn_load_image(const NnDims& d, const NnParams& p, float* s) {
  const NnImage m = nn_image(d);
  for (int e = threadIdx.x; e < d.din * kNnH; e += blockDim.x) {   // [64][Din] -> [Din][64]
    const int o = e / d.din, i = e - o * d.din;
    s[m.w_in + i * kNnH + o] = p.w_in[e];
  }
  for (int e = threadIdx.x; e < kNnH; e += blockDim.x) s[m.b_in + e] = p.b_in[e];
  for (int e = threadIdx.x; e < (d.layers - 1) * kNnH * kNnH; e += blockDim.x) s[m.w_hid + e] = p.w_hid[e];
  for (int e = threadIdx.x; e < (d.layers - 1) * kNnH; e += blockDim.x) s[m.b_hid + e] = p.b_hid[e];
  for (int e = threadIdx.x; e < d.dout * kNnH; e += blockDim.x) s[m.w_out + e] = p.w_out[e];
  for (int e = threadIdx.x; e < nn_pad4(d.dout); e += blockDim.x) s[m.b_out + e] = e < d.dout ? p.b_out[e] : 0.f;
}

// t = tanh(b + Wt^T z) for the first layer; z_i = zcol[i * zstride]
__device__ __forceinline__ void nn_first_layer(const float* zcol, int zstride, int din, const float* __restrict__ wt,
                                               const float* __restrict__ b, float (&t)[kNnH]) {
#pragma unroll
  for (int o = 0; o < kNnH; o += 4) {
    const float4 bv = *reinterpret_cast<const float4*>(b + o);
    t[o] = bv.x; t[o + 1] = bv.y; t[o + 2] = bv.z; t[o + 3] = bv.w;
  }
  for (int i = 0; i < din; ++i) {
    const float zi = zcol[i * zstride];
#pragma unroll
    for (int o = 0; o < kNnH; o += 4) {
      const float4 w = *reinterpret_cast<const float4*>(wt + i * kNnH + o);
      t[o] = fmaf(zi, w.x, t[o]); t[o + 1] = fmaf(zi, w.y, t[o + 1]);
      t[o + 2] = fmaf(zi, w.z, t[o + 2]); t[o + 3] = fmaf(zi, w.w, t[o + 3]);
    }
  }
#pragma unroll
  for (int o = 0; o < kNnH; ++o) t[o] = tanhf(t[o]);
}

// t = tanh(b + W h), W [64 out][64 in]: eight output rows at a time, four partial sums each
__device__ __forceinline__ void nn_hidden_layer(const float (&h)[kNnH], const float* __restrict__ w,
                                                const float* __restrict__ b, float (&t)[kNnH]) {
#pragma unroll
  for (int ob = 0; ob < kNnH; ob += 8) {
    float acc[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) acc[q] = b[ob + q];
#pragma unroll
    for (int i = 0; i < kNnH; i += 4) {
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        const float4 wv = *reinterpret_cast<const float4*>(w + (ob + q) * kNnH + i);
        acc[q] = fmaf(h[i], wv.x, acc[q]); acc[q] = fmaf(h[i + 1], wv.y, acc[q]);
        acc[q] = fmaf(h[i + 2], wv.z, acc[q]); acc[q] = fmaf(h[i + 3], wv.w, acc[q]);
      }
    }
#pragma unroll
    for (int q = 0; q < 8; ++q) t[ob + q] = tanhf(acc[q]);
  }
}

// b + W h for one 64-long row of W
__device__ __forceinline__ float nn_row_dot(const float (&h)[kNnH], const float* __restrict__ w, float b) {
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
  for (int i = 0; i < kNnH; i += 4) {
    const float4 wv = *reinterpret_cast<const float4*>(w + i);
    a0 = fmaf(h[i], wv.x, a0); a1 = fmaf(h[i + 1], wv.y, a1);
    a2 = fmaf(h[i + 2], wv.z, a2); a3 = fmaf(h[i + 3], wv.w, a3);
  }
  return b + ((a0 + a1) + (a2 + a3));
}

// g += c * W[row], one row of 64
__device__ __forceinline__ void nn_row_axpy(float c, const float* __restrict__ w, float (&g)[kNnH]) {
#pragma unroll
  for (int i = 0; i < kNnH; i += 4) {
    const float4 wv = *reinterpret_cast<const float4*>(w + i);
    g[i] = fmaf(c, wv.x, g[i]); g[i + 1] = fmaf(c, wv.y, g[i + 1]);
    g[i + 2] = fmaf(c, wv.z, g[i + 2]); g[i + 3] = fmaf(c, wv.w, g[i + 3]);
  }
}

__global__ void __launch_bounds__(kNnFwdThreads)
nn_fwd_kernel(const float* __restrict__ z, int64_t n, NnDims d, NnParams prm, float* __restrict__ x) {
  extern __shared__ __align__(16) float smem[];
  pdl_enter();
  nn_load_image(d, prm, smem);
  __syncthreads();
  const NnImage m = nn_image(d);
  const int64_t ntiles = (n + kNnFwdThreads - 1) / kNnFwdThreads;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t p = tile * kNnFwdThreads + threadIdx.x;
    if (p >= n) break;
    float h[kNnH], t[kNnH];
    nn_first_layer(z + p * d.din, 1, d.din, smem + m.w_in, smem + m.b_in, h);
    for (int l = 0; l < d.layers - 1; ++l) {
      nn_hidden_layer(h, smem + m.w_hid + l * kNnH * kNnH, smem + m.b_hid + l * kNnH, t);
#pragma unroll
      for (int j = 0; j < kNnH; ++j) h[j] = t[j];
    }
    for (int k = 0; k < d.dout; ++k) x[p * d.dout + k] = nn_row_dot(h, smem + m.w_out + k * kNnH, smem[m.b_out + k]);
  }
}

// ---- backward --------------------------------------------------------------------------------------------------
// Cooperative tile products over the T particles of shared-memory columns ([row][tp], tp = T + 4):
//   acc[r][c] += sum_p a[r][p] b[c][p]
// The 64 x 64 hidden-layer product is cut into 128 blocks of 4 x 8; block (ob, ib) owns rows ob + 16 q and columns
// ib + 8 r, so the eight threads of a quarter warp read eight different bank groups.
__device__ __forceinline__ void nn_tile_wgrad64(const float* __restrict__ a, const float* __restrict__ bm, int T,
                                                int tp, float* acc) {
  for (int blk = threadIdx.x; blk < 128; blk += blockDim.x) {
    const int ob = blk >> 3, ib = blk & 7;
    float s[4][8];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 8; ++r) s[q][r] = 0.f;
    for (int p = 0; p < T; p += 4) {
      float4 av[4], bv[8];
#pragma unroll
      for (int q = 0; q < 4; ++q) av[q] = *reinterpret_cast<const float4*>(a + (ob + 16 * q) * tp + p);
#pragma unroll
      for (int r = 0; r < 8; ++r) bv[r] = *reinterpret_cast<const float4*>(bm + (ib + 8 * r) * tp + p);
#pragma unroll
      for (int q = 0; q < 4; ++q)
#pragma unroll
        for (int r = 0; r < 8; ++r) {
          s[q][r] = fmaf(av[q].x, bv[r].x, s[q][r]); s[q][r] = fmaf(av[q].y, bv[r].y, s[q][r]);
          s[q][r] = fmaf(av[q].z, bv[r].z, s[q][r]); s[q][r] = fmaf(av[q].w, bv[r].w, s[q][r]);
        }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int r = 0; r < 8; ++r) acc[(ob + 16 * q) * kNnH + ib + 8 * r] += s[q][r];
  }
}

// sum over the tile of one shared-memory row
__device__ __forceinline__ float nn_tile_rowsum(const float* __restrict__ a, int T) {
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  for (int p = 0; p < T; p += 4) {
    const float4 v = *reinterpret_cast<const float4*>(a + p);
    s0 += v.x; s1 += v.y; s2 += v.z; s3 += v.w;
  }
  return (s0 + s1) + (s2 + s3);
}

// sum over the tile of a row times each of `rows` rows of bm (rows <= 8)
__device__ __forceinline__ void nn_tile_rowdots(const float* __restrict__ a, const float* __restrict__ bm, int rows,
                                                int T, int tp, float (&s)[kMaxDim]) {
#pragma unroll
  for (int r = 0; r < kMaxDim; ++r) s[r] = 0.f;
  for (int p = 0; p < T; p += 4) {
    const float4 av = *reinterpret_cast<const float4*>(a + p);
#pragma unroll
    for (int r = 0; r < kMaxDim; ++r) {
      if (r < rows) {
        const float4 bv = *reinterpret_cast<const float4*>(bm + r * tp + p);
        s[r] = fmaf(av.x, bv.x, s[r]); s[r] = fmaf(av.y, bv.y, s[r]);
        s[r] = fmaf(av.z, bv.z, s[r]); s[r] = fmaf(av.w, bv.w, s[r]);
      }
    }
  }
}

__global__ void __launch_bounds__(128)
nn_bwd_kernel(const float* __restrict__ z, const float* __restrict__ gx, int64_t n, NnDims d, NnParams prm,
              int acc_in_smem, float* __restrict__ gz, float* __restrict__ partials) {
  extern __shared__ __align__(16) float smem[];
  const int T = blockDim.x, tp = T + 4, tid = threadIdx.x;
  const NnImage m = nn_image(d);
  const NnGrads gl = nn_grads(d);
  float* act = smem + m.floats;                          // [L][64][tp]
  float* zs = act + (size_t)d.layers * kNnH * tp;        // [Din][tp]
  float* gxs = zs + d.din * tp;                          // [Dout][tp]
  float* acc = acc_in_smem ? gxs + d.dout * tp : partials + (size_t)blockIdx.x * gl.floats;
  pdl_enter();
  nn_load_image(d, prm, smem);
  for (int e = tid; e < gl.floats; e += T) acc[e] = 0.f;
  __syncthreads();

  const int64_t ntiles = (n + T - 1) / T;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t p = tile * T + tid;
    const bool valid = p < n;
    // padding particles: z = 0 and dL/dx = 0, so every delta of theirs is 0 and they add nothing
    for (int i = 0; i < d.din; ++i) zs[i * tp + tid] = valid ? z[p * d.din + i] : 0.f;
    for (int k = 0; k < d.dout; ++k) gxs[k * tp + tid] = valid ? gx[p * d.dout + k] : 0.f;

    // forward, activations to the thread's columns
    float h[kNnH], g[kNnH];
    nn_first_layer(zs + tid, tp, d.din, smem + m.w_in, smem + m.b_in, h);
#pragma unroll
    for (int j = 0; j < kNnH; ++j) act[j * tp + tid] = h[j];
    for (int l = 1; l < d.layers; ++l) {
      nn_hidden_layer(h, smem + m.w_hid + (l - 1) * kNnH * kNnH, smem + m.b_hid + (l - 1) * kNnH, g);
      float* col = act + (size_t)l * kNnH * tp + tid;
#pragma unroll
      for (int j = 0; j < kNnH; ++j) {
        h[j] = g[j];
        col[j * tp] = g[j];
      }
    }
    __syncthreads();

    // output layer: dW_out[k][i] = sum_p gx[k] t_L[i], db_out[k] = sum_p gx[k]
    const float* tl = act + (size_t)(d.layers - 1) * kNnH * tp;
    for (int i = tid; i < kNnH; i += T) {
      float s[kMaxDim];
      nn_tile_rowdots(tl + i * tp, gxs, d.dout, T, tp, s);
#pragma unroll
      for (int k = 0; k < kMaxDim; ++k)
        if (k < d.dout) acc[gl.w_out + k * kNnH + i] += s[k];
    }
    for (int k = tid; k < d.dout; k += T) acc[gl.b_out + k] += nn_tile_rowsum(gxs + k * tp, T);
    // delta_L = (W_out^T gx) (1 - t_L^2)
#pragma unroll
    for (int j = 0; j < kNnH; ++j) g[j] = 0.f;
    for (int k = 0; k < d.dout; ++k) nn_row_axpy(gxs[k * tp + tid], smem + m.w_out + k * kNnH, g);
#pragma unroll
    for (int j = 0; j < kNnH; ++j) h[j] = g[j] * fmaf(-h[j], h[j], 1.f);
    __syncthreads();
    {
      float* col = act + (size_t)(d.layers - 1) * kNnH * tp + tid;
#pragma unroll
      for (int j = 0; j < kNnH; ++j) col[j * tp] = h[j];
    }

    // hidden layers, last to first: h holds delta_l, slot l-1 delta_l, slot l-2 t_{l-1}
    for (int l = d.layers; l >= 2; --l) {
      const float* dl = act + (size_t)(l - 1) * kNnH * tp;
      float* tprev = act + (size_t)(l - 2) * kNnH * tp;
      const float* w = smem + m.w_hid + (l - 2) * kNnH * kNnH;
      __syncthreads();
      nn_tile_wgrad64(dl, tprev, T, tp, acc + gl.w_hid + (l - 2) * kNnH * kNnH);
      for (int o = tid; o < kNnH; o += T) acc[gl.b_hid + (l - 2) * kNnH + o] += nn_tile_rowsum(dl + o * tp, T);
#pragma unroll
      for (int j = 0; j < kNnH; ++j) g[j] = 0.f;
#pragma unroll
      for (int o = 0; o < kNnH; ++o) nn_row_axpy(h[o], w + o * kNnH, g);
#pragma unroll
      for (int j = 0; j < kNnH; ++j) {
        const float t = tprev[j * tp + tid];
        h[j] = g[j] * fmaf(-t, t, 1.f);
      }
      __syncthreads();
#pragma unroll
      for (int j = 0; j < kNnH; ++j) tprev[j * tp + tid] = h[j];
    }
    __syncthreads();

    // first layer: dW_in[o][i] = sum_p delta_1[o] z[i], db_in[o] = sum_p delta_1[o]; dL/dz = W_in^T delta_1
    for (int o = tid; o < kNnH; o += T) {
      float s[kMaxDim];
      nn_tile_rowdots(act + o * tp, zs, d.din, T, tp, s);
#pragma unroll
      for (int i = 0; i < kMaxDim; ++i)
        if (i < d.din) acc[gl.w_in + o * d.din + i] += s[i];
      acc[gl.b_in + o] += nn_tile_rowsum(act + o * tp, T);
    }
    if (gz && valid) {
      for (int i = 0; i < d.din; ++i) {
        const float* wt = smem + m.w_in + i * kNnH;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
        for (int o = 0; o < kNnH; o += 4) {
          const float4 wv = *reinterpret_cast<const float4*>(wt + o);
          a0 = fmaf(h[o], wv.x, a0); a1 = fmaf(h[o + 1], wv.y, a1);
          a2 = fmaf(h[o + 2], wv.z, a2); a3 = fmaf(h[o + 3], wv.w, a3);
        }
        gz[p * d.din + i] = (a0 + a1) + (a2 + a3);
      }
    }
    __syncthreads();
  }
  if (acc_in_smem) {
    float* dst = partials + (size_t)blockIdx.x * gl.floats;
    for (int e = tid; e < gl.floats; e += T) dst[e] = acc[e];
  }
}

// adds the CTAs' partials in CTA order and scatters them to the six gradient tensors
__global__ void nn_reduce_kernel(const float* __restrict__ partials, int nparts, NnDims d, float* __restrict__ gw_in,
                                 float* __restrict__ gb_in, float* __restrict__ gw_hid, float* __restrict__ gb_hid,
                                 float* __restrict__ gw_out, float* __restrict__ gb_out) {
  pdl_enter();
  const NnGrads gl = nn_grads(d);
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= gl.floats) return;
  float s = 0.f;
  for (int c = 0; c < nparts; ++c) s += partials[(size_t)c * gl.floats + e];
  if (e < gl.b_in) gw_in[e] = s;
  else if (e < gl.w_hid) gb_in[e - gl.b_in] = s;
  else if (e < gl.b_hid) gw_hid[e - gl.w_hid] = s;
  else if (e < gl.w_out) gb_hid[e - gl.b_hid] = s;
  else if (e < gl.b_out) gw_out[e - gl.w_out] = s;
  else gb_out[e - gl.b_out] = s;
}

static bool nn_supported(int din, int dout, int hidden_units, int hidden_layers) {
  return din >= 1 && din <= kMaxDim && dout >= 1 && dout <= kMaxDim && hidden_units == kNnH && hidden_layers >= 1 &&
         hidden_layers <= kNnMaxLayers;
}

static size_t nn_fwd_smem(const NnDims& d) { return (size_t)nn_image(d).floats * 4; }

// Backward launch plan: the largest tile (128, 64 or 32 particles) whose activations fit beside the weights, the
// gradient accumulator in shared memory when it still fits, and as many CTAs as are resident at once (one partial
// each), but no more than there are tiles.
struct NnBwdPlan {
  int threads, acc_in_smem, grid;
  size_t smem;
};

static int nn_bwd_plan(int64_t n, const NnDims& d, NnBwdPlan& p) {
  const size_t wbytes = (size_t)nn_image(d).floats * 4;
  const size_t gbytes = (size_t)nn_grads(d).floats * 4;
  p.threads = 0;
  for (int t = 128; t >= 32; t >>= 1) {
    const size_t s = wbytes + (size_t)(d.layers * kNnH + d.din + d.dout) * (t + 4) * 4;
    if (s <= kNnMaxSmem) {
      p.threads = t;
      p.acc_in_smem = s + gbytes <= kNnMaxSmem;
      p.smem = p.acc_in_smem ? s + gbytes : s;
      break;
    }
  }
  if (!p.threads) return MFB_E_UNSUPPORTED;
  MFB_CUDA(cudaFuncSetAttribute(nn_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  int per_sm = 0;
  MFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nn_bwd_kernel, p.threads, p.smem));
  const int64_t ntiles = (n + p.threads - 1) / p.threads;
  int64_t grid = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 1);
  p.grid = (int)(grid < ntiles ? grid : ntiles);
  return 0;
}

}  // namespace mfb

using namespace mfb;

extern "C" {

int mfb_nn_supported(int din, int dout, int hidden_units, int hidden_layers) {
  return nn_supported(din, dout, hidden_units, hidden_layers) ? 1 : 0;
}

int mfb_nn_fwd(const float* z, int64_t n, int din, int dout, int hidden_units, int hidden_layers, const float* w_in,
               const float* b_in, const float* w_hid, const float* b_hid, const float* w_out, const float* b_out,
               float* x, void* stream) {
  MFB_CHECK_ARG(z && w_in && b_in && w_out && b_out && x && n >= 1);
  if (!nn_supported(din, dout, hidden_units, hidden_layers)) return MFB_E_UNSUPPORTED;
  MFB_CHECK_ARG(hidden_layers == 1 || (w_hid && b_hid));
  const NnDims d = {din, dout, hidden_layers};
  const NnParams prm = {w_in, b_in, w_hid, b_hid, w_out, b_out};
  const size_t smem = nn_fwd_smem(d);
  MFB_CUDA(cudaFuncSetAttribute(nn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 0;
  MFB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, nn_fwd_kernel, kNnFwdThreads, smem));
  const int64_t ntiles = (n + kNnFwdThreads - 1) / kNnFwdThreads;
  int64_t grid = (int64_t)sm_count() * (per_sm > 0 ? per_sm : 1);
  if (grid > ntiles) grid = ntiles;
  MFB_CUDA(launch_pdl(nn_fwd_kernel, dim3((unsigned)grid), dim3(kNnFwdThreads), smem, (cudaStream_t)stream, z, n, d,
                      prm, x));
  return launch_status();
}

int64_t mfb_nn_bwd_workspace_bytes(int64_t n, int din, int dout, int hidden_units, int hidden_layers) {
  if (n < 1 || !nn_supported(din, dout, hidden_units, hidden_layers)) return 0;
  const NnDims d = {din, dout, hidden_layers};
  NnBwdPlan p;
  if (nn_bwd_plan(n, d, p)) return 0;
  return (int64_t)p.grid * nn_grads(d).floats * 4;
}

int mfb_nn_bwd(const float* z, const float* gx, int64_t n, int din, int dout, int hidden_units, int hidden_layers,
               const float* w_in, const float* b_in, const float* w_hid, const float* b_hid, const float* w_out,
               const float* b_out, float* gz, float* gw_in, float* gb_in, float* gw_hid, float* gb_hid, float* gw_out,
               float* gb_out, void* workspace, int64_t workspace_bytes, void* stream) {
  MFB_CHECK_ARG(z && gx && w_in && b_in && w_out && b_out && gw_in && gb_in && gw_out && gb_out && workspace &&
                n >= 1);
  if (!nn_supported(din, dout, hidden_units, hidden_layers)) return MFB_E_UNSUPPORTED;
  MFB_CHECK_ARG(hidden_layers == 1 || (w_hid && b_hid && gw_hid && gb_hid));
  const NnDims d = {din, dout, hidden_layers};
  const NnParams prm = {w_in, b_in, w_hid, b_hid, w_out, b_out};
  NnBwdPlan p;
  int rc = nn_bwd_plan(n, d, p);
  if (rc) return rc;
  const int gfloats = nn_grads(d).floats;
  if (workspace_bytes < (int64_t)p.grid * gfloats * 4) return MFB_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* partials = (float*)workspace;
  MFB_CUDA(launch_pdl(nn_bwd_kernel, dim3((unsigned)p.grid), dim3(p.threads), p.smem, st, z, gx, n, d, prm,
                      p.acc_in_smem, gz, partials));
  MFB_CUDA(launch_pdl(nn_reduce_kernel, dim3((unsigned)((gfloats + 255) / 256)), dim3(256), 0, st,
                      (const float*)partials, p.grid, d, gw_in, gb_in, gw_hid, gb_hid, gw_out, gb_out));
  return launch_status();
}

}  // extern "C"
