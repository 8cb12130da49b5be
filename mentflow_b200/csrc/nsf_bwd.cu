// Backward of one neural-spline-flow layer (hand-written; replaces torch autograd through zuko's
// MaskedMLP + MonotonicRQSTransform graph, which stores ~10.9 KB of activations per particle).
//
// Nothing from the forward pass is kept except the layer input v (24 B/particle): activations
// are recomputed.  Pipeline of one call (all buffers feature-major [row][N] so that every
// access along the particle axis is coalesced):
//
//   1. nsf_bwd_spline_kernel   recompute MLP (weights in smem, thread per particle), write the
//                              post-ReLU activations h_l, run the spline forward+backward per
//                              feature -> gphi [D*64][N] (gradient w.r.t. the raw conditioner
//                              outputs, incl. softmax / soft-clip Jacobians) and the direct
//                              gradient w.r.t. v through the spline (+ base-density term).
//   2. per MLP layer, last to first:
//        wgrad  dW[in][out] = sum_p h[in][p] g[out][p]     (split over particles, fixed-order reduce)
//        bgrad  db[out]     = sum_p g[out][p]
//        dgrad  g_prev[in][p] = (h[in][p] > 0) * sum_out W[out][in] g[out][p]
//   3. nsf_bwd_input_kernel    gv = direct + W1^T g1.
//
// Gradients land directly in the packed parameter layout of the forward kernel, so the host
// maps them back to zuko-layout tensors (and applies the masks) by plain autograd through
// NSFGenerator.packed_parameters().
#include "nsf_tc_common.cuh"

namespace mfb {

constexpr int kBwdThreads = 256;

// ---- 1. recompute + spline backward ---------------------------------------------------------
// Spline forward+backward for one feature.  col[j*stride]: raw parameters in, gradient w.r.t. the
// raw parameters out (in place).  gy = dL/dy, gl = dL/d(ladj).  Returns dL/dv (direct).
__device__ __forceinline__ float rq_spline_backward(float* col, int stride, int nb, float v, float gy, float gl) {
  const int ptotal = 3 * nb - 1;
  // raw -> clipped (in place), remember nothing: the clip derivative is recomputed from raw via
  // c = r / (1 + a|r|)  =>  1 + a|r| = 1 / (1 - a|c|)  =>  dc/dr = (1 - a|c|)^2
  float mw = -INFINITY, mh = -INFINITY;
  for (int j = 0; j < nb; ++j) {
    float r = col[j * stride];
    r = r / (1.0f + kClipW * fabsf(r));
    col[j * stride] = r;
    mw = fmaxf(mw, r);
    float q = col[(nb + j) * stride];
    q = q / (1.0f + kClipW * fabsf(q));
    col[(nb + j) * stride] = q;
    mh = fmaxf(mh, q);
  }
  // knot sums in double (see knot_search in nsf_common.cuh); the exponentials are recomputed where
  // they are needed instead of being stored (col holds the clipped parameters for the clip derivative)
  const bool inside = v > -kBound && v <= kBound;
  if (!inside) {  // identity outside the spline box: no parameter gradient
    for (int j = 0; j < ptotal; ++j) col[j * stride] = 0.f;
    return gy;
  }
  double swd = 0.0, shd = 0.0;
  for (int j = 0; j < nb; ++j) {
    swd += (double)expf(col[j * stride] - mw);
    shd += (double)expf(col[(nb + j) * stride] - mh);
  }
  const float sw = (float)swd, sh = (float)shd;
  const double target = ((double)v + (double)kBound) * (0.5 / (double)kBound) * swd;
  double cumd = 0.0;
  int kbin = nb - 1;
  for (int j = 0; j < nb - 1; ++j) {
    const double nxt = cumd + (double)expf(col[j * stride] - mw);
    if (target <= nxt) {
      kbin = j;
      break;
    }
    cumd = nxt;
  }
  const float ekw = expf(col[kbin * stride] - mw);
  const float wk = (float)((double)ekw / swd);
  const float x0 = (float)(2.0 * (double)kBound * (cumd / swd) - (double)kBound);
  double cumhd = 0.0;
  for (int j = 0; j < kbin; ++j) cumhd += (double)expf(col[(nb + j) * stride] - mh);
  const float cumh = (float)(cumhd / shd);
  const float hk = (float)((double)expf(col[(nb + kbin) * stride] - mh) / shd);
  float* cold = col + 2 * nb * stride;
  float d0 = 1.0f, d1 = 1.0f, c0 = 0.f, c1 = 0.f;
  if (kbin > 0) {
    const float r = cold[(kbin - 1) * stride];
    c0 = r / (1.0f + kClipD * fabsf(r));
    d0 = expf(c0);
  }
  if (kbin < nb - 1) {
    const float r = cold[kbin * stride];
    c1 = r / (1.0f + kClipD * fabsf(r));
    d1 = expf(c1);
  }
  const float dx = 2.0f * kBound * wk, dy = 2.0f * kBound * hk;
  const float s = hk / wk;
  float t = (float)((target - cumd) / (double)ekw);
  t = fminf(fmaxf(t, 0.0f), 1.0f);
  const float omt = 1.0f - t, q = t * omt;
  const float A = d0 + d1 - 2.0f * s;
  const float den = fmaf(A, q, s);
  const float n1 = s * t * t + d0 * q;
  const float n2 = 2.0f * s * q + d0 * omt * omt + d1 * t * t;
  // partial derivatives (scripts/proto_spline_bwd.py is the float64 prototype of this block)
  const float dq_dt = 1.0f - 2.0f * t;
  const float dden_dt = A * dq_dt, dden_ds = 1.0f - 2.0f * q, dden_dd = q;
  const float r1 = n1 / den;
  const float inv_den = 1.0f / den, inv_n2 = 1.0f / n2;
  const float dy_dt = dy * (2.0f * s * t + d0 * dq_dt - r1 * dden_dt) * inv_den;
  const float dy_ds = dy * (t * t - r1 * dden_ds) * inv_den;
  const float dy_dd0 = dy * (q - r1 * dden_dd) * inv_den;
  const float dy_dd1 = dy * (-r1 * dden_dd) * inv_den;
  const float dl_dt = (2.0f * s * dq_dt - 2.0f * d0 * omt + 2.0f * d1 * t) * inv_n2 - 2.0f * dden_dt * inv_den;
  const float dl_ds = 2.0f / s + 2.0f * q * inv_n2 - 2.0f * dden_ds * inv_den;
  const float dl_dd0 = omt * omt * inv_n2 - 2.0f * dden_dd * inv_den;
  const float dl_dd1 = t * t * inv_n2 - 2.0f * dden_dd * inv_den;
  const float g_t = gy * dy_dt + gl * dl_dt;
  const float g_s = gy * dy_ds + gl * dl_ds;
  const float g_d0 = gy * dy_dd0 + gl * dl_dd0;
  const float g_d1 = gy * dy_dd1 + gl * dl_dd1;
  const float g_dy = gy * r1;
  const float gv = g_t / dx;
  const float g_x0 = -gv;
  const float g_dx = -g_t * t / dx;
  // gradients w.r.t. the normalised widths / heights
  const float gW_lo = 2.0f * kBound * g_x0;                  // j < k
  const float gW_k = 2.0f * kBound * g_dx - g_s * s / wk;    // j = k
  const float gH_lo = 2.0f * kBound * gy;                    // j < k   (dL/dy0 = gy)
  const float gH_k = 2.0f * kBound * g_dy + g_s / wk;
  // softmax backward needs dot = sum_j gW_j W_j
  const float cumw_lo = (x0 + kBound) / (2.0f * kBound);     // sum_{j<k} W_j
  const float dotW = gW_lo * cumw_lo + gW_k * wk;
  const float dotH = gH_lo * cumh + gH_k * hk;
  for (int j = 0; j < nb; ++j) {
    const float cw = col[j * stride];
    const float Wj = expf(cw - mw) / sw;
    const float gj = (j < kbin ? gW_lo : (j == kbin ? gW_k : 0.f)) - dotW;
    const float a = 1.0f - kClipW * fabsf(cw);
    col[j * stride] = Wj * gj * a * a;
    const float ch = col[(nb + j) * stride];
    const float Hj = expf(ch - mh) / sh;
    const float gh = (j < kbin ? gH_lo : (j == kbin ? gH_k : 0.f)) - dotH;
    const float b = 1.0f - kClipW * fabsf(ch);
    col[(nb + j) * stride] = Hj * gh * b * b;
  }
  for (int j = 0; j < nb - 1; ++j) {
    float g = 0.f;
    if (j == kbin - 1) {
      const float a = 1.0f - kClipD * fabsf(c0);
      g = g_d0 * d0 * a * a;
    } else if (j == kbin) {
      const float a = 1.0f - kClipD * fabsf(c1);
      g = g_d1 * d1 * a * a;
    }
    cold[j * stride] = g;
  }
  return gv;
}

template <int D>
__global__ void __launch_bounds__(kNsfThreads, 1)
nsf_bwd_spline_kernel(const float* __restrict__ v, const float* __restrict__ gy, const float* __restrict__ glogq,
                      int64_t n, int hidden_layers, int nb, const float* __restrict__ params, int64_t nparams,
                      FeatureOrder order, int first_layer, float* __restrict__ acts /* [L][64][n] */,
                      float* __restrict__ gphi /* [D*64][n] */, float* __restrict__ gvd /* [n][D] */,
                      float* __restrict__ gmax /* [n]: max |gphi| of the particle (row scale of the tcgen05 dgrad) */,
                      int* __restrict__ gmaxes /* [0]: batch maximum of |gphi| as float bits (atomicMax) */) {
  extern __shared__ __align__(16) float smem[];
  float* s_par = smem;
  float* s_scr = smem + ((nparams + 3) & ~(int64_t)3);
  const int tid = threadIdx.x;
  {
    const float4* src = reinterpret_cast<const float4*>(params);
    float4* dst = reinterpret_cast<float4*>(s_par);
    for (int i = tid; i < (int)(nparams >> 2); i += kNsfThreads) dst[i] = src[i];
    for (int i = (int)(nparams & ~(int64_t)3) + tid; i < (int)nparams; i += kNsfThreads) s_par[i] = params[i];
  }
  __syncthreads();
  const float* W1t = s_par;
  const float* b1 = W1t + D * kH;
  const float* hid = b1 + kH;
  const float* Wout = hid + (size_t)(hidden_layers - 1) * (kH * kH + kH);
  const float* bout = Wout + (size_t)D * kH * kPP;
  float* col = s_scr + tid;
  const int ptotal = 3 * nb - 1;

  const int64_t ntiles = (n + kNsfThreads - 1) / kNsfThreads;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t p = tile * kNsfThreads + tid;
    const bool valid = p < n;
    float vin[D], gyv[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      vin[i] = valid ? v[p * D + i] : 0.f;
      gyv[i] = valid ? gy[p * D + i] : 0.f;
    }
    const float glq = (valid && glogq) ? glogq[p] : 0.f;

    float h[kH];
#pragma unroll
    for (int j4 = 0; j4 < kH / 4; ++j4) {
      float4 acc = *reinterpret_cast<const float4*>(b1 + 4 * j4);
#pragma unroll
      for (int i = 0; i < D; ++i) {
        const float4 w = *reinterpret_cast<const float4*>(W1t + i * kH + 4 * j4);
        acc.x = fmaf(vin[i], w.x, acc.x); acc.y = fmaf(vin[i], w.y, acc.y);
        acc.z = fmaf(vin[i], w.z, acc.z); acc.w = fmaf(vin[i], w.w, acc.w);
      }
      h[4 * j4 + 0] = fmaxf(acc.x, 0.f); h[4 * j4 + 1] = fmaxf(acc.y, 0.f);
      h[4 * j4 + 2] = fmaxf(acc.z, 0.f); h[4 * j4 + 3] = fmaxf(acc.w, 0.f);
    }
    if (valid) {
#pragma unroll
      for (int j = 0; j < kH; ++j) acts[(size_t)j * n + p] = h[j];
    }
    for (int l = 0; l < hidden_layers - 1; ++l) {
      const float* wt = hid + (size_t)l * (kH * kH + kH);
      const float* bias = wt + kH * kH;
#pragma unroll 1
      for (int jc = 0; jc < kH / 8; ++jc) {
        float acc[8];
        dense8(h, wt + jc * 8, bias + jc * 8, acc);
#pragma unroll
        for (int qq = 0; qq < 8; ++qq) col[(jc * 8 + qq) * kNsfThreads] = fmaxf(acc[qq], 0.f);
      }
      float* a_out = acts + (size_t)(l + 1) * kH * n;
#pragma unroll
      for (int j = 0; j < kH; ++j) {
        h[j] = col[j * kNsfThreads];
        if (valid) a_out[(size_t)j * n + p] = h[j];
      }
    }
    float gvo[D];
    float amax = 0.f;
#pragma unroll 1
    for (int f = 0; f < D; ++f) {
      const float* bf = bout + f * kPP;
      if (order.v[f] == 0) {
        for (int j = 0; j < ptotal; ++j) col[j * kNsfThreads] = bf[j];
      } else {
        const float* wf = Wout + (size_t)f * kH * kPP;
        const int nchunk = (ptotal + 7) >> 3;
#pragma unroll 1
        for (int jc = 0; jc < nchunk; ++jc) {
          float acc[8];
          dense8(h, wf + jc * 8, bf + jc * 8, acc);
#pragma unroll
          for (int qq = 0; qq < 8; ++qq) col[(jc * 8 + qq) * kNsfThreads] = acc[qq];
        }
      }
      float vf = vin[0], gyf = gyv[0];
#pragma unroll
      for (int i = 1; i < D; ++i) {
        vf = (f == i) ? vin[i] : vf;
        gyf = (f == i) ? gyv[i] : gyf;
      }
      // logq_out = logq_in - ladj  =>  dL/d(ladj) = -dL/dlogq
      float g = rq_spline_backward(col, kNsfThreads, nb, vf, gyf, -glq);
      if (first_layer) g -= glq * vf;  // d/dv of log N(v; 0, I)
#pragma unroll
      for (int i = 0; i < D; ++i)
        if (f == i) gvo[i] = g;
      if (valid) {
        float* gp = gphi + (size_t)f * kPP * n + p;
        for (int j = 0; j < ptotal; ++j) {
          const float gj = col[j * kNsfThreads];
          gp[(size_t)j * n] = gj;
          amax = fmaxf(amax, fabsf(gj));
        }
        for (int j = ptotal; j < kPP; ++j) gp[(size_t)j * n] = 0.f;
      }
    }
    if (valid) {
#pragma unroll
      for (int i = 0; i < D; ++i) gvd[p * D + i] = gvo[i];
      if (gmax) gmax[p] = amax;
    }
    if (gmaxes) {
      float wm = valid ? amax : 0.f;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
      if ((tid & 31) == 0) atomicMax(gmaxes, __float_as_int(wm));
    }
  }
}

// ---- 2a. dgrad: out[i][p] = (hprev[i][p] > 0) * sum_m Wom[m][i] g[m][p] -------------------------------
// Wom = out-major weights [M][64] (M = rows of g).  Thread per particle, 64 accumulators.
__global__ void __launch_bounds__(kBwdThreads)
nsf_dgrad_kernel(const float* __restrict__ g, int M, int64_t n, const float* __restrict__ wom,
                 const float* __restrict__ hprev, float* __restrict__ out) {
  extern __shared__ __align__(16) float s_w[];  // [mchunk][64]
  constexpr int kChunk = 128;
  for (int64_t p0 = (int64_t)blockIdx.x * kBwdThreads; p0 < n; p0 += (int64_t)gridDim.x * kBwdThreads) {
    const int64_t p = p0 + threadIdx.x;
    const bool valid = p < n;
    float acc[kH];
#pragma unroll
    for (int i = 0; i < kH; ++i) acc[i] = 0.f;
    for (int m0 = 0; m0 < M; m0 += kChunk) {
      const int mc = (M - m0 < kChunk) ? (M - m0) : kChunk;
      __syncthreads();
      for (int i = threadIdx.x; i < mc * (kH / 4); i += kBwdThreads)
        reinterpret_cast<float4*>(s_w)[i] = reinterpret_cast<const float4*>(wom + (size_t)m0 * kH)[i];
      __syncthreads();
      for (int m = 0; m < mc; ++m) {
        const float gm = valid ? g[(size_t)(m0 + m) * n + p] : 0.f;
        const float* wr = s_w + m * kH;
#pragma unroll
        for (int i4 = 0; i4 < kH / 4; ++i4) {
          const float4 w = *reinterpret_cast<const float4*>(wr + 4 * i4);
          acc[4 * i4 + 0] = fmaf(w.x, gm, acc[4 * i4 + 0]);
          acc[4 * i4 + 1] = fmaf(w.y, gm, acc[4 * i4 + 1]);
          acc[4 * i4 + 2] = fmaf(w.z, gm, acc[4 * i4 + 2]);
          acc[4 * i4 + 3] = fmaf(w.w, gm, acc[4 * i4 + 3]);
        }
      }
    }
    if (valid) {
#pragma unroll
      for (int i = 0; i < kH; ++i) out[(size_t)i * n + p] = hprev[(size_t)i * n + p] > 0.f ? acc[i] : 0.f;
    }
  }
}

// ---- 2b. wgrad: C[i][j] = sum_p A[i][p] B[j][p], i < 64, j in a 64-column block ------------------
// grid = (nsplit, ncolblocks).  256 threads, thread (ti, tj) of 16x16 owns rows ti+16a, cols tj+16b.
constexpr int kWgTileP = 32;
constexpr int kWgLd = kWgTileP + 4;

__global__ void __launch_bounds__(256)
nsf_wgrad_kernel(const float* __restrict__ A, const float* __restrict__ B, int64_t n, int64_t per_split,
                 float* __restrict__ partial /* [nsplit][ncolblocks][64][64] */) {
  __shared__ __align__(16) float As[kH * kWgLd];
  __shared__ __align__(16) float Bs[kH * kWgLd];
  const int tid = threadIdx.x, ti = tid >> 4, tj = tid & 15;
  const int cb = blockIdx.y;
  const float* Bb = B + (size_t)cb * kH * n;
  const int64_t pbeg = (int64_t)blockIdx.x * per_split;
  int64_t pend = pbeg + per_split;
  if (pend > n) pend = n;
  float acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.f;
  for (int64_t p0 = pbeg; p0 < pend; p0 += kWgTileP) {
    __syncthreads();
    // 64 rows x 32 particles per matrix: 2048 floats, 8 per thread
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const int idx = tid + r * 256;
      const int row = idx >> 5, pp = idx & 31;
      const int64_t p = p0 + pp;
      const bool ok = p < pend;
      As[row * kWgLd + pp] = ok ? A[(size_t)row * n + p] : 0.f;
      Bs[row * kWgLd + pp] = ok ? Bb[(size_t)row * n + p] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int p4 = 0; p4 < kWgTileP; p4 += 4) {
      float4 av[4], bv[4];
#pragma unroll
      for (int a = 0; a < 4; ++a) av[a] = *reinterpret_cast<const float4*>(As + (ti + 16 * a) * kWgLd + p4);
#pragma unroll
      for (int b = 0; b < 4; ++b) bv[b] = *reinterpret_cast<const float4*>(Bs + (tj + 16 * b) * kWgLd + p4);
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) {
          acc[a][b] = fmaf(av[a].x, bv[b].x, acc[a][b]);
          acc[a][b] = fmaf(av[a].y, bv[b].y, acc[a][b]);
          acc[a][b] = fmaf(av[a].z, bv[b].z, acc[a][b]);
          acc[a][b] = fmaf(av[a].w, bv[b].w, acc[a][b]);
        }
    }
  }
  float* out = partial + ((size_t)blockIdx.x * gridDim.y + cb) * kH * kH;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) out[(ti + 16 * a) * kH + tj + 16 * b] = acc[a][b];
}

// out[cb][i][j] (+)= sum_s partial[s][cb][i][j]; out block cb starts at out + cb*block_stride
__global__ void nsf_wgrad_reduce_kernel(const float* __restrict__ partial, int nsplit, int ncb, int64_t block_stride,
                                        float* __restrict__ out, int accumulate) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= ncb * kH * kH) return;
  const int cb = idx / (kH * kH), e = idx % (kH * kH);
  float s = 0.f;
  for (int k = 0; k < nsplit; ++k) s += partial[((size_t)k * ncb + cb) * kH * kH + e];
  float* o = out + (size_t)cb * block_stride + e;
  *o = accumulate ? *o + s : s;
}

// ---- 2c. bias grad: out[r] (+)= sum_p g[r][p]: one CTA per row, fixed-order block reduction -------
__global__ void __launch_bounds__(256)
nsf_rowsum_kernel(const float* __restrict__ g, int64_t n, float* __restrict__ out, int out_stride_rows,
                  int rows_per_group, int group_pad, int accumulate) {
  // row r of g maps to out[(r / rows_per_group) * (rows_per_group + group_pad) + r % rows_per_group]
  __shared__ double red[8];
  const int r = blockIdx.x;
  double s = 0.0;
  for (int64_t p = threadIdx.x; p < n; p += 256) s += (double)g[(size_t)r * n + p];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    (void)out_stride_rows;
    float* o = out + (size_t)(r / rows_per_group) * (rows_per_group + group_pad) + (r % rows_per_group);
    *o = accumulate ? *o + (float)t : (float)t;
  }
}

// ---- 2d. first-layer weight grad: dW1t[d][j] = sum_p v[p][d] g1[j][p] --------------------------------
template <int D>
__global__ void __launch_bounds__(256)
nsf_wgrad_in_kernel(const float* __restrict__ v, const float* __restrict__ g1, int64_t n, int64_t per_cta,
                    float* __restrict__ partial /* [grid][D][64] */) {
  __shared__ float s_acc[8][D * kH];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = lane; i < D * kH; i += 32) s_acc[warp][i] = 0.f;
  __syncwarp();
  const int64_t pbeg = (int64_t)blockIdx.x * per_cta;
  int64_t pend = pbeg + per_cta;
  if (pend > n) pend = n;
  for (int64_t p0 = pbeg + warp * 32; p0 < pend; p0 += 256) {
    const int64_t p = p0 + lane;
    const bool ok = p < pend;
    float vr[D];
#pragma unroll
    for (int d = 0; d < D; ++d) vr[d] = ok ? v[p * D + d] : 0.f;
    for (int j = 0; j < kH; ++j) {
      const float g = ok ? g1[(size_t)j * n + p] : 0.f;
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const float s = warp_sum(vr[d] * g);
        if (lane == 0) s_acc[warp][d * kH + j] += s;
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < D * kH; i += 256) {
    float s = 0.f;
    for (int w = 0; w < 8; ++w) s += s_acc[w][i];
    partial[(size_t)blockIdx.x * D * kH + i] = s;
  }
}

__global__ void nsf_sum_partials_kernel(const float* __restrict__ partial, int nparts, int len, float* __restrict__ out,
                                        int accumulate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= len) return;
  float s = 0.f;
  for (int k = 0; k < nparts; ++k) s += partial[(size_t)k * len + i];
  out[i] = accumulate ? out[i] + s : s;
}

// ---- 3. input gradient: gv[p][d] = gvd[p][d] + sum_j W1om[j][d] g1[j][p] ------------------------------
template <int D>
__global__ void __launch_bounds__(256)
nsf_bwd_input_kernel(const float* __restrict__ gvd, const float* __restrict__ g1, int64_t n,
                     const float* __restrict__ w1om /* [64][D] */, float* __restrict__ gv) {
  __shared__ float s_w[kH * D];
  for (int i = threadIdx.x; i < kH * D; i += 256) s_w[i] = w1om[i];
  __syncthreads();
  for (int64_t p = (int64_t)blockIdx.x * 256 + threadIdx.x; p < n; p += (int64_t)gridDim.x * 256) {
    float acc[D];
#pragma unroll
    for (int d = 0; d < D; ++d) acc[d] = gvd[p * D + d];
    for (int j = 0; j < kH; ++j) {
      const float g = g1[(size_t)j * n + p];
#pragma unroll
      for (int d = 0; d < D; ++d) acc[d] = fmaf(s_w[j * D + d], g, acc[d]);
    }
#pragma unroll
    for (int d = 0; d < D; ++d) gv[p * D + d] = acc[d];
  }
}


// ---- host-side orchestration of one layer ----------------------------------------------------------------
// tcgen05 data-gradient chain (nsf_tc_bwd.cu); MFB_E_UNSUPPORTED for shapes it is not compiled for
int64_t nsf_tc_dgrad_image_bytes(int d);
int nsf_tc_dgrad(const float* gphi, const float* gmax, const uint32_t* masks, const float* gvd, int64_t n, int d,
                 int hidden_layers, const float* params, const int32_t* order, float* gz, float* gv, void* image,
                 int* gmaxes, cudaStream_t st);
// tcgen05 weight + bias gradients of the whole layer (nsf_tc_bwd.cu)
int64_t nsf_tc_wgrad_partial_floats(int d);
int nsf_tc_wgrad(const float* gphi, const float* gz, const float* acts, const float* v, int64_t n, int d,
                 int hidden_layers, const int32_t* order, const int* gmaxes, float* partial, float* gparams,
                 int accumulate, cudaStream_t st);

struct BwdPlan {
  int64_t acts, gphi, masks, ga, gb, gvd, gmax, gmaxes, image, partial, total;  // float offsets (ga: [L][64][n] when the tcgen05 chain runs)
  int nsplit;
  int64_t per_split;
};

static BwdPlan plan_bwd(int64_t n, int d, int hidden_layers) {
  BwdPlan P;
  int64_t off = 0;
  auto take = [&](int64_t floats) {
    int64_t o = off;
    off += (floats + 3) & ~(int64_t)3;
    return o;
  };
  const int64_t npad = (n + 127) / 128 * 128;   // the tensor-core kernels store these matrices tile-major
  P.acts = take((int64_t)hidden_layers * kH * npad);
  P.gphi = take((int64_t)d * kPP * npad);
  P.masks = take((int64_t)hidden_layers * 2 * npad);   // ReLU masks of the tensor-core path (uint32)
  P.ga = take((int64_t)hidden_layers * kH * npad);
  P.gb = take((int64_t)kH * n);
  P.gvd = take(n * d);
  P.gmax = take(n);
  P.gmaxes = take(8);
  P.image = take((nsf_tc_dgrad_image_bytes(d) + 3) / 4 + 256);   // dgrad operand image (+ slack to align it to 1 KB)
  const int sms = sm_count();
  int nsplit = (4 * sms + d - 1) / d;
  int64_t tiles = (n + kWgTileP - 1) / kWgTileP;
  if (nsplit > tiles) nsplit = (int)tiles;
  if (nsplit < 1) nsplit = 1;
  int64_t per = ((tiles + nsplit - 1) / nsplit) * kWgTileP;
  P.nsplit = (int)((n + per - 1) / per);
  P.per_split = per;
  {
    int64_t pf = (int64_t)P.nsplit * d * kH * kH, tcf = nsf_tc_wgrad_partial_floats(d);
    P.partial = take(pf > tcf ? pf : tcf);
  }
  P.total = off;
  return P;
}

template <int D>
static int run_layer_bwd(const float* v, const float* gy, const float* glogq, int64_t n, int hidden_layers, int nb,
                         const float* params, const float* params_om, const void* tc_image, const int32_t* order_host,
                         int first, float* gv, float* gparams, int accumulate, float* ws, cudaStream_t st) {
  const BwdPlan P = plan_bwd(n, D, hidden_layers);
  const int64_t np = nsf_param_floats(D, hidden_layers);
  float* acts = ws + P.acts;
  float* gphi = ws + P.gphi;
  float* ga = ws + P.ga;
  float* gb = ws + P.gb;
  float* gvd = ws + P.gvd;
  float* partial = ws + P.partial;
  const int sms = sm_count();
  int* gmaxes = reinterpret_cast<int*>(ws + P.gmaxes);
  MFB_CUDA(cudaMemsetAsync(gmaxes, 0, 8 * sizeof(int), st));
  if (tc_image) {
    // 1. recompute + spline backward, 1b. data gradients of the whole conditioner (ga[l] = dL/d(pre-activation) of
    //    hidden layer l, gv = dL/dv), 1c. every weight and bias gradient of the layer: three tensor-core kernels
    //    that share the tile-major workspace layout
    uint32_t* masks = reinterpret_cast<uint32_t*>(ws + P.masks);
    int rc = nsf_tc_spline_bwd(v, gy, glogq, n, D, tc_image, order_host, first, acts, gphi, masks, gvd, ws + P.gmax,
                               gmaxes, st);
    if (rc) return rc;
    unsigned char* image = reinterpret_cast<unsigned char*>(((uintptr_t)(ws + P.image) + 1023) & ~(uintptr_t)1023);
    rc = nsf_tc_dgrad(gphi, ws + P.gmax, masks, gvd, n, D, hidden_layers, params, order_host, ga, gv, image, gmaxes, st);
    if (rc) return rc;
    rc = nsf_tc_wgrad(gphi, ga, acts, v, n, D, hidden_layers, order_host, gmaxes, partial, gparams, accumulate, st);
    return rc ? rc : launch_status();
  }
  // 1. recompute + spline backward on the CUDA cores
  {
    FeatureOrder order = {};
    for (int i = 0; i < D; ++i) order.v[i] = order_host[i];
    const size_t smem = (size_t)((np + 3) & ~(int64_t)3) * 4 + (size_t)kPP * kNsfThreads * 4;
    if (smem > 227 * 1024) return MFB_E_UNSUPPORTED;
    MFB_CUDA(cudaFuncSetAttribute(nsf_bwd_spline_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t tiles = (n + kNsfThreads - 1) / kNsfThreads;
    int grid = (int)(tiles < sms ? tiles : sms);
    nsf_bwd_spline_kernel<D><<<grid, kNsfThreads, smem, st>>>(v, gy, glogq, n, hidden_layers, nb, params, np, order,
                                                              first, acts, gphi, gvd, ws + P.gmax, gmaxes);
    int rc = launch_status();
    if (rc) return rc;
  }
  // packed (forward) layout offsets
  const int64_t off_w1 = 0, off_b1 = (int64_t)D * kH, off_hid = off_b1 + kH;
  const int64_t off_wout = off_hid + (int64_t)(hidden_layers - 1) * (kH * kH + kH);
  const int64_t off_bout = off_wout + (int64_t)D * kH * kPP;
  // out-major layout offsets: W1 [64][D] | Wl [64][64] x (L-1) | Wout [D*64][64]
  const int64_t om_w1 = 0, om_hid = (int64_t)kH * D, om_wout = om_hid + (int64_t)(hidden_layers - 1) * kH * kH;
  const int blocks_p = (int)((n + kBwdThreads - 1) / kBwdThreads);
  const int dgrid = blocks_p < 4 * sms ? blocks_p : 4 * sms;
  const size_t dsmem = 128 * kH * 4;
  // 2. output layer
  const float* h_last = acts + (size_t)(hidden_layers - 1) * kH * n;
  {
    dim3 grid(P.nsplit, D);
    nsf_wgrad_kernel<<<grid, 256, 0, st>>>(h_last, gphi, n, P.per_split, partial);
    nsf_wgrad_reduce_kernel<<<(D * kH * kH + 255) / 256, 256, 0, st>>>(partial, P.nsplit, D, (int64_t)kH * kPP,
                                                                        gparams + off_wout, accumulate);
    nsf_rowsum_kernel<<<D * kPP, 256, 0, st>>>(gphi, n, gparams + off_bout, 0, kPP, 0, accumulate);
    nsf_dgrad_kernel<<<dgrid, kBwdThreads, dsmem, st>>>(gphi, D * kPP, n, params_om + om_wout, h_last, ga);
    int rc = launch_status();
    if (rc) return rc;
  }
  // hidden layers, last to first: gcur holds dL/d(pre-activation) of hidden layer l+1 (index l+1 in acts)
  float* gcur = ga;
  float* gnext = gb;
  for (int l = hidden_layers - 2; l >= 0; --l) {
    const float* h_prev = acts + (size_t)l * kH * n;
    float* gw = gparams + off_hid + (int64_t)l * (kH * kH + kH);
    dim3 grid(P.nsplit, 1);
    nsf_wgrad_kernel<<<grid, 256, 0, st>>>(h_prev, gcur, n, P.per_split, partial);
    nsf_wgrad_reduce_kernel<<<(kH * kH + 255) / 256, 256, 0, st>>>(partial, P.nsplit, 1, 0, gw, accumulate);
    nsf_rowsum_kernel<<<kH, 256, 0, st>>>(gcur, n, gw + kH * kH, 0, kH, 0, accumulate);
    nsf_dgrad_kernel<<<dgrid, kBwdThreads, dsmem, st>>>(gcur, kH, n, params_om + om_hid + (int64_t)l * kH * kH,
                                                         h_prev, gnext);
    int rc = launch_status();
    if (rc) return rc;
    float* t = gcur;
    gcur = gnext;
    gnext = t;
  }
  // first layer: gcur = dL/d(pre-activation 1)
  {
    int64_t per_cta = ((n + 2 * sms - 1) / (2 * sms) + 255) / 256 * 256;
    int gridw = (int)((n + per_cta - 1) / per_cta);
    nsf_wgrad_in_kernel<D><<<gridw, 256, 0, st>>>(v, gcur, n, per_cta, partial);
    nsf_sum_partials_kernel<<<(D * kH + 255) / 256, 256, 0, st>>>(partial, gridw, D * kH, gparams + off_w1, accumulate);
    nsf_rowsum_kernel<<<kH, 256, 0, st>>>(gcur, n, gparams + off_b1, 0, kH, 0, accumulate);
    nsf_bwd_input_kernel<D><<<dgrid, 256, 0, st>>>(gvd, gcur, n, params_om + om_w1, gv);
  }
  return launch_status();
}

}  // namespace mfb

using namespace mfb;

extern "C" {

int64_t mfb_nsf_layer_bwd_workspace_bytes(int64_t n, int d, int hidden_layers) {
  if (n < 1 || d < 2 || d > 6 || hidden_layers < 1) return 0;
  return plan_bwd(n, d, hidden_layers).total * 4;
}

int64_t mfb_nsf_layer_param_om_floats(int d, int hidden_units, int hidden_layers) {
  if (d < 2 || d > 6 || hidden_units != kH || hidden_layers < 1) return 0;
  return (int64_t)kH * d + (int64_t)(hidden_layers - 1) * kH * kH + (int64_t)d * kPP * kH;
}

int mfb_nsf_layer_bwd(const float* v, const float* gy, const float* glogq, int64_t n, int d, int hidden_units,
                      int hidden_layers, int bins, const float* params, const float* params_om, const void* tc_image,
                      const int32_t* order_host, int first_layer, float* gv, float* gparams, int accumulate,
                      void* workspace, int64_t workspace_bytes, void* stream) {
  MFB_CHECK_ARG(v && gy && params && params_om && order_host && gv && gparams && workspace && n >= 1);
  if (hidden_units != kH || hidden_layers < 1 || bins < 2 || 3 * bins - 1 > kPP || d < 2 || d > 6)
    return MFB_E_UNSUPPORTED;
  if (tc_image) {
    const int rc = nsf_tc_check(d, hidden_layers, bins, tc_image, order_host, v);
    if (rc) return rc;
  }
  if (workspace_bytes < mfb_nsf_layer_bwd_workspace_bytes(n, d, hidden_layers)) return MFB_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
#define MFB_BWD(DD)                                                                                                 \
  return run_layer_bwd<DD>(v, gy, glogq, n, hidden_layers, bins, params, params_om, tc_image, order_host, first_layer, \
                           gv, gparams, accumulate, ws, st)
  switch (d) {
    case 2: MFB_BWD(2);
    case 3: MFB_BWD(3);
    case 4: MFB_BWD(4);
    case 5: MFB_BWD(5);
    case 6: MFB_BWD(6);
    default: return MFB_E_UNSUPPORTED;
  }
#undef MFB_BWD
}

}  // extern "C"
