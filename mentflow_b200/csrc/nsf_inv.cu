// Density direction of the neural spline flow: v = A^{-1}(y) for one autoregressive layer,
// plus the forward log|det J| at the recovered v.
//
// Replaces generate/flows/zuko.py:21-22, 31-32, 43-50 (log_prob / inverse / inverse_steps) ->
// zuko AutoregressiveTransform._inverse (D fixed-point sweeps from v = 0, each one a full
// conditioner evaluation followed by MonotonicRQSTransform._inverse) and the extra forward
// call_and_ladj zuko makes afterwards.  Here: one kernel per layer, D conditioner sweeps per
// particle with the weights in shared memory; sweep s only updates the features whose order
// is >= s (the others are already exact), and the last sweep also yields log dy/dv, so the
// extra forward pass disappears.
#include "nsf_tc_common.cuh"

namespace mfb {

// inverse of one univariate spline; parameters in col[j*stride] (destroyed).  Returns v with
// RQS(v) = y and, if want_ladj, adds log dy/dv (forward direction) at v to ladj.
__device__ __forceinline__ float rq_spline_inverse(float* col, int stride, int nb, float y, bool want_ladj,
                                                   float& ladj) {
  if (!(y > -kBound && y <= kBound)) return y;  // identity outside the box
  // knot sums in double, as in the forward direction (knot_search): the bin in y, then the same bin in x
  float* colh = col + nb * stride;
  softmax_inplace(colh, stride, nb);
  const KnotPos kp = knot_search(colh, stride, nb, y);
  const int kbin = kp.k;
  const float hk = (float)((double)colh[kbin * stride] / kp.sum);
  const float yy = (float)((kp.target - kp.cum) * (2.0 * (double)kBound) / kp.sum);   // y - y0
  softmax_inplace(col, stride, nb);
  double sum_w = 0.0, cumw = 0.0;
  for (int j = 0; j < nb; ++j) {
    const double e = (double)col[j * stride];
    if (j < kbin) cumw += e;
    sum_w += e;
  }
  const double x0 = 2.0 * (double)kBound * (cumw / sum_w) - (double)kBound;
  const float wk = (float)((double)col[kbin * stride] / sum_w);
  const float* cold = col + 2 * nb * stride;
  float d0 = 1.0f, d1 = 1.0f;
  if (kbin > 0) {
    const float r = cold[(kbin - 1) * stride];
    d0 = expf(r / (1.0f + kClipD * fabsf(r)));
  }
  if (kbin < nb - 1) {
    const float r = cold[kbin * stride];
    d1 = expf(r / (1.0f + kClipD * fabsf(r)));
  }
  const float dx = 2.0f * kBound * wk, dy = 2.0f * kBound * hk;
  const float s = hk / wk;
  const float A = d0 + d1 - 2.0f * s;
  const float a = dy * (s - d0) + yy * A;
  const float b = dy * d0 - yy * A;
  const float c = -s * yy;
  float t = 2.0f * c / (-b - sqrtf(fmaxf(b * b - 4.0f * a * c, 0.f)));
  t = fminf(fmaxf(t, 0.0f), 1.0f);
  if (want_ladj) {
    const float omt = 1.0f - t, q = t * omt;
    const float den = fmaf(A, q, s);
    const float jac = s * s * (2.0f * s * q + d0 * omt * omt + d1 * t * t) / (den * den);
    ladj += logf(jac);
  }
  return (float)(x0 + (double)t * (double)dx);
}

template <int D>
__global__ void __launch_bounds__(kNsfThreads, 1)
nsf_layer_inv_kernel(const float* __restrict__ y, int64_t n, int hidden_layers, int nb,
                     const float* __restrict__ params, int64_t nparams, FeatureOrder order,
                     const float* __restrict__ ladj_in, int last_layer, float* __restrict__ v_out,
                     float* __restrict__ ladj_out) {
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
    float yin[D], vcur[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      yin[i] = valid ? y[p * D + i] : 0.f;
      vcur[i] = 0.f;
    }
    float ladj = 0.f;
#pragma unroll 1
    for (int sweep = 0; sweep < D; ++sweep) {
      const bool last = sweep == D - 1;
      float h[kH];
#pragma unroll
      for (int j4 = 0; j4 < kH / 4; ++j4) {
        float4 acc = *reinterpret_cast<const float4*>(b1 + 4 * j4);
#pragma unroll
        for (int i = 0; i < D; ++i) {
          const float4 w = *reinterpret_cast<const float4*>(W1t + i * kH + 4 * j4);
          acc.x = fmaf(vcur[i], w.x, acc.x); acc.y = fmaf(vcur[i], w.y, acc.y);
          acc.z = fmaf(vcur[i], w.z, acc.z); acc.w = fmaf(vcur[i], w.w, acc.w);
        }
        h[4 * j4 + 0] = fmaxf(acc.x, 0.f); h[4 * j4 + 1] = fmaxf(acc.y, 0.f);
        h[4 * j4 + 2] = fmaxf(acc.z, 0.f); h[4 * j4 + 3] = fmaxf(acc.w, 0.f);
      }
      for (int l = 0; l < hidden_layers - 1; ++l) {
        const float* wt = hid + (size_t)l * (kH * kH + kH);
        const float* bias = wt + kH * kH;
#pragma unroll 1
        for (int jc = 0; jc < kH / 8; ++jc) {
          float acc[8];
          dense8(h, wt + jc * 8, bias + jc * 8, acc);
#pragma unroll
          for (int q = 0; q < 8; ++q) col[(jc * 8 + q) * kNsfThreads] = fmaxf(acc[q], 0.f);
        }
#pragma unroll
        for (int j = 0; j < kH; ++j) h[j] = col[j * kNsfThreads];
      }
#pragma unroll 1
      for (int f = 0; f < D; ++f) {
        // features of order < sweep are already exact (their conditioners saw exact inputs);
        // on the last sweep every feature is revisited once more to collect log dy/dv
        if (order.v[f] < sweep && !last) continue;
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
            for (int q = 0; q < 8; ++q) col[(jc * 8 + q) * kNsfThreads] = acc[q];
          }
        }
        float yf = yin[0];
#pragma unroll
        for (int i = 1; i < D; ++i) yf = (f == i) ? yin[i] : yf;
        const float vf = rq_spline_inverse(col, kNsfThreads, nb, yf, last, ladj);
#pragma unroll
        for (int i = 0; i < D; ++i)
          if (f == i) vcur[i] = vf;
      }
    }
    if (valid) {
#pragma unroll
      for (int i = 0; i < D; ++i) v_out[p * D + i] = vcur[i];
      if (ladj_out) {
        float tot = (ladj_in ? ladj_in[p] : 0.f) + ladj;
        if (last_layer) {  // log q(x) = log N(z; 0, I) - sum of forward ladj
          float ss = 0.f;
#pragma unroll
          for (int i = 0; i < D; ++i) ss = fmaf(vcur[i], vcur[i], ss);
          tot = -0.5f * ss - (float)D * kHalfLog2Pi - tot;
        }
        ladj_out[p] = tot;
      }
    }
  }
}

template <int D>
static int launch_nsf_inv(const float* y, int64_t n, int hidden_layers, int nb, const float* params,
                          const FeatureOrder& order, const float* ladj_in, int last, float* v, float* ladj_out,
                          cudaStream_t st) {
  const int64_t np = nsf_param_floats(D, hidden_layers);
  const size_t smem = (size_t)((np + 3) & ~(int64_t)3) * 4 + (size_t)kPP * kNsfThreads * 4;
  if (smem > 227 * 1024) return MFB_E_UNSUPPORTED;
  MFB_CUDA(cudaFuncSetAttribute(nsf_layer_inv_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t tiles = (n + kNsfThreads - 1) / kNsfThreads;
  int64_t grid = sm_count();
  if (grid > tiles) grid = tiles;
  nsf_layer_inv_kernel<D><<<(int)grid, kNsfThreads, smem, st>>>(y, n, hidden_layers, nb, params, np, order, ladj_in,
                                                                  last, v, ladj_out);
  return launch_status();
}

}  // namespace mfb

using namespace mfb;

extern "C" int mfb_nsf_layer_inv(const float* y, int64_t n, int d, int hidden_units, int hidden_layers, int bins,
                                 const float* params, const void* tc_image, const int32_t* order_host,
                                 const float* ladj_in, int last_layer, float* v, float* ladj_out, void* stream) {
  MFB_CHECK_ARG(y && params && order_host && v && n >= 0);
  if (hidden_units != kH || hidden_layers < 1 || bins < 2 || 3 * bins - 1 > kPP) return MFB_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  if (tc_image)
    return nsf_tc_inv(y, n, d, hidden_layers, bins, tc_image, order_host, ladj_in, last_layer, v, ladj_out, st);
  if (n == 0) return 0;
  FeatureOrder ord = {};
  for (int i = 0; i < d && i < kMaxDim; ++i) ord.v[i] = order_host[i];
  switch (d) {
    case 2: return launch_nsf_inv<2>(y, n, hidden_layers, bins, params, ord, ladj_in, last_layer, v, ladj_out, st);
    case 3: return launch_nsf_inv<3>(y, n, hidden_layers, bins, params, ord, ladj_in, last_layer, v, ladj_out, st);
    case 4: return launch_nsf_inv<4>(y, n, hidden_layers, bins, params, ord, ladj_in, last_layer, v, ladj_out, st);
    case 5: return launch_nsf_inv<5>(y, n, hidden_layers, bins, params, ord, ladj_in, last_layer, v, ladj_out, st);
    case 6: return launch_nsf_inv<6>(y, n, hidden_layers, bins, params, ord, ladj_in, last_layer, v, ladj_out, st);
    default: return MFB_E_UNSUPPORTED;
  }
}
