// Neural spline flow layer: masked-MLP conditioner fused with the monotonic rational-quadratic
// spline and its log|det J|.
//
// Replaces, per autoregressive layer (reference call sites generate/flows/zuko.py:24-29 ->
// zuko 1.3.1 MaskedAutoregressiveTransform.meta / MonotonicRQSTransform.call_and_ladj, restated
// in SURVEY.md App. A and oracle/zuko_nsf.py):
//   phi = MaskedMLP(v)            4 masked SGEMMs + 3 ReLU            (zuko/nn.py)
//   soft-clip, 2 softmax, pad, 2 cumsum, exp, searchsorted, 6 gathers, RQ formula, log, where, sum
//
// This file is the fp32 CUDA-core version ("stage A"): one thread per particle, the layer's
// (pre-masked, transposed) weights resident in shared memory for the lifetime of a persistent
// CTA, activations of the current layer in registers, outputs of a layer staged through a
// per-thread column of shared memory (conflict free).  Spline parameters never touch HBM.
#include "nsf_tc_common.cuh"

namespace mfb {

template <int D>
__global__ void __launch_bounds__(kNsfThreads, 1)
nsf_layer_fwd_kernel(const float* __restrict__ v, int64_t n, int hidden_layers, int nb,
                     const float* __restrict__ params, int64_t nparams, FeatureOrder order,
                     const float* __restrict__ logq_in, int first_layer, float* __restrict__ y,
                     float* __restrict__ logq_out) {
  extern __shared__ __align__(16) float smem[];
  float* s_par = smem;
  float* s_scr = smem + ((nparams + 3) & ~(int64_t)3);  // [64][kNsfThreads]
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
  const float* hid = b1 + kH;  // (L-1) blocks of [64][64] + [64]
  const float* Wout = hid + (size_t)(hidden_layers - 1) * (kH * kH + kH);
  const float* bout = Wout + (size_t)D * kH * kPP;
  float* col = s_scr + tid;

  const int64_t ntiles = (n + kNsfThreads - 1) / kNsfThreads;
  for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int64_t p = tile * kNsfThreads + tid;
    const bool valid = p < n;
    float vin[D];
#pragma unroll
    for (int i = 0; i < D; ++i) vin[i] = valid ? v[p * D + i] : 0.f;

    float h[kH];
    // first masked layer (D -> 64)
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
    // hidden -> hidden layers
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
    // output layer, one feature at a time, fused with the spline
    float ladj = 0.f;
    float yout[D];
    const int ptotal = 3 * nb - 1;
#pragma unroll 1
    for (int f = 0; f < D; ++f) {
      const float* bf = bout + f * kPP;
      if (order.v[f] == 0) {
        // first feature in the layer's order: its spline is unconditional (bias only)
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
      float vf = vin[0];
#pragma unroll
      for (int i = 1; i < D; ++i) vf = (f == i) ? vin[i] : vf;
      const float yf = rq_spline_forward(col, kNsfThreads, nb, vf, ladj);
#pragma unroll
      for (int i = 0; i < D; ++i)
        if (f == i) yout[i] = yf;
    }
    if (valid) {
#pragma unroll
      for (int i = 0; i < D; ++i) y[p * D + i] = yout[i];
      if (logq_out) {
        float base;
        if (first_layer) {
          float ss = 0.f;
#pragma unroll
          for (int i = 0; i < D; ++i) ss = fmaf(vin[i], vin[i], ss);
          base = -0.5f * ss - (float)D * kHalfLog2Pi;
        } else {
          base = logq_in[p];
        }
        logq_out[p] = base - ladj;
      }
    }
  }
}

template <int D>
static int launch_nsf_fwd(const float* v, int64_t n, int hidden_layers, int nb, const float* params,
                          const FeatureOrder& order, const float* logq_in, int first, float* y, float* logq_out,
                          cudaStream_t st) {
  const int64_t np = nsf_param_floats(D, hidden_layers);
  const size_t smem = (size_t)((np + 3) & ~(int64_t)3) * 4 + (size_t)kPP * kNsfThreads * 4;
  if (smem > 227 * 1024) return MFB_E_UNSUPPORTED;
  MFB_CUDA(cudaFuncSetAttribute(nsf_layer_fwd_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int64_t tiles = (n + kNsfThreads - 1) / kNsfThreads;
  int64_t grid = sm_count();
  if (grid > tiles) grid = tiles;
  nsf_layer_fwd_kernel<D><<<(int)grid, kNsfThreads, smem, st>>>(v, n, hidden_layers, nb, params, np, order,
                                                                  logq_in, first, y, logq_out);
  return launch_status();
}

}  // namespace mfb

using namespace mfb;

extern "C" {

int64_t mfb_nsf_layer_param_floats(int d, int hidden_units, int hidden_layers, int bins) {
  if (d < 2 || d > 6 || hidden_units != kH || hidden_layers < 1 || bins < 2 || 3 * bins - 1 > kPP) return 0;
  return nsf_param_floats(d, hidden_layers);
}

int mfb_nsf_layer_fwd(const float* v, int64_t n, int d, int hidden_units, int hidden_layers, int bins,
                      const float* params, const void* tc_image, const int32_t* order_host, const float* logq_in,
                      int first_layer, float* y, float* logq_out, void* stream) {
  MFB_CHECK_ARG(v && params && order_host && y && n >= 0);
  if (hidden_units != kH || hidden_layers < 1 || bins < 2 || 3 * bins - 1 > kPP) return MFB_E_UNSUPPORTED;
  MFB_CHECK_ARG(first_layer || !logq_out || logq_in);
  cudaStream_t st = (cudaStream_t)stream;
  if (tc_image)
    return nsf_tc_fwd(v, n, d, hidden_layers, bins, tc_image, order_host, logq_in, first_layer, y, logq_out, st);
  if (n == 0) return 0;
  FeatureOrder ord = {};
  for (int i = 0; i < d && i < kMaxDim; ++i) ord.v[i] = order_host[i];
  switch (d) {
    case 2: return launch_nsf_fwd<2>(v, n, hidden_layers, bins, params, ord, logq_in, first_layer, y, logq_out, st);
    case 3: return launch_nsf_fwd<3>(v, n, hidden_layers, bins, params, ord, logq_in, first_layer, y, logq_out, st);
    case 4: return launch_nsf_fwd<4>(v, n, hidden_layers, bins, params, ord, logq_in, first_layer, y, logq_out, st);
    case 5: return launch_nsf_fwd<5>(v, n, hidden_layers, bins, params, ord, logq_in, first_layer, y, logq_out, st);
    case 6: return launch_nsf_fwd<6>(v, n, hidden_layers, bins, params, ord, logq_in, first_layer, y, logq_out, st);
    default: return MFB_E_UNSUPPORTED;
  }
}

}  // extern "C"
