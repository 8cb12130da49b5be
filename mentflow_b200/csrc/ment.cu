// Classical MENT: density rho(x) = prior(x) * prod_k h_k(u_k(x)), its integration / sampling
// and the Gauss-Seidel update of the Lagrange tables.
//
// u_k(x) = w_k . x for a linear transfer map.  Behind a chain linear* -> MultipoleTransform -> linear* (the kMP
// instantiations) u_k(x) = w_k . x + a_k Re(z^m) + b_k Im(z^m), z = wa . x + i wb . x (multipole.cuh); rows of linear
// maps in such a model carry order 0 and skip the kick.  Integrate mode then maps the screen back with the folded
// inverse of the chain, x = L u + p Re(zi^m) + q Im(zi^m), zi = r0 . u + i r2 . u.
//
// Replaces (reference file:line, relative to mentflow/):
//   ment.py:239-249, 227-234, 45-52   MENT.prob: per measurement a full matmul, a device->numpy
//                                     ->scipy RegularGridInterpolator (fp64, single thread)->device
//                                     round trip, clamp, product; then * exp(prior.log_prob)
//   sample.py:27-57, 99-104           GridSampler: prob on the full res^D grid, multinomial over
//                                     cells (<= 2^24 categories), uniform jitter
//   ment.py:267-317                   _simulate_integrate: Python loop over measured pixels
//   ment.py:360-367                   Python per-bin loop of the Gauss-Seidel update
#include "common.cuh"
#include "multipole.cuh"

#include <type_traits>

namespace mfb {

constexpr int kMentThreads = 256;
// Minimum resident CTAs per SM of the kernels with multipole terms: 5 (<= 51 registers) stops ptxas from spilling in
// the kick's complex powers, where with no minimum it picks 40 - 48 registers and spills in the 5-D and 6-D variants.
// The linear kernels keep no minimum (0).
template <bool kMP>
constexpr int ment_min_ctas() { return kMP ? 5 : 0; }
// The ragged kernels (screens of different sizes) are kernels of their own, so that the uniform kernels keep their
// code: they carry the table offsets beside the uniform kernels' state, and at the uniform minimum the integrate kernel
// spills (with kicks, D = 6 ... 8; without, D = 8).  Minimum 4 with kicks (<= 64 registers), 3 without (<= 80).
template <bool kMP>
constexpr int ment_ragged_min_ctas() { return kMP ? 4 : 3; }

struct MentGrid {            // regular grid of cell centres (GridSampler) or an integration grid
  int ndim;
  int shape[kMaxDim];
  float lo[kMaxDim];         // first centre
  float step[kMaxDim];       // centre spacing
};

struct MentPrior {
  float neg_half_inv_s2;     // -0.5 / scale^2 (0 for a flat prior)
  float log_norm;            // -D log s - D/2 log 2pi (log of the constant for a flat prior)
};

// shared-memory tables: coords[K][B] (bin centres) and values[K][B] (h_k)
// dinv[i] = 1 / (c[i+1] - c[i]) in double, tabulated once per CTA: the normalised distance is then a double
// multiply instead of a double division (one ulp of double apart: invisible after the cast to fp32)
__device__ __forceinline__ float lagrange_eval(const float* __restrict__ c, const float* __restrict__ h,
                                               const double* __restrict__ dinv, int B, float inv_step, float u) {
  // scipy RegularGridInterpolator(method="linear", bounds_error=False, fill_value=0) on the bin
  // centres, evaluated in double like the reference (ment.py:45-52), then cast to fp32 (:233)
  if (!(u >= c[0] && u <= c[B - 1])) return 0.f;
  int i = (int)((u - c[0]) * inv_step);
  i = min(max(i, 0), B - 2);
  while (i > 0 && u < c[i]) --i;
  while (i < B - 2 && u > c[i + 1]) ++i;
  const double w = ((double)u - (double)c[i]) * dinv[i];
  return (float)((double)h[i] * (1.0 - w) + (double)h[i + 1] * w);
}

// Lagrange functions of two-dimensional screens (ment.py:36-49: N-D RegularGridInterpolator): K2 tables of
// Bx x By values on the bin-centre grid of each screen, bilinear in between, zero outside the box of the
// centres.  They stay in global memory (85 x 85 floats per screen: L1 / L2 resident), four reads per point.
struct Tables2D {
  int k, bx, by;
  const float* proj;    // [k][2][D]  rows of the transfer matrix that land on the screen's two axes
  const float* cx;      // [k][bx]    bin centres, first axis
  const float* cy;      // [k][by]
  const float* tab;     // [k][bx][by]
};
// (kMP) the multipole rows of the 2-D screens travel beside Tables2D as mp2[k][2][2D+4]: the two rows of a screen share
// wa, wb and the order, each has its own a, b.

// z^m of the mp row `row` (layout of multipole.cuh) at x, and u + a Re(z^m) + b Im(z^m).  mp_z is false for order 0
// (a linear map in a model with kicks): the kick is skipped, since 0 * z^m would turn a huge z into NaN.
// kLdg: the row is in global memory.
template <bool kLdg>
__device__ __forceinline__ float mp_load(const float* __restrict__ p) {
  if constexpr (kLdg) return __ldg(p); else return *p;
}
template <int D, bool kLdg>
__device__ __forceinline__ bool mp_z(const float* __restrict__ row, const float (&x)[D], float& zr, float& zi) {
  const int m = (int)mp_load<kLdg>(row + 2 * D + 2) - 1;
  if (m < 1) return false;
  float xm = 0.f, ym = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) {
    xm = fmaf(mp_load<kLdg>(row + i), x[i], xm);
    ym = fmaf(mp_load<kLdg>(row + D + i), x[i], ym);
  }
  float pr, pi;
  zpow(xm, ym, m, zr, zi, pr, pi);
  return true;
}
template <int D, bool kLdg>
__device__ __forceinline__ float mp_add(const float* __restrict__ row, float zr, float zi, float u) {
  return fmaf(mp_load<kLdg>(row + 2 * D + 1), zi, fmaf(mp_load<kLdg>(row + 2 * D), zr, u));
}

// interval index and normalised distance on one axis (scipy find_indices: searchsorted - 1, clipped)
__device__ __forceinline__ bool axis_locate(const float* __restrict__ c, int B, float u, int& i, double& w) {
  if (!(u >= c[0] && u <= c[B - 1])) return false;
  const float inv = (float)(B - 1) / (c[B - 1] - c[0]);
  i = (int)((u - c[0]) * inv);
  i = min(max(i, 0), B - 2);
  while (i > 0 && u < c[i]) --i;
  while (i < B - 2 && u > c[i + 1]) ++i;
  const double x0 = (double)c[i], x1 = (double)c[i + 1];
  w = ((double)u - x0) / (x1 - x0);
  return true;
}

// the four corners tb[0], tb[1], tb[by], tb[by + 1] of the cell at normalised distances (wx, wy)
__device__ __forceinline__ float bilinear(const float* __restrict__ tb, int by, double wx, double wy) {
  const double v00 = (double)__ldg(tb), v01 = (double)__ldg(tb + 1);
  const double v10 = (double)__ldg(tb + by), v11 = (double)__ldg(tb + by + 1);
  return (float)(v00 * (1.0 - wx) * (1.0 - wy) + v01 * (1.0 - wx) * wy + v10 * wx * (1.0 - wy) + v11 * wx * wy);
}

// kRagged (screens of different sizes): off2[3][t2.k + 1] holds the start of table k in t2.cx, t2.cy and t2.tab, so
// bx_k = off2[k + 1] - off2[k] and by_k = off2[t2.k + 2 + k] - off2[t2.k + 1 + k]; t2.bx and t2.by are unused
template <int D, bool kMP = false, bool kRagged = false>
__device__ __forceinline__ float tables2d_product(const float (&x)[D], const Tables2D& t2,
                                                  const float* __restrict__ mp2 = nullptr,
                                                  const int32_t* __restrict__ off2 = nullptr) {
  float prob = 1.0f;
  for (int k = 0; k < t2.k; ++k) {
    const float* pr = t2.proj + (size_t)k * 2 * D;
    float ux = 0.f, uy = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) {
      ux = fmaf(__ldg(pr + i), x[i], ux);
      uy = fmaf(__ldg(pr + D + i), x[i], uy);
    }
    if constexpr (kMP) {
      const float* row = mp2 + (size_t)k * 2 * MFB_MP_STRIDE(D);
      float zr, zi;
      if (mp_z<D, true>(row, x, zr, zi)) {
        ux = mp_add<D, true>(row, zr, zi, ux);
        uy = mp_add<D, true>(row + MFB_MP_STRIDE(D), zr, zi, uy);
      }
    }
    int ix, iy;
    double wx, wy;
    float h = 0.f;
    if constexpr (kRagged) {
      const int32_t* ox = off2 + k;
      const int32_t* oy = ox + t2.k + 1;
      const int x0 = __ldg(ox), y0 = __ldg(oy);
      const int bx = __ldg(ox + 1) - x0, by = __ldg(oy + 1) - y0;
      if (axis_locate(t2.cx + x0, bx, ux, ix, wx) && axis_locate(t2.cy + y0, by, uy, iy, wy))
        h = bilinear(t2.tab + __ldg(oy + t2.k + 1) + (size_t)ix * by + iy, by, wx, wy);
    } else if (axis_locate(t2.cx + (size_t)k * t2.bx, t2.bx, ux, ix, wx) &&
               axis_locate(t2.cy + (size_t)k * t2.by, t2.by, uy, iy, wy)) {
      h = bilinear(t2.tab + ((size_t)k * t2.bx + ix) * t2.by + iy, t2.by, wx, wy);
    }
    h = fminf(fmaxf(h, 0.0f), 1.0e10f);   // ment.py:246
    prob *= h;
    if (prob == 0.f) break;               // every remaining factor is finite (clamped): the product stays 0
  }
  return prob;
}

// kRagged: table k holds s_off[k] .. s_off[k + 1] - 1 of s_c, s_h and s_dinv (B unused); the end of one table is
// the start of the next, so each table loads one offset
template <int D, bool kMP = false, bool kRagged = false>
__device__ __forceinline__ float ment_density(const float (&x)[D], const float* __restrict__ s_proj,
                                              const float* __restrict__ s_c, const float* __restrict__ s_h,
                                              const float* __restrict__ s_inv, const double* __restrict__ s_dinv, int K,
                                              int B, MentPrior prior, const float* __restrict__ s_mp = nullptr,
                                              const int32_t* __restrict__ s_off = nullptr) {
  float prob = 1.0f;
  int end = 0;
  if constexpr (kRagged) end = s_off[0];
  for (int k = 0; k < K; ++k) {
    float u = 0.f;
#pragma unroll
    for (int i = 0; i < D; ++i) u = fmaf(s_proj[k * D + i], x[i], u);
    if constexpr (kMP) {
      const float* row = s_mp + (size_t)k * MFB_MP_STRIDE(D);
      float zr, zi;
      if (mp_z<D, false>(row, x, zr, zi)) u = mp_add<D, false>(row, zr, zi, u);
    }
    float h;
    if constexpr (kRagged) {
      const int o = end;
      end = s_off[k + 1];
      h = lagrange_eval(s_c + o, s_h + o, s_dinv + o, end - o, s_inv[k], u);
    } else {
      h = lagrange_eval(s_c + (size_t)k * B, s_h + (size_t)k * B, s_dinv + (size_t)k * B, B, s_inv[k], u);
    }
    h = fminf(fmaxf(h, 0.0f), 1.0e10f);   // ment.py:246
    prob *= h;
    if (prob == 0.f) break;               // every remaining factor is finite (clamped): the product stays 0 -- on a 6-D
                                          // sampler grid 9 cells in 10 project outside some screen
  }
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < D; ++i) ss = fmaf(x[i], x[i], ss);
  return prob * expf(fmaf(prior.neg_half_inv_s2, ss, prior.log_norm));
}

// kRagged: B is the total T of the K tables, table k is coords[off[k] .. off[k + 1]); the offsets go to s_off[K + 1]
// (0 for an empty family, whose off may be NULL) and dinv of a table's last centre is never read
template <bool kRagged = false>
__device__ __forceinline__ void load_tables(float* s_proj, float* s_c, float* s_h, float* s_inv, double* s_dinv,
                                            const float* __restrict__ proj, const float* __restrict__ coords,
                                            const float* __restrict__ tables, int K, int B, int D,
                                            int32_t* s_off = nullptr, const int32_t* __restrict__ off = nullptr) {
  for (int i = threadIdx.x; i < K * D; i += blockDim.x) s_proj[i] = proj[i];
  if constexpr (kRagged) {
    for (int i = threadIdx.x; i <= K; i += blockDim.x) s_off[i] = K > 0 ? off[i] : 0;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
      s_c[i] = coords[i];
      s_h[i] = tables[i];
      s_dinv[i] = i + 1 < B ? 1.0 / ((double)coords[i + 1] - (double)coords[i]) : 0.0;
    }
    for (int k = threadIdx.x; k < K; k += blockDim.x) {
      const int o = off[k], n = off[k + 1] - o;
      s_inv[k] = (float)(n - 1) / (coords[o + n - 1] - coords[o]);
    }
  } else {
    for (int i = threadIdx.x; i < K * B; i += blockDim.x) {
      s_c[i] = coords[i];
      s_h[i] = tables[i];
      s_dinv[i] = (i % B < B - 1) ? 1.0 / ((double)coords[i + 1] - (double)coords[i]) : 0.0;
    }
    for (int k = threadIdx.x; k < K; k += blockDim.x)
      s_inv[k] = (float)(B - 1) / (coords[(size_t)k * B + B - 1] - coords[(size_t)k * B]);
  }
}

// (kMP) the multipole rows of the 1-D screens, [K][2D+4], follow the tables in shared memory
__device__ __forceinline__ float* mp_smem(double* s_dinv, int K, int B) {
  return reinterpret_cast<float*>(s_dinv + (size_t)K * B);
}
// the same after the T entries of ragged tables
__device__ __forceinline__ float* mp_smem(double* s_dinv, size_t T) {
  return reinterpret_cast<float*>(s_dinv + T);
}

// Shared-memory image of the 1-D family: proj[K][D] (padded to 4 floats) | (kRagged) off[K + 1] (padded to 2) | c[T]
// | h[T] | inv[K] (padded to 2) | dinv[T] (double) | (kMP) mp.  Declares s_proj .. s_dinv, s_off and T in the body.
#define MFB_MENT_SMEM(kRagged)                                                                                         \
  extern __shared__ __align__(16) float sm[];                                                                          \
  float* s_proj = sm;                                                                                                  \
  float* s_c = s_proj + (((size_t)K * D + 3) & ~(size_t)3);                                                            \
  int32_t* s_off = nullptr;                                                                                            \
  if constexpr (kRagged) {                                                                                             \
    s_off = reinterpret_cast<int32_t*>(s_c);                                                                           \
    s_c += (K + 2) & ~1;                                                                                               \
  }                                                                                                                    \
  const size_t T = kRagged ? (size_t)B : (size_t)K * B;                                                                \
  float* s_h = s_c + T;                                                                                                \
  float* s_inv = s_h + T;                                                                                              \
  double* s_dinv = reinterpret_cast<double*>(s_inv + ((K + 1) & ~1))

// MODE 0: explicit points x[G][D];  MODE 1: points of a regular grid generated from the index
// kMP: mp[K][2D+4] and mp2[K2][2][2D+4] add the multipole terms to the projections
// MODE 0: explicit points x[G][D];  MODE 1: points of a regular grid generated from the index
// kMP: mp[K][2D+4] and mp2[K2][2][2D+4] add the multipole terms to the projections
template <int D, int MODE, bool kMP = false>
__global__ void __launch_bounds__(kMentThreads, ment_min_ctas<kMP>())
ment_prob_kernel(const float* __restrict__ x, int64_t G, MentGrid grid, const float* __restrict__ proj,
                 const float* __restrict__ coords, const float* __restrict__ tables, int K, int B,
                 MentPrior prior, const Tables2D t2, float* __restrict__ out, const float* __restrict__ mp = nullptr,
                 const float* __restrict__ mp2 = nullptr) {
  extern __shared__ __align__(16) float sm[];
  float* s_proj = sm;
  float* s_c = s_proj + (((size_t)K * D + 3) & ~(size_t)3);
  float* s_h = s_c + (size_t)K * B;
  float* s_inv = s_h + (size_t)K * B;
  double* s_dinv = reinterpret_cast<double*>(s_inv + ((K + 1) & ~1));
  load_tables(s_proj, s_c, s_h, s_inv, s_dinv, proj, coords, tables, K, B, D);
  float* s_mp = nullptr;
  if constexpr (kMP) {
    s_mp = mp_smem(s_dinv, K, B);
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(D); i += blockDim.x) s_mp[i] = mp[i];
  }
  __syncthreads();
  for (int64_t g = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; g < G; g += (int64_t)gridDim.x * kMentThreads) {
    float xr[D];
    if (MODE == 0) {
#pragma unroll
      for (int i = 0; i < D; ++i) xr[i] = x[g * D + i];
    } else {
      int64_t rem = g;  // 'ij' ordering: last axis fastest (utils/grid.py:9-10)
#pragma unroll
      for (int i = D - 1; i >= 0; --i) {
        const int idx = (int)(rem % grid.shape[i]);
        rem /= grid.shape[i];
        xr[i] = fmaf((float)idx, grid.step[i], grid.lo[i]);
      }
    }
    float rho = ment_density<D, kMP>(xr, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp);
    if (t2.k > 0) rho *= tables2d_product<D, kMP>(xr, t2, mp2);
    out[g] = rho;
  }
}

// The same over tables in the ragged layout: off[K + 1] and off2[3][t2.k + 1] (nt: the 1-D entries in all)
template <int D, int MODE, bool kMP>
__global__ void __launch_bounds__(kMentThreads, ment_ragged_min_ctas<kMP>())
ment_prob_ragged_kernel(const float* __restrict__ x, int64_t G, MentGrid grid, const float* __restrict__ proj,
                        const float* __restrict__ coords, const float* __restrict__ tables, int K, int nt,
                        MentPrior prior, const Tables2D t2, float* __restrict__ out, const float* __restrict__ mp,
                        const float* __restrict__ mp2, const int32_t* __restrict__ off,
                        const int32_t* __restrict__ off2) {
  const int B = nt;
  MFB_MENT_SMEM(true);
  load_tables<true>(s_proj, s_c, s_h, s_inv, s_dinv, proj, coords, tables, K, B, D, s_off, off);
  float* s_mp = nullptr;
  if constexpr (kMP) {
    s_mp = mp_smem(s_dinv, T);
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(D); i += blockDim.x) s_mp[i] = mp[i];
  }
  __syncthreads();
  for (int64_t g = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; g < G; g += (int64_t)gridDim.x * kMentThreads) {
    float xr[D];
    if (MODE == 0) {
#pragma unroll
      for (int i = 0; i < D; ++i) xr[i] = x[g * D + i];
    } else {
      int64_t rem = g;
#pragma unroll
      for (int i = D - 1; i >= 0; --i) {
        const int idx = (int)(rem % grid.shape[i]);
        rem /= grid.shape[i];
        xr[i] = fmaf((float)idx, grid.step[i], grid.lo[i]);
      }
    }
    float rho = ment_density<D, kMP, true>(xr, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp, s_off);
    if (t2.k > 0) rho *= tables2d_product<D, kMP, true>(xr, t2, mp2, off2);
    out[g] = rho;
  }
}

// integrate mode (ment.py:267-317) for a 1-D screen: pred[b] = sum_q rho(Minv [c_b ; t_q])
// one CTA per measured pixel, deterministic block reduction
// kMP: the density has multipole rows (mp, mp2 as in ment_prob_kernel), minv is L of the folded inverse and
// imp[4D+2] = [r0 | r2 | p | q | order | 0] its kick (order 0: a linear map, x = L u)
template <int D, bool kMP = false>
__global__ void __launch_bounds__(kMentThreads, ment_min_ctas<kMP>())
ment_integrate_kernel(const float* __restrict__ meas_coords, int nb_meas, int meas_axis,
                      const float* __restrict__ meas_coords2, int nb_meas2, int meas_axis2, MentGrid igrid,
                      const float* __restrict__ minv /* [D][D] */, const float* __restrict__ proj,
                      const float* __restrict__ coords, const float* __restrict__ tables, int K, int B,
                      MentPrior prior, const Tables2D t2, float* __restrict__ pred,
                      const float* __restrict__ mp = nullptr, const float* __restrict__ mp2 = nullptr,
                      const float* __restrict__ imp = nullptr) {
  extern __shared__ __align__(16) float sm[];
  float* s_proj = sm;
  float* s_c = s_proj + (((size_t)K * D + 3) & ~(size_t)3);
  float* s_h = s_c + (size_t)K * B;
  float* s_inv = s_h + (size_t)K * B;
  __shared__ float s_minv[D * D];
  __shared__ double red[kMentThreads / 32];
  double* s_dinv = reinterpret_cast<double*>(s_inv + ((K + 1) & ~1));
  load_tables(s_proj, s_c, s_h, s_inv, s_dinv, proj, coords, tables, K, B, D);
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) s_minv[i] = minv[i];
  float* s_mp = nullptr;
  float* s_imp = nullptr;
  if constexpr (kMP) {
    s_mp = mp_smem(s_dinv, K, B);
    s_imp = s_mp + (size_t)K * MFB_MP_STRIDE(D);
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(D); i += blockDim.x) s_mp[i] = mp[i];
    for (int i = threadIdx.x; i < 4 * D + 2; i += blockDim.x) s_imp[i] = imp[i];
  }
  __syncthreads();
  int64_t Q = 1;
  for (int i = 0; i < igrid.ndim; ++i) Q *= igrid.shape[i];
  // pixel of the screen: b (1-D) or (b / nb_meas2, b % nb_meas2) (2-D, meas_axis2 >= 0)
  const int b = blockIdx.x;
  const float cm = meas_coords[meas_axis2 >= 0 ? b / nb_meas2 : b];
  const float cm2 = meas_axis2 >= 0 ? meas_coords2[b % nb_meas2] : 0.f;
  float acc = 0.f;  // the reference sums fp32 densities with torch.sum
  double dacc = 0.0;
  for (int64_t q = threadIdx.x; q < Q; q += kMentThreads) {
    float u[D];
    int64_t rem = q;
    int ia = igrid.ndim - 1;
#pragma unroll
    for (int i = D - 1; i >= 0; --i) {
      if (i == meas_axis) {
        u[i] = cm;
      } else if (i == meas_axis2) {
        u[i] = cm2;
      } else {
        const int idx = (int)(rem % igrid.shape[ia]);
        rem /= igrid.shape[ia];
        u[i] = fmaf((float)idx, igrid.step[ia], igrid.lo[ia]);
        --ia;
      }
    }
    float xr[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < D; ++j) s = fmaf(u[j], s_minv[i * D + j], s);
      xr[i] = s;
    }
    if constexpr (kMP) {
      // kick of the inverse map: zi = r0 . u + i r2 . u, x += p Re(zi^m) + q Im(zi^m)
      const int m = (int)s_imp[4 * D] - 1;
      if (m >= 1) {
        float xm = 0.f, ym = 0.f;
#pragma unroll
        for (int j = 0; j < D; ++j) {
          xm = fmaf(s_imp[j], u[j], xm);
          ym = fmaf(s_imp[D + j], u[j], ym);
        }
        float zr, zi, pr, pi;
        zpow(xm, ym, m, zr, zi, pr, pi);
#pragma unroll
        for (int i = 0; i < D; ++i) xr[i] = fmaf(s_imp[3 * D + i], zi, fmaf(s_imp[2 * D + i], zr, xr[i]));
      }
    }
    float rho = ment_density<D, kMP>(xr, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp);
    if (t2.k > 0) rho *= tables2d_product<D, kMP>(xr, t2, mp2);
    dacc += (double)rho;
  }
  (void)acc;
  dacc = warp_sum(dacc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dacc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < kMentThreads / 32; ++i) t += red[i];
    pred[b] = (float)t;
  }
}

// The same over tables in the ragged layout (as ment_prob_ragged_kernel)
template <int D, bool kMP>
__global__ void __launch_bounds__(kMentThreads, ment_ragged_min_ctas<kMP>())
ment_integrate_ragged_kernel(const float* __restrict__ meas_coords, int nb_meas, int meas_axis,
                             const float* __restrict__ meas_coords2, int nb_meas2, int meas_axis2, MentGrid igrid,
                             const float* __restrict__ minv, const float* __restrict__ proj,
                             const float* __restrict__ coords, const float* __restrict__ tables, int K, int nt,
                             MentPrior prior, const Tables2D t2, float* __restrict__ pred,
                             const float* __restrict__ mp, const float* __restrict__ mp2,
                             const float* __restrict__ imp, const int32_t* __restrict__ off,
                             const int32_t* __restrict__ off2) {
  constexpr bool kRagged = true;
  const int B = nt;
  MFB_MENT_SMEM(kRagged);
  __shared__ float s_minv[D * D];
  __shared__ double red[kMentThreads / 32];
  load_tables<kRagged>(s_proj, s_c, s_h, s_inv, s_dinv, proj, coords, tables, K, B, D, s_off, off);
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) s_minv[i] = minv[i];
  float* s_mp = nullptr;
  float* s_imp = nullptr;
  if constexpr (kMP) {
    s_mp = mp_smem(s_dinv, T);
    s_imp = s_mp + (size_t)K * MFB_MP_STRIDE(D);
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(D); i += blockDim.x) s_mp[i] = mp[i];
    for (int i = threadIdx.x; i < 4 * D + 2; i += blockDim.x) s_imp[i] = imp[i];
  }
  __syncthreads();
  int64_t Q = 1;
  for (int i = 0; i < igrid.ndim; ++i) Q *= igrid.shape[i];
  // pixel of the screen: b (1-D) or (b / nb_meas2, b % nb_meas2) (2-D, meas_axis2 >= 0)
  const int b = blockIdx.x;
  const float cm = meas_coords[meas_axis2 >= 0 ? b / nb_meas2 : b];
  const float cm2 = meas_axis2 >= 0 ? meas_coords2[b % nb_meas2] : 0.f;
  float acc = 0.f;  // the reference sums fp32 densities with torch.sum
  double dacc = 0.0;
  for (int64_t q = threadIdx.x; q < Q; q += kMentThreads) {
    float u[D];
    int64_t rem = q;
    int ia = igrid.ndim - 1;
#pragma unroll
    for (int i = D - 1; i >= 0; --i) {
      if (i == meas_axis) {
        u[i] = cm;
      } else if (i == meas_axis2) {
        u[i] = cm2;
      } else {
        const int idx = (int)(rem % igrid.shape[ia]);
        rem /= igrid.shape[ia];
        u[i] = fmaf((float)idx, igrid.step[ia], igrid.lo[ia]);
        --ia;
      }
    }
    float xr[D];
#pragma unroll
    for (int i = 0; i < D; ++i) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < D; ++j) s = fmaf(u[j], s_minv[i * D + j], s);
      xr[i] = s;
    }
    if constexpr (kMP) {
      // kick of the inverse map: zi = r0 . u + i r2 . u, x += p Re(zi^m) + q Im(zi^m)
      const int m = (int)s_imp[4 * D] - 1;
      if (m >= 1) {
        float xm = 0.f, ym = 0.f;
#pragma unroll
        for (int j = 0; j < D; ++j) {
          xm = fmaf(s_imp[j], u[j], xm);
          ym = fmaf(s_imp[D + j], u[j], ym);
        }
        float zr, zi, pr, pi;
        zpow(xm, ym, m, zr, zi, pr, pi);
#pragma unroll
        for (int i = 0; i < D; ++i) xr[i] = fmaf(s_imp[3 * D + i], zi, fmaf(s_imp[2 * D + i], zr, xr[i]));
      }
    }
    float rho = ment_density<D, kMP, kRagged>(xr, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp, s_off);
    if (t2.k > 0) rho *= tables2d_product<D, kMP, kRagged>(xr, t2, mp2, off2);
    dacc += (double)rho;
  }
  (void)acc;
  dacc = warp_sum(dacc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = dacc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < kMentThreads / 32; ++i) t += red[i];
    pred[b] = (float)t;
  }
}

// ---- inclusive scan of (rho + pad): an exact integer prefix -----------------------------------
// A prefix summed in double in two different associations (tile offsets from tree-summed tile sums, entries inside a
// tile from serial thread sums) decreases at tile starts by a few ulps, and its total misses the last entry.  So the
// scan runs on integers instead: every cell is worth units = rn((rho + pad) * scale) with scale = 2^e chosen from the
// float64 total so that the total sits in [2^61, 2^62), the units are summed exactly in uint64 (the order no longer
// matters), and cdf = units / scale.  Hence, by construction: the cdf is non-decreasing, the total is cdf[G-1] bit
// for bit, a cell of zero weight has cdf[i] == cdf[i-1], and the result is the same on every run.  Resolution 2^-62 of
// the total.  Passes: float64 tile sums -> scale -> unit tile sums -> exclusive unit prefix -> cdf.
constexpr int kScanThreads = 256;
constexpr int kScanItems = 16;  // per thread
constexpr int kScanTile = kScanThreads * kScanItems;

__device__ __forceinline__ uint64_t warp_sum_u64(uint64_t v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// kUnits = false: the float64 sum of (rho + pad) over each tile (only the total is used: it picks the scale);
// kUnits = true: the exact sum of the units of each tile, written over the float64 sums as uint64.
template <bool kUnits>
__global__ void __launch_bounds__(kScanThreads)
scan_tile_sums_kernel(const float* __restrict__ rho, int64_t G, double pad, const double* __restrict__ scale,
                      double* __restrict__ tile_sums) {
  using T = typename std::conditional<kUnits, uint64_t, double>::type;
  __shared__ T red[kScanThreads / 32];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  const double sc = kUnits ? *scale : 1.0;
  T s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < G) {
      const double v = (double)rho[base + i] + pad;
      if constexpr (kUnits) s += __double2ull_rn(v * sc); else s += v;
    }
  }
  if constexpr (kUnits) s = warp_sum_u64(s); else s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    T t = 0;
    for (int i = 0; i < kScanThreads / 32; ++i) t += red[i];
    reinterpret_cast<T*>(tile_sums)[blockIdx.x] = t;
  }
}

// scale = 2^(62 - e) for a float64 total in [2^(e-1), 2^e): the units of all cells add up to just below 2^62 (the
// float64 total is off by a relative G * 2^-53 at most, the rounding of the units by G / 2: far from 2^64).  An empty
// or non-finite total keeps scale 1; a total below 2^-961 (a subnormal pad) gets 2^1023, the largest power of two.
__global__ void __launch_bounds__(1024)
scan_scale_kernel(const double* __restrict__ tile_sums, int64_t ntiles, double* __restrict__ scale) {
  __shared__ double red[32];
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < ntiles; i += 1024) s += tile_sums[i];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 32; ++i) t += red[i];
    int e = 0;
    frexp(t, &e);
    *scale = (t > 0.0 && isfinite(t)) ? ldexp(1.0, min(62 - e, 1023)) : 1.0;
  }
}

// exclusive prefix of the unit tile sums, one block of 1024 threads: every thread adds its contiguous chunk serially, the
// 1024 chunk sums are scanned with a shuffle / shared-memory tree, then the chunk is written back as exclusive offsets.
// Integer sums: any order gives the same offsets.  (A single thread walking 4096 tiles took 244 us of a 3.3 ms MENT
// update.)  total = units of all cells / scale, exactly as scan_apply_kernel converts cdf[G-1].
__global__ void __launch_bounds__(1024)
scan_tile_offsets_kernel(uint64_t* __restrict__ tile_sums, int64_t ntiles, const double* __restrict__ scale,
                         double* __restrict__ total) {
  __shared__ uint64_t warp_tot[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t chunk = (ntiles + 1023) / 1024;
  const int64_t i0 = (int64_t)tid * chunk, i1 = (i0 + chunk < ntiles) ? i0 + chunk : ntiles;
  uint64_t s = 0;
  for (int64_t i = i0; i < i1; ++i) s += tile_sums[i];
  // inclusive scan of the chunk sums over the block
  uint64_t inc = s;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint64_t up = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += up;
  }
  if (lane == 31) warp_tot[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    uint64_t w = warp_tot[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint64_t up = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += up;
    }
    warp_tot[lane] = w;   // inclusive over warps
  }
  __syncthreads();
  uint64_t run = (warp > 0 ? warp_tot[warp - 1] : 0) + (inc - s);   // exclusive prefix of this thread's chunk
  for (int64_t i = i0; i < i1; ++i) {
    const uint64_t v = tile_sums[i];
    tile_sums[i] = run;
    run += v;
  }
  if (tid == 1023) *total = __ull2double_rn(warp_tot[31]) * (1.0 / *scale);
}

__global__ void __launch_bounds__(kScanThreads)
scan_apply_kernel(const float* __restrict__ rho, int64_t G, double pad, const double* __restrict__ scale,
                  const uint64_t* __restrict__ tile_offsets, double* __restrict__ cdf) {
  __shared__ uint64_t s_thread[kScanThreads];
  const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
  const double sc = *scale, inv = 1.0 / sc;   // powers of two: exact
  uint64_t loc[kScanItems];
  uint64_t s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) {
    if (base + i < G) s += __double2ull_rn(((double)rho[base + i] + pad) * sc);
    loc[i] = s;
  }
  s_thread[threadIdx.x] = s;
  __syncthreads();
  // exclusive prefix over the 256 thread sums (serial per thread over <= 255 values: tiny)
  uint64_t off = tile_offsets[blockIdx.x];
  for (int t = 0; t < (int)threadIdx.x; ++t) off += s_thread[t];
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (base + i < G) cdf[base + i] = __ull2double_rn(off + loc[i]) * inv;
}

// ---- Philox4x32-10 -------------------------------------------------------------------------------------
struct Philox {
  uint32_t c[4];
};
__device__ __forceinline__ Philox philox4x32(uint64_t counter, uint32_t stream, uint64_t seed, uint32_t word3 = 0u) {
  uint32_t c0 = (uint32_t)counter, c1 = (uint32_t)(counter >> 32), c2 = stream, c3 = word3;
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  Philox p;
  p.c[0] = c0; p.c[1] = c1; p.c[2] = c2; p.c[3] = c3;
  return p;
}
__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * (1.0f / 16777216.0f); }  // [0,1)

// draw `size` particles: cell ~ pmf (binary search in the CDF), then uniform inside the cell
// (sample.py:34-57).  jitter != 0 adds 0.5*U(-delta, delta) per axis (:53-55).
// Pivot levels over the cdf (see cdf_sample_kernel): level 0 is the cdf itself, level l >= 1 holds
// cdf[min(4^l (j + 1), G) - 1] for j < size[l] = ceil(size[l-1] / 4); the top level has at most four keys.  Levels are
// stored back to back, each starting on a 32-byte boundary.
constexpr int kCdfMaxLevels = 34;
struct CdfLevels {
  int n;                          // number of levels including level 0
  int64_t size[kCdfMaxLevels];
  int64_t off[kCdfMaxLevels];     // offset of level l >= 1 in the pivot array (doubles)
  int64_t total;                  // doubles in the pivot array
};
static CdfLevels cdf_levels(int64_t g) {
  CdfLevels lv = {};
  lv.size[0] = g;
  lv.n = 1;
  int64_t off = 0;
  while (lv.size[lv.n - 1] > 4 && lv.n < kCdfMaxLevels) {
    const int64_t sz = (lv.size[lv.n - 1] + 3) / 4;
    lv.size[lv.n] = sz;
    lv.off[lv.n] = off;
    off += (sz + 3) & ~(int64_t)3;
    ++lv.n;
  }
  lv.total = off;
  return lv;
}
__global__ void cdf_pivots_kernel(const double* __restrict__ cdf, int64_t G, const CdfLevels lv, double* __restrict__ pivots) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < lv.total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int l = 1;
    while (l + 1 < lv.n && idx >= lv.off[l + 1]) ++l;
    const int64_t j = idx - lv.off[l];
    double v = 0.0;
    if (j < lv.size[l]) {
      int64_t last = ((j + 1) << (2 * l)) - 1;
      if (last > G - 1) last = G - 1;
      v = cdf[last];
    }
    pivots[idx] = v;
  }
}

template <int D>
__global__ void __launch_bounds__(kMentThreads)
cdf_sample_kernel(const double* __restrict__ cdf, int64_t G, const double* __restrict__ total, MentGrid grid,
                  int jitter, uint64_t seed, uint64_t offset, int64_t size, float* __restrict__ out,
                  const double* __restrict__ pivots, const CdfLevels lv) {
  const double tot = *total;
  for (int64_t s = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; s < size; s += (int64_t)gridDim.x * kMentThreads) {
    const Philox r0 = philox4x32(offset + (uint64_t)s, 0u, seed);
    // 53-bit uniform for the cell choice
    const double uu = ((double)(((uint64_t)r0.c[0] << 21) ^ (uint64_t)(r0.c[1] >> 11)) + 0.5) * (1.0 / 9007199254740992.0);
    const double target = uu * tot;
    // first index with cdf > target.  Plain bisection wastes three quarters of every 32-byte sector it fetches (the
    // kernel is bound by L2 sector requests, 22 per sample); the pivot levels pack four keys per sector: level l holds
    // the last cdf entry of every group of 4^l cells, one sector per level decides among four children -- 12 requests
    // for 16^6 cells, the top six from L1.  The cdf is non-decreasing and tot == cdf[G-1] (exact integer prefix,
    // scan_tile_sums_kernel), so the keys of every level are non-decreasing, counting the keys <= target picks the
    // first child whose last key exceeds the target, and the cell found is the bisection's: the first with cdf > target,
    // which has positive weight.  Only uu * tot == tot (uu rounds to 1 with probability 2^-53) leaves no key above the
    // target; the descent then ends on the last cell, G - 1.
    int64_t grp = 0;
    for (int l = lv.n - 1; l >= 1; --l) {
      const double* keys = pivots + lv.off[l] + 4 * grp;
      const int64_t left = lv.size[l] - 4 * grp;          // valid keys in this group (>= 1)
      const double2 k01 = *reinterpret_cast<const double2*>(keys);
      const double2 k23 = *reinterpret_cast<const double2*>(keys + 2);
      int i = (k01.x <= target) ? 1 : 0;
      i += (left > 1 && k01.y <= target) ? 1 : 0;
      i += (left > 2 && k23.x <= target) ? 1 : 0;
      i = (i < left - 1) ? i : (int)(left - 1);            // the group's last key (>= its parent's key > target) covers it
      i = i < 3 ? i : 3;
      grp = 4 * grp + i;
    }
    int64_t lo;
    {
      const int64_t base = 4 * grp, left = G - base;
      lo = base;
      if (left > 1 && cdf[base] <= target) lo = base + 1;
      if (left > 2 && lo == base + 1 && cdf[base + 1] <= target) lo = base + 2;
      if (left > 3 && lo == base + 2 && cdf[base + 2] <= target) lo = base + 3;
    }
    int64_t rem = lo;
    uint32_t rnd[2 * kMaxDim];
    rnd[0] = r0.c[2];
    rnd[1] = r0.c[3];
#pragma unroll
    for (int b = 0; b < (2 * D + 1) / 4 + 1; ++b) {
      const Philox rb = philox4x32(offset + (uint64_t)s, 1u + b, seed);
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (2 + 4 * b + q < 2 * kMaxDim) rnd[2 + 4 * b + q] = rb.c[q];
    }
#pragma unroll
    for (int i = D - 1; i >= 0; --i) {
      const int idx = (int)(rem % grid.shape[i]);
      rem /= grid.shape[i];
      // grid.lo / grid.step here describe cell EDGES: lb = lo + idx*step
      const float lb = fmaf((float)idx, grid.step[i], grid.lo[i]);
      float v = fmaf(grid.step[i], u01(rnd[2 * i]), lb);
      // fp32 rounding must not push the point onto the cell's upper edge (= into the next cell): on a 1000-cell axis
      // that happened to 3e-5 of the draws
      const float ub = fmaf((float)(idx + 1), grid.step[i], grid.lo[i]);
      v = (v < ub) ? v : nextafterf(ub, lb);
      if (jitter) v += 0.5f * grid.step[i] * (2.0f * u01(rnd[2 * i + 1]) - 1.0f);
      out[s * D + i] = v;
    }
  }
}

// ---- Metropolis-Hastings chains (MetropolisHastingsSampler) ---------------------------------------------
// Chain c (global index), step t: the Philox blocks philox4x32(c, t, seed, b), b = 0 .. kMhBlocks - 1, give the words
// w[4b + q].  Pair j (< ceil(D/2)) is Box-Muller on (w[2j], w[2j+1]): r = sqrt(-2 log u1), u1 in (0, 1], angle
// 2 pi u2, u2 in [0, 1); xi[2j] = r cos, xi[2j+1] = r sin (dropped for odd D at the last pair).  The next word,
// w[2 ceil(D/2)], is the acceptance uniform in (0, 1].  t = 0 is the start draw (its uniform is unused).
template <int D>
__host__ __device__ constexpr int mh_blocks() { return (2 * ((D + 1) / 2) + 1 + 3) / 4; }

__device__ __forceinline__ float u01_open(uint32_t r) { return (float)((r >> 8) + 1u) * (1.0f / 16777216.0f); }  // (0,1]

// Box-Muller on one pair of words
__device__ __forceinline__ void mh_normals(uint32_t w0, uint32_t w1, float& a0, float& a1) {
  const float r = sqrtf(-2.0f * logf(u01_open(w0)));
  float s, co;
  sincospif(2.0f * u01(w1), &s, &co);
  a0 = r * co;
  a1 = r * s;
}

// x_0: the start point, or start_scale * xi of step 0
template <int D>
__device__ __forceinline__ void mh_start(uint64_t c, uint64_t seed, const float* __restrict__ start, float start_scale,
                                         float (&x)[D]) {
  if (start) {
#pragma unroll
    for (int i = 0; i < D; ++i) x[i] = start[i];
    return;
  }
#pragma unroll
  for (int b = 0; b < mh_blocks<D>(); ++b) {
    const Philox p = philox4x32(c, 0u, seed, (uint32_t)b);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = 2 * b + h;                       // pair j: xi[2j], xi[2j+1]
      if (2 * j < D) {
        float a0, a1;
        mh_normals(p.c[2 * h], p.c[2 * h + 1], a0, a1);
        x[2 * j] = start_scale * a0;
        if (2 * j + 1 < D) x[2 * j + 1] = start_scale * a1;
      }
    }
  }
}

// proposal of step t >= 1: xp_i = x_i + (L xi)_i, (L xi)_i = fmaf chain from 0 over j = 0 .. i ascending
// (L lower triangular, row-major [D][D]); returns the acceptance uniform.  The pairs are consumed as they are drawn:
// pair j adds columns 2j, 2j+1 to every row, which keeps each row's chain in ascending order without holding xi.
template <int D>
__device__ __forceinline__ float mh_propose(uint64_t c, uint32_t t, uint64_t seed, const float* __restrict__ chol,
                                            const float (&x)[D], float (&xp)[D]) {
  constexpr int kPairs = (D + 1) / 2;
#pragma unroll
  for (int i = 0; i < D; ++i) xp[i] = 0.f;
  float u = 0.f;
#pragma unroll
  for (int b = 0; b < mh_blocks<D>(); ++b) {
    const Philox p = philox4x32(c, t, seed, (uint32_t)b);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = 2 * b + h;
      if (j < kPairs) {
        float a0, a1;
        mh_normals(p.c[2 * h], p.c[2 * h + 1], a0, a1);
#pragma unroll
        for (int i = 2 * j; i < D; ++i) {
          xp[i] = fmaf(chol[i * D + 2 * j], a0, xp[i]);
          if (2 * j + 1 <= i) xp[i] = fmaf(chol[i * D + 2 * j + 1], a1, xp[i]);
        }
      } else if (j == kPairs) {
        u = u01_open(p.c[2 * h]);
      }
    }
  }
#pragma unroll
  for (int i = 0; i < D; ++i) xp[i] = x[i] + xp[i];
  return u;
}

// the acceptance uniform of step t alone
template <int D>
__device__ __forceinline__ float mh_uniform(uint64_t c, uint32_t t, uint64_t seed) {
  constexpr int kWord = 2 * ((D + 1) / 2);
  return u01_open(philox4x32(c, t, seed, (uint32_t)(kWord / 4)).c[kWord % 4]);
}

// the acceptance rule: a chain at zero density takes every finite proposal, a chain at positive density never takes a
// zero-density one, a NaN or inf proposal is never taken
__device__ __forceinline__ bool mh_accept(float rho_prop, float u, float rho) {
  return isfinite(rho_prop) && rho_prop >= u * rho;
}

struct MhChains {
  uint64_t chain0;          // global index of the first chain
  int64_t n;                // chains
  const float* start;       // [D] or NULL
  float start_scale;
  const float* chol;        // [D][D] lower Cholesky factor of the proposal covariance
  int64_t burnin, steps, thin;
  uint64_t seed;
};

// one thread per chain: x and rho(x) stay in registers, rho is ment_prob_kernel's arithmetic; only the recorded
// states x_{burnin + r thin}, r < steps, are written, chain i's at rows i * steps + r of out
// Minimum resident CTAs of the chain kernel: 3 (<= 80 registers) up to D = 7, 2 at D = 8, with and without kicks.  The
// chain state x, the proposal and the Philox words sit beside the density's registers: at the density kernels'
// minimum (5 with kicks) ptxas spills from D = 1 on, and with no minimum it picks 64 - 80 registers and spills in
// some dimensions.
template <int D>
constexpr int mh_min_ctas() { return D < 8 ? 3 : 2; }
// the ragged chain kernel: at 3 CTAs it spills a word at D = 1 and 2, so those take 2
template <int D>
constexpr int mh_ragged_min_ctas() { return D > 2 && D < 8 ? 3 : 2; }
template <int D, bool kMP>
__global__ void __launch_bounds__(kMentThreads, mh_min_ctas<D>())
ment_mh_kernel(const float* __restrict__ proj, const float* __restrict__ coords, const float* __restrict__ tables,
               int K, int B, MentPrior prior, const Tables2D t2, const float* __restrict__ mp,
               const float* __restrict__ mp2, const MhChains ch, float* __restrict__ out,
               unsigned long long* __restrict__ accepted) {
  extern __shared__ __align__(16) float sm[];
  __shared__ float s_chol[D * D];
  float* s_proj = sm;
  float* s_c = s_proj + (((size_t)K * D + 3) & ~(size_t)3);
  float* s_h = s_c + (size_t)K * B;
  float* s_inv = s_h + (size_t)K * B;
  double* s_dinv = reinterpret_cast<double*>(s_inv + ((K + 1) & ~1));
  load_tables(s_proj, s_c, s_h, s_inv, s_dinv, proj, coords, tables, K, B, D);
  float* s_mp = nullptr;
  if constexpr (kMP) {
    s_mp = mp_smem(s_dinv, K, B);
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(D); i += blockDim.x) s_mp[i] = mp[i];
  }
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) s_chol[i] = ch.chol[i];
  __syncthreads();
  const int64_t total = ch.burnin + (ch.steps - 1) * ch.thin;
  unsigned long long acc = 0;
  for (int64_t i = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; i < ch.n; i += (int64_t)gridDim.x * kMentThreads) {
    const uint64_t c = ch.chain0 + (uint64_t)i;
    float x[D];
    mh_start<D>(c, ch.seed, ch.start, ch.start_scale, x);
    float rho = ment_density<D, kMP>(x, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp);
    if (t2.k > 0) rho *= tables2d_product<D, kMP>(x, t2, mp2);
    float* row = out + i * ch.steps * D;
    int64_t next = ch.burnin;         // next step to record
    for (int64_t t = 0;; ++t) {
      if (t > 0) {
        float xp[D];
        const float u = mh_propose<D>(c, (uint32_t)t, ch.seed, s_chol, x, xp);
        float rp = ment_density<D, kMP>(xp, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp);
        if (t2.k > 0) rp *= tables2d_product<D, kMP>(xp, t2, mp2);
        if (mh_accept(rp, u, rho)) {
#pragma unroll
          for (int j = 0; j < D; ++j) x[j] = xp[j];
          rho = rp;
          ++acc;
        }
      }
      if (t == next) {
#pragma unroll
        for (int j = 0; j < D; ++j) row[j] = x[j];
        row += D;
        next += ch.thin;
      }
      if (t == total) break;
    }
  }
  acc = warp_sum_u64(acc);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(accepted, acc);
}

// The same chains over tables in the ragged layout (as ment_prob_ragged_kernel)
template <int D, bool kMP>
__global__ void __launch_bounds__(kMentThreads, mh_ragged_min_ctas<D>())
ment_mh_ragged_kernel(const float* __restrict__ proj, const float* __restrict__ coords,
                      const float* __restrict__ tables, int K, int nt, MentPrior prior, const Tables2D t2,
                      const float* __restrict__ mp, const float* __restrict__ mp2, const MhChains ch,
                      float* __restrict__ out, unsigned long long* __restrict__ accepted,
                      const int32_t* __restrict__ off, const int32_t* __restrict__ off2) {
  constexpr bool kRagged = true;
  const int B = nt;
  MFB_MENT_SMEM(kRagged);
  __shared__ float s_chol[D * D];
  load_tables<kRagged>(s_proj, s_c, s_h, s_inv, s_dinv, proj, coords, tables, K, B, D, s_off, off);
  float* s_mp = nullptr;
  if constexpr (kMP) {
    s_mp = mp_smem(s_dinv, T);
    for (int i = threadIdx.x; i < K * MFB_MP_STRIDE(D); i += blockDim.x) s_mp[i] = mp[i];
  }
  for (int i = threadIdx.x; i < D * D; i += blockDim.x) s_chol[i] = ch.chol[i];
  __syncthreads();
  const int64_t total = ch.burnin + (ch.steps - 1) * ch.thin;
  unsigned long long acc = 0;
  for (int64_t i = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; i < ch.n; i += (int64_t)gridDim.x * kMentThreads) {
    const uint64_t c = ch.chain0 + (uint64_t)i;
    float x[D];
    mh_start<D>(c, ch.seed, ch.start, ch.start_scale, x);
    float rho = ment_density<D, kMP, kRagged>(x, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp, s_off);
    if (t2.k > 0) rho *= tables2d_product<D, kMP, kRagged>(x, t2, mp2, off2);
    float* row = out + i * ch.steps * D;
    int64_t next = ch.burnin;         // next step to record
    for (int64_t t = 0;; ++t) {
      if (t > 0) {
        float xp[D];
        const float u = mh_propose<D>(c, (uint32_t)t, ch.seed, s_chol, x, xp);
        float rp = ment_density<D, kMP, kRagged>(xp, s_proj, s_c, s_h, s_inv, s_dinv, K, B, prior, s_mp, s_off);
        if (t2.k > 0) rp *= tables2d_product<D, kMP, kRagged>(xp, t2, mp2, off2);
        if (mh_accept(rp, u, rho)) {
#pragma unroll
          for (int j = 0; j < D; ++j) x[j] = xp[j];
          rho = rp;
          ++acc;
        }
      }
      if (t == next) {
#pragma unroll
        for (int j = 0; j < D; ++j) row[j] = x[j];
        row += D;
        next += ch.thin;
      }
      if (t == total) break;
    }
  }
  acc = warp_sum_u64(acc);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(accepted, acc);
}

// the same steps one at a time around a density the library cannot see: t = 0 writes the start draws, t >= 1 the
// proposals from the current states x
template <int D>
__global__ void __launch_bounds__(kMentThreads)
mh_propose_kernel(const float* __restrict__ x, int64_t n, uint64_t chain0, const float* __restrict__ start,
                  float start_scale, const float* __restrict__ chol, uint32_t t, uint64_t seed, float* __restrict__ xp) {
  for (int64_t i = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kMentThreads) {
    const uint64_t c = chain0 + (uint64_t)i;
    float y[D];
    if (t == 0) {
      mh_start<D>(c, seed, start, start_scale, y);
    } else {
      float xr[D];
#pragma unroll
      for (int j = 0; j < D; ++j) xr[j] = x[i * D + j];
      mh_propose<D>(c, t, seed, chol, xr, y);
    }
#pragma unroll
    for (int j = 0; j < D; ++j) xp[i * D + j] = y[j];
  }
}

template <int D>
__global__ void __launch_bounds__(kMentThreads)
mh_accept_kernel(float* __restrict__ x, float* __restrict__ rho, const float* __restrict__ xp,
                 const float* __restrict__ rho_prop, int64_t n, uint64_t chain0, uint32_t t, uint64_t seed,
                 unsigned long long* __restrict__ accepted) {
  unsigned long long acc = 0;
  for (int64_t i = (int64_t)blockIdx.x * kMentThreads + threadIdx.x; i < n; i += (int64_t)gridDim.x * kMentThreads) {
    const float u = mh_uniform<D>(chain0 + (uint64_t)i, t, seed);
    const float rp = rho_prop[i];
    if (mh_accept(rp, u, rho[i])) {
#pragma unroll
      for (int j = 0; j < D; ++j) x[i * D + j] = xp[i * D + j];
      rho[i] = rp;
      ++acc;
    }
  }
  acc = warp_sum_u64(acc);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(accepted, acc);
}

// Gauss-Seidel update of one table (ment.py:360-367)
__global__ void gs_update_kernel(float* __restrict__ table, const float* __restrict__ meas,
                                 const float* __restrict__ pred, int n, float lr, float thresh) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float p = pred[i];
  if (p < thresh) p = 0.f;
  const float g = meas[i];
  if (g != 0.f && p != 0.f) table[i] *= 1.0f + lr * (g / p - 1.0f);
}

static size_t ment_smem(int K, int B, int d) {
  return ((((size_t)K * d + 3) & ~(size_t)3) + 2 * (size_t)K * B + ((K + 1) & ~1)) * 4 + (size_t)K * B * 8 + 16;
}
// kMP: the 1-D screens' multipole rows and the inverse kick of integrate mode follow (MentSmem::end)
static size_t ment_smem_mp(int K, int B, int d) {
  return ment_smem(K, B, d) + ((size_t)K * MFB_MP_STRIDE(d) + 4 * (size_t)d + 2) * 4;
}
// the ragged layout of K tables of T bins in all: ment_smem's image plus the offsets off[K + 1]
static size_t ment_smem_ragged(int K, int T, int d) {
  return ((((size_t)K * d + 3) & ~(size_t)3) + ((K + 2) & ~1) + 2 * (size_t)T + ((K + 1) & ~1)) * 4 +
         (size_t)T * 8 + 16;
}
static size_t ment_smem_ragged_mp(int K, int T, int d) {
  return ment_smem_ragged(K, T, d) + ((size_t)K * MFB_MP_STRIDE(d) + 4 * (size_t)d + 2) * 4;
}
// b: the bins of every table (uniform) or the total (ragged)
static size_t ment_smem_of(bool ragged, bool kick, int K, int b, int d) {
  if (ragged) return kick ? ment_smem_ragged_mp(K, b, d) : ment_smem_ragged(K, b, d);
  return kick ? ment_smem_mp(K, b, d) : ment_smem(K, b, d);
}
constexpr size_t kMentSmemCap = 200 * 1024;

static MentGrid make_grid(int ndim, const int32_t* shape, const float* lo, const float* step) {
  MentGrid g;
  g.ndim = ndim;
  for (int i = 0; i < kMaxDim; ++i) {
    g.shape[i] = i < ndim ? shape[i] : 1;
    g.lo[i] = i < ndim ? lo[i] : 0.f;
    g.step[i] = i < ndim ? step[i] : 0.f;
  }
  return g;
}

// The 1-D family (k tables of b bins, or ragged: offsets off and b bins in all, at least 2 per table) and the 2-D
// family t2 (ragged: offsets off2); behind kicks a non-empty family needs its multipole rows
static bool tables_ok(bool ragged, int k, int b, const int32_t* off, const float* proj, const float* coords,
                      const float* tables, const float* mp, const Tables2D& t2, const int32_t* off2, const float* mp2,
                      bool kick) {
  const bool sizes1 = ragged ? off && (int64_t)b >= 2 * (int64_t)k : b >= 2;
  const bool sizes2 = ragged ? off2 != nullptr : t2.bx >= 2 && t2.by >= 2;
  if (k < 0 || (k > 0 && !(proj && coords && tables && sizes1))) return false;
  if (t2.k < 0 || (t2.k > 0 && !(t2.proj && t2.cx && t2.cy && t2.tab && sizes2))) return false;
  return !kick || ((k == 0 || mp) && (t2.k == 0 || mp2));
}

// set the kernel's dynamic shared memory and launch it with kMentThreads threads per CTA
template <typename... P, typename... A>
static int launch_ment(void (*kernel)(P...), int64_t blocks, size_t smem, cudaStream_t st, A... args) {
  MFB_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kernel<<<(int)blocks, kMentThreads, smem, st>>>(args...);
  return launch_status();
}

// ragged: the tables in the ragged layout (off, off2; B is the 1-D total), through the _ragged_ kernels
template <int D>
static int launch_prob(int mode, bool kick, bool ragged, const float* x, int64_t G, const MentGrid& grid,
                       const float* proj, const float* coords, const float* tables, int K, int B, const int32_t* off,
                       const int32_t* off2, const float* mp, const Tables2D& t2, const float* mp2, MentPrior prior,
                       float* out, cudaStream_t st) {
  const size_t smem = ment_smem_of(ragged, kick, K, B, D);
  if (smem > kMentSmemCap) return MFB_E_UNSUPPORTED;
  int64_t blocks = (G + kMentThreads - 1) / kMentThreads;
  int64_t cap = (int64_t)sm_count() * 8;
  blocks = blocks < cap ? blocks : cap;
  if (ragged) {
    const auto kernel = mode == 0 ? (kick ? ment_prob_ragged_kernel<D, 0, true> : ment_prob_ragged_kernel<D, 0, false>)
                                  : (kick ? ment_prob_ragged_kernel<D, 1, true> : ment_prob_ragged_kernel<D, 1, false>);
    return launch_ment(kernel, blocks, smem, st, x, G, grid, proj, coords, tables, K, B, prior, t2, out, mp, mp2, off,
                       off2);
  }
  const auto kernel = mode == 0 ? (kick ? ment_prob_kernel<D, 0, true> : ment_prob_kernel<D, 0, false>)
                                : (kick ? ment_prob_kernel<D, 1, true> : ment_prob_kernel<D, 1, false>);
  return launch_ment(kernel, blocks, smem, st, x, G, grid, proj, coords, tables, K, B, prior, t2, out, mp, mp2);
}

template <int D>
static int launch_integrate(bool kick, bool ragged, const float* mc, int nb, int ax, const float* mc2, int nb2,
                            int ax2, const MentGrid& grid, const float* minv, const float* imp, const float* proj,
                            const float* coords, const float* tables, int k, int b, const int32_t* off,
                            const int32_t* off2, const float* mp, const Tables2D& t2, const float* mp2, MentPrior pr,
                            float* pred, cudaStream_t st) {
  const size_t smem = ment_smem_of(ragged, kick, k, b, D);
  if (smem > kMentSmemCap) return MFB_E_UNSUPPORTED;
  const int pixels = ax2 >= 0 ? nb * nb2 : nb;
  if (ragged) {
    const auto kernel = kick ? ment_integrate_ragged_kernel<D, true> : ment_integrate_ragged_kernel<D, false>;
    return launch_ment(kernel, pixels, smem, st, mc, nb, ax, mc2, nb2, ax2, grid, minv, proj, coords, tables, k, b, pr,
                       t2, pred, mp, mp2, imp, off, off2);
  }
  const auto kernel = kick ? ment_integrate_kernel<D, true> : ment_integrate_kernel<D, false>;
  return launch_ment(kernel, pixels, smem, st, mc, nb, ax, mc2, nb2, ax2, grid, minv, proj, coords, tables, k, b, pr,
                     t2, pred, mp, mp2, imp);
}

// one CTA per 256 chains, no grid-stride cap: a chain is a whole run, and the block scheduler evens out chains of
// different cost better than a thread walking several of them
static int mh_grid(int64_t n) { return (int)((n + kMentThreads - 1) / kMentThreads); }

template <int D>
static int launch_mh(bool kick, bool ragged, const float* proj, const float* coords, const float* tables, int K, int B,
                     const int32_t* off, const int32_t* off2, const float* mp, const Tables2D& t2, const float* mp2,
                     MentPrior prior, const MhChains& ch, float* out, int64_t* accepted, cudaStream_t st) {
  const size_t smem = ment_smem_of(ragged, kick, K, B, D);
  if (smem > kMentSmemCap) return MFB_E_UNSUPPORTED;
  unsigned long long* acc = reinterpret_cast<unsigned long long*>(accepted);
  if (ragged) {
    const auto kernel = kick ? ment_mh_ragged_kernel<D, true> : ment_mh_ragged_kernel<D, false>;
    return launch_ment(kernel, mh_grid(ch.n), smem, st, proj, coords, tables, K, B, prior, t2, mp, mp2, ch, out, acc,
                       off, off2);
  }
  const auto kernel = kick ? ment_mh_kernel<D, true> : ment_mh_kernel<D, false>;
  return launch_ment(kernel, mh_grid(ch.n), smem, st, proj, coords, tables, K, B, prior, t2, mp, mp2, ch, out, acc);
}

// the last step of a run must fit the 32-bit stream word: burnin + (steps - 1) thin < 2^32
static bool mh_steps_ok(int64_t burnin, int64_t steps, int64_t thin) {
  if (burnin < 0 || steps < 1 || thin < 1 || burnin > (int64_t)UINT32_MAX) return false;
  return steps - 1 <= ((int64_t)UINT32_MAX - burnin) / thin;
}

}  // namespace mfb

using namespace mfb;

extern "C" {

// The tables of a call: the 1-D family with b bins per table (uniform) or off[k + 1] and b bins in all (ragged), and
// the 2-D family t2 (ragged: off2[3][t2.k + 1]).  An empty 1-D family takes b = 2 (uniform) or 0 (ragged).
struct MentTables {
  bool ragged;
  int k, b;
  const int32_t* off;
  const float *proj, *coords, *tables, *mp;
  Tables2D t2;
  const int32_t* off2;
  const float* mp2;
  bool ok(bool kick) const { return tables_ok(ragged, k, b, off, proj, coords, tables, mp, t2, off2, mp2, kick); }
  int bins() const { return k > 0 ? b : (ragged ? 0 : 2); }
};

static MentTables uniform_tables(const float* proj, const float* coords, const float* tables, int k, int b,
                                 const float* mp, const float* proj2, const float* cx2, const float* cy2,
                                 const float* tables2, int k2, int bx, int by, const float* mp2) {
  return MentTables{false, k, b, nullptr, proj, coords, tables, mp, Tables2D{k2, bx, by, proj2, cx2, cy2, tables2},
                    nullptr, mp2};
}

static MentTables ragged_tables(const float* proj, const float* coords, const float* tables, int k,
                                const int32_t* offsets, int total, const float* mp, const float* proj2,
                                const float* cx2, const float* cy2, const float* tables2, int k2,
                                const int32_t* offsets2, const float* mp2) {
  return MentTables{true, k, total, offsets, proj, coords, tables, mp,
                    Tables2D{k2, 0, 0, proj2, cx2, cy2, tables2}, offsets2, mp2};
}

// rho at the g points x (mode 0) or on the g cells of `grid` (mode 1): the body of the mfb_ment_prob* entry points
static int ment_prob_impl(int mode, const float* x, int64_t g, const MentGrid& grid, int d, const MentTables& t,
                          float prior_neg_half_inv_s2, float prior_log_norm, float* out, void* stream) {
  const bool kick = t.mp || t.mp2;
  MFB_CHECK_ARG(out && d >= 1 && d <= kMaxDim);
  MFB_CHECK_ARG(t.ok(kick));
  if (g == 0) return 0;
  const MentPrior pr{prior_neg_half_inv_s2, prior_log_norm};
  cudaStream_t st = (cudaStream_t)stream;
#define MFB_CALL(DD)                                                                                                   \
  launch_prob<DD>(mode, kick, t.ragged, x, g, grid, t.proj, t.coords, t.tables, t.k, t.bins(), t.off, t.off2, t.mp,   \
                  t.t2, t.mp2, pr, out, st)
  switch (d) {
    case 1: return MFB_CALL(1);
    case 2: return MFB_CALL(2);
    case 3: return MFB_CALL(3);
    case 4: return MFB_CALL(4);
    case 5: return MFB_CALL(5);
    case 6: return MFB_CALL(6);
    case 7: return MFB_CALL(7);
    default: return MFB_CALL(8);
  }
#undef MFB_CALL
}

static int ment_prob_points(const float* x, int64_t g, int d, const MentTables& t, float prior_neg_half_inv_s2,
                            float prior_log_norm, float* out, void* stream) {
  MFB_CHECK_ARG(x && g >= 0);
  return ment_prob_impl(0, x, g, make_grid(0, nullptr, nullptr, nullptr), d, t, prior_neg_half_inv_s2, prior_log_norm,
                        out, stream);
}

static int ment_prob_grid(int d, const int32_t* shape_host, const float* first_centre_host, const float* step_host,
                          const MentTables& t, float prior_neg_half_inv_s2, float prior_log_norm, float* out,
                          void* stream) {
  MFB_CHECK_ARG(shape_host && first_centre_host && step_host && d >= 1 && d <= kMaxDim);
  int64_t g = 1;
  for (int i = 0; i < d; ++i) {
    MFB_CHECK_ARG(shape_host[i] >= 1);
    g *= shape_host[i];
  }
  return ment_prob_impl(1, nullptr, g, make_grid(d, shape_host, first_centre_host, step_host), d, t,
                        prior_neg_half_inv_s2, prior_log_norm, out, stream);
}

static int ment_integrate(int d, const float* meas_coords, int nb_meas, int meas_axis, const float* meas_coords2,
                          int nb_meas2, int meas_axis2, int n_int_axes, const int32_t* int_shape_host,
                          const float* int_first_host, const float* int_step_host, const float* linv,
                          const float* inv_mp, const MentTables& t, float prior_neg_half_inv_s2,
                          float prior_log_norm, float* pred, void* stream) {
  const bool kick = t.mp || t.mp2 || inv_mp;
  MFB_CHECK_ARG(meas_coords && linv && (inv_mp || !kick) && pred && int_shape_host && int_first_host && int_step_host);
  const int n_meas = meas_axis2 >= 0 ? 2 : 1;
  MFB_CHECK_ARG(d >= 2 && d <= kMaxDim && n_int_axes == d - n_meas && n_int_axes >= 1);
  MFB_CHECK_ARG(meas_axis >= 0 && meas_axis < d && nb_meas >= 1 && meas_axis2 < d && meas_axis2 != meas_axis);
  MFB_CHECK_ARG(meas_axis2 < 0 || (meas_coords2 && nb_meas2 >= 1));
  MFB_CHECK_ARG(t.ok(kick));
  const MentPrior pr{prior_neg_half_inv_s2, prior_log_norm};
  const MentGrid grid = make_grid(n_int_axes, int_shape_host, int_first_host, int_step_host);
  cudaStream_t st = (cudaStream_t)stream;
#define MFB_CALL(DD)                                                                                                   \
  launch_integrate<DD>(kick, t.ragged, meas_coords, nb_meas, meas_axis, meas_coords2, nb_meas2, meas_axis2, grid,     \
                       linv, inv_mp, t.proj, t.coords, t.tables, t.k, t.bins(), t.off, t.off2, t.mp, t.t2, t.mp2, pr, \
                       pred, st)
  switch (d) {
    case 2: return MFB_CALL(2);
    case 3: return MFB_CALL(3);
    case 4: return MFB_CALL(4);
    case 5: return MFB_CALL(5);
    case 6: return MFB_CALL(6);
    case 7: return MFB_CALL(7);
    default: return MFB_CALL(8);
  }
#undef MFB_CALL
}

int mfb_ment_prob(const float* x, int64_t g, int d, const float* proj, const float* coords, const float* tables, int k,
                  int b, const float* mp, const float* proj2, const float* cx2, const float* cy2, const float* tables2,
                  int k2, int bx, int by, const float* mp2, float prior_neg_half_inv_s2, float prior_log_norm,
                  float* out, void* stream) {
  return ment_prob_points(x, g, d,
                          uniform_tables(proj, coords, tables, k, b, mp, proj2, cx2, cy2, tables2, k2, bx, by, mp2),
                          prior_neg_half_inv_s2, prior_log_norm, out, stream);
}

int mfb_ment_prob_ragged(const float* x, int64_t g, int d, const float* proj, const float* coords,
                         const float* tables, int k, const int32_t* offsets, int total, const float* mp,
                         const float* proj2, const float* cx2, const float* cy2, const float* tables2, int k2,
                         const int32_t* offsets2, const float* mp2, float prior_neg_half_inv_s2, float prior_log_norm,
                         float* out, void* stream) {
  return ment_prob_points(
      x, g, d, ragged_tables(proj, coords, tables, k, offsets, total, mp, proj2, cx2, cy2, tables2, k2, offsets2, mp2),
      prior_neg_half_inv_s2, prior_log_norm, out, stream);
}

int mfb_ment_prob_grid(int d, const int32_t* shape_host, const float* first_centre_host, const float* step_host,
                       const float* proj, const float* coords, const float* tables, int k, int b, const float* mp,
                       const float* proj2, const float* cx2, const float* cy2, const float* tables2, int k2, int bx,
                       int by, const float* mp2, float prior_neg_half_inv_s2, float prior_log_norm, float* out,
                       void* stream) {
  return ment_prob_grid(d, shape_host, first_centre_host, step_host,
                        uniform_tables(proj, coords, tables, k, b, mp, proj2, cx2, cy2, tables2, k2, bx, by, mp2),
                        prior_neg_half_inv_s2, prior_log_norm, out, stream);
}

int mfb_ment_prob_grid_ragged(int d, const int32_t* shape_host, const float* first_centre_host,
                              const float* step_host, const float* proj, const float* coords, const float* tables,
                              int k, const int32_t* offsets, int total, const float* mp, const float* proj2,
                              const float* cx2, const float* cy2, const float* tables2, int k2,
                              const int32_t* offsets2, const float* mp2, float prior_neg_half_inv_s2,
                              float prior_log_norm, float* out, void* stream) {
  return ment_prob_grid(
      d, shape_host, first_centre_host, step_host,
      ragged_tables(proj, coords, tables, k, offsets, total, mp, proj2, cx2, cy2, tables2, k2, offsets2, mp2),
      prior_neg_half_inv_s2, prior_log_norm, out, stream);
}

int mfb_ment_integrate(int d, const float* meas_coords, int nb_meas, int meas_axis, const float* meas_coords2,
                       int nb_meas2, int meas_axis2, int n_int_axes, const int32_t* int_shape_host,
                       const float* int_first_host, const float* int_step_host, const float* linv, const float* inv_mp,
                       const float* proj, const float* coords, const float* tables, int k, int b, const float* mp,
                       const float* proj2, const float* cx2, const float* cy2, const float* tables2, int k2, int bx,
                       int by, const float* mp2, float prior_neg_half_inv_s2, float prior_log_norm, float* pred,
                       void* stream) {
  return ment_integrate(d, meas_coords, nb_meas, meas_axis, meas_coords2, nb_meas2, meas_axis2, n_int_axes,
                        int_shape_host, int_first_host, int_step_host, linv, inv_mp,
                        uniform_tables(proj, coords, tables, k, b, mp, proj2, cx2, cy2, tables2, k2, bx, by, mp2),
                        prior_neg_half_inv_s2, prior_log_norm, pred, stream);
}

int mfb_ment_integrate_ragged(int d, const float* meas_coords, int nb_meas, int meas_axis, const float* meas_coords2,
                              int nb_meas2, int meas_axis2, int n_int_axes, const int32_t* int_shape_host,
                              const float* int_first_host, const float* int_step_host, const float* linv,
                              const float* inv_mp, const float* proj, const float* coords, const float* tables, int k,
                              const int32_t* offsets, int total, const float* mp, const float* proj2,
                              const float* cx2, const float* cy2, const float* tables2, int k2,
                              const int32_t* offsets2, const float* mp2, float prior_neg_half_inv_s2,
                              float prior_log_norm, float* pred, void* stream) {
  return ment_integrate(
      d, meas_coords, nb_meas, meas_axis, meas_coords2, nb_meas2, meas_axis2, n_int_axes, int_shape_host,
      int_first_host, int_step_host, linv, inv_mp,
      ragged_tables(proj, coords, tables, k, offsets, total, mp, proj2, cx2, cy2, tables2, k2, offsets2, mp2),
      prior_neg_half_inv_s2, prior_log_norm, pred, stream);
}

int64_t mfb_cdf_workspace_bytes(int64_t g) {
  if (g < 1) return 0;
  const int64_t ntiles = (g + kScanTile - 1) / kScanTile;
  return (((ntiles + 2) + 3) & ~(int64_t)3) * 8 + cdf_levels(g).total * 8;   // total | tile sums | scale | pivot levels
}

/* cdf[i] = sum_{j<=i} (rho[j] + pad), an exact prefix at 2^-62 of the total (scan_tile_sums_kernel); the total,
   written to workspace[0] (device), is cdf[g-1] */
int mfb_cdf_build(const float* rho, int64_t g, double pad, double* cdf, void* workspace, int64_t workspace_bytes,
                  void* stream) {
  MFB_CHECK_ARG(rho && cdf && workspace && g >= 1);
  if (workspace_bytes < mfb_cdf_workspace_bytes(g)) return MFB_E_WORKSPACE;
  const int64_t ntiles = (g + kScanTile - 1) / kScanTile;
  double* total = (double*)workspace;
  double* tiles = total + 1;            // float64 tile sums, then the uint64 unit sums, then their exclusive prefix
  double* scale = tiles + ntiles;
  cudaStream_t st = (cudaStream_t)stream;
  scan_tile_sums_kernel<false><<<(int)ntiles, kScanThreads, 0, st>>>(rho, g, pad, nullptr, tiles);
  scan_scale_kernel<<<1, 1024, 0, st>>>(tiles, ntiles, scale);
  scan_tile_sums_kernel<true><<<(int)ntiles, kScanThreads, 0, st>>>(rho, g, pad, scale, tiles);
  uint64_t* units = reinterpret_cast<uint64_t*>(tiles);
  scan_tile_offsets_kernel<<<1, 1024, 0, st>>>(units, ntiles, scale, total);
  scan_apply_kernel<<<(int)ntiles, kScanThreads, 0, st>>>(rho, g, pad, scale, units, cdf);
  const CdfLevels lv = cdf_levels(g);
  if (lv.total > 0) {
    double* pivots = (double*)workspace + (((ntiles + 2) + 3) & ~(int64_t)3);
    int64_t pb = (lv.total + 255) / 256;
    if (pb > 4096) pb = 4096;
    cdf_pivots_kernel<<<(int)pb, 256, 0, st>>>(cdf, g, lv, pivots);
  }
  return launch_status();
}

int mfb_cdf_sample(const double* cdf, int64_t g, const void* workspace, int d, const int32_t* shape_host,
                   const float* first_edge_host, const float* cell_host, int jitter, uint64_t seed, uint64_t offset,
                   int64_t size, float* out, void* stream) {
  MFB_CHECK_ARG(cdf && workspace && shape_host && first_edge_host && cell_host && out && g >= 1 && size >= 0);
  MFB_CHECK_ARG(d >= 1 && d <= kMaxDim);
  if (size == 0) return 0;
  MentGrid grid = make_grid(d, shape_host, first_edge_host, cell_host);
  const double* total = (const double*)workspace;
  const int64_t ntiles = (g + kScanTile - 1) / kScanTile;
  const CdfLevels lv = cdf_levels(g);
  const double* pivots = (const double*)workspace + (((ntiles + 2) + 3) & ~(int64_t)3);
  int64_t blocks = (size + kMentThreads - 1) / kMentThreads;
  int64_t cap = (int64_t)sm_count() * 8;
  const int gridx = (int)(blocks < cap ? blocks : cap);
  cudaStream_t st = (cudaStream_t)stream;
#define MFB_SAMPLE(DD) \
  cdf_sample_kernel<DD><<<gridx, kMentThreads, 0, st>>>(cdf, g, total, grid, jitter, seed, offset, size, out, pivots, lv)
  switch (d) {
    case 1: MFB_SAMPLE(1); break;
    case 2: MFB_SAMPLE(2); break;
    case 3: MFB_SAMPLE(3); break;
    case 4: MFB_SAMPLE(4); break;
    case 5: MFB_SAMPLE(5); break;
    case 6: MFB_SAMPLE(6); break;
    case 7: MFB_SAMPLE(7); break;
    default: MFB_SAMPLE(8); break;
  }
#undef MFB_SAMPLE
  return launch_status();
}

static int ment_mh(int d, const MentTables& t, float prior_neg_half_inv_s2, float prior_log_norm, uint64_t chain0,
                   int64_t nchains, const float* start, float start_scale, const float* chol, int64_t burnin,
                   int64_t steps, int64_t thin, uint64_t seed, float* out, int64_t* accepted, void* stream) {
  const bool kick = t.mp || t.mp2;
  MFB_CHECK_ARG(out && chol && accepted && d >= 1 && d <= kMaxDim && nchains >= 0 && mh_steps_ok(burnin, steps, thin));
  MFB_CHECK_ARG(start || isfinite(start_scale));
  MFB_CHECK_ARG((uint64_t)nchains <= UINT64_MAX - chain0 && nchains <= INT64_MAX / (steps * d) &&
                nchains <= (int64_t)INT32_MAX * kMentThreads);
  MFB_CHECK_ARG(t.ok(kick));
  if (nchains == 0) return 0;
  const MentPrior pr{prior_neg_half_inv_s2, prior_log_norm};
  const MhChains ch{chain0, nchains, start, start_scale, chol, burnin, steps, thin, seed};
  cudaStream_t st = (cudaStream_t)stream;
#define MFB_CALL(DD)                                                                                                   \
  launch_mh<DD>(kick, t.ragged, t.proj, t.coords, t.tables, t.k, t.bins(), t.off, t.off2, t.mp, t.t2, t.mp2, pr, ch,  \
                out, accepted, st)
  switch (d) {
    case 1: return MFB_CALL(1);
    case 2: return MFB_CALL(2);
    case 3: return MFB_CALL(3);
    case 4: return MFB_CALL(4);
    case 5: return MFB_CALL(5);
    case 6: return MFB_CALL(6);
    case 7: return MFB_CALL(7);
    default: return MFB_CALL(8);
  }
#undef MFB_CALL
}

int mfb_ment_mh(int d, const float* proj, const float* coords, const float* tables, int k, int b, const float* mp,
                const float* proj2, const float* cx2, const float* cy2, const float* tables2, int k2, int bx, int by,
                const float* mp2, float prior_neg_half_inv_s2, float prior_log_norm, uint64_t chain0, int64_t nchains,
                const float* start, float start_scale, const float* chol, int64_t burnin, int64_t steps, int64_t thin,
                uint64_t seed, float* out, int64_t* accepted, void* stream) {
  return ment_mh(d, uniform_tables(proj, coords, tables, k, b, mp, proj2, cx2, cy2, tables2, k2, bx, by, mp2),
                 prior_neg_half_inv_s2, prior_log_norm, chain0, nchains, start, start_scale, chol, burnin, steps, thin,
                 seed, out, accepted, stream);
}

int mfb_ment_mh_ragged(int d, const float* proj, const float* coords, const float* tables, int k,
                       const int32_t* offsets, int total, const float* mp, const float* proj2, const float* cx2,
                       const float* cy2, const float* tables2, int k2, const int32_t* offsets2, const float* mp2,
                       float prior_neg_half_inv_s2, float prior_log_norm, uint64_t chain0, int64_t nchains,
                       const float* start, float start_scale, const float* chol, int64_t burnin, int64_t steps,
                       int64_t thin, uint64_t seed, float* out, int64_t* accepted, void* stream) {
  return ment_mh(d,
                 ragged_tables(proj, coords, tables, k, offsets, total, mp, proj2, cx2, cy2, tables2, k2, offsets2, mp2),
                 prior_neg_half_inv_s2, prior_log_norm, chain0, nchains, start, start_scale, chol, burnin, steps, thin,
                 seed, out, accepted, stream);
}

int mfb_mh_propose(const float* x, int64_t n, int d, uint64_t chain0, const float* start, float start_scale,
                   const float* chol, int64_t t, uint64_t seed, float* xp, void* stream) {
  MFB_CHECK_ARG(xp && n >= 0 && d >= 1 && d <= kMaxDim && t >= 0 && t <= (int64_t)UINT32_MAX);
  MFB_CHECK_ARG(t == 0 ? (start || isfinite(start_scale)) : (x && chol));
  MFB_CHECK_ARG((uint64_t)n <= UINT64_MAX - chain0);
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
#define MFB_CALL(DD) \
  mh_propose_kernel<DD><<<mh_grid(n), kMentThreads, 0, st>>>(x, n, chain0, start, start_scale, chol, (uint32_t)t, seed, xp)
  switch (d) {
    case 1: MFB_CALL(1); break;
    case 2: MFB_CALL(2); break;
    case 3: MFB_CALL(3); break;
    case 4: MFB_CALL(4); break;
    case 5: MFB_CALL(5); break;
    case 6: MFB_CALL(6); break;
    case 7: MFB_CALL(7); break;
    default: MFB_CALL(8); break;
  }
#undef MFB_CALL
  return launch_status();
}

int mfb_mh_accept(float* x, float* rho, const float* xp, const float* rho_prop, int64_t n, int d, uint64_t chain0,
                  int64_t t, uint64_t seed, int64_t* accepted, void* stream) {
  MFB_CHECK_ARG(x && rho && xp && rho_prop && accepted && n >= 0 && d >= 1 && d <= kMaxDim);
  MFB_CHECK_ARG(t >= 1 && t <= (int64_t)UINT32_MAX && (uint64_t)n <= UINT64_MAX - chain0);
  if (n == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* acc = reinterpret_cast<unsigned long long*>(accepted);
#define MFB_CALL(DD) \
  mh_accept_kernel<DD><<<mh_grid(n), kMentThreads, 0, st>>>(x, rho, xp, rho_prop, n, chain0, (uint32_t)t, seed, acc)
  switch (d) {
    case 1: MFB_CALL(1); break;
    case 2: MFB_CALL(2); break;
    case 3: MFB_CALL(3); break;
    case 4: MFB_CALL(4); break;
    case 5: MFB_CALL(5); break;
    case 6: MFB_CALL(6); break;
    case 7: MFB_CALL(7); break;
    default: MFB_CALL(8); break;
  }
#undef MFB_CALL
  return launch_status();
}

int mfb_gs_update(float* table, const float* meas, const float* pred, int n, float lr, float thresh, void* stream) {
  MFB_CHECK_ARG(table && meas && pred && n >= 1);
  gs_update_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(table, meas, pred, n, lr, thresh);
  return launch_status();
}

}  // extern "C"
