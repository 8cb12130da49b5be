// Thin multipole kick folded into a projection: shared by the KDE kernels (kde1d.cu) and the classical MENT
// density (ment.cu).
#pragma once

#include "common.cuh"

namespace mfb {

// ---- thin multipole kick folded into the projection ---------------------------------------------
// For a transfer map  linear -> MultipoleTransform -> linear  (mentflow/simulate/transform.py:78-146,
// experiments/rec_2d/nonlinear/setup.py:24-44) the measured coordinate is
//   u = w . x + a Re(z^m) + b Im(z^m),   z = (wa . x) + i (wb . x),   m = order - 1,
// with w, wa, wb, a, b built on the host from the matrices and the kick strength (the reference's
// U[:,3] = X[:,1] + ... quirk is linear and lives in w).  mp row = [wa (d) | wb (d) | a | b | order | 0].
#define MFB_MP_STRIDE(d) (2 * (d) + 4)
struct MpTerms {
  float wa[kMaxDim], wb[kMaxDim];
  float a, b;
  int m;   // power of z
};
__device__ __forceinline__ void load_mp(MpTerms& t, const float* __restrict__ row, int d) {
#pragma unroll
  for (int i = 0; i < kMaxDim; ++i) {
    t.wa[i] = i < d ? row[i] : 0.f;
    t.wb[i] = i < d ? row[d + i] : 0.f;
  }
  t.a = row[2 * d];
  t.b = row[2 * d + 1];
  t.m = (int)row[2 * d + 2] - 1;
}
// z^m and z^(m-1) (m >= 1) by repeated complex multiplication
__device__ __forceinline__ void zpow(float xm, float ym, int m, float& zr, float& zi, float& pr, float& pi) {
  zr = 1.f; zi = 0.f; pr = 1.f; pi = 0.f;
  for (int t = 0; t < m; ++t) {
    pr = zr; pi = zi;
    const float nr = zr * xm - zi * ym, ni = zr * ym + zi * xm;
    zr = nr; zi = ni;
  }
}
__device__ __forceinline__ float project_row_mp(const float* __restrict__ xr, const float (&w)[kMaxDim], const MpTerms& t,
                                                int d) {
  float u = 0.f, xm = 0.f, ym = 0.f;
#pragma unroll
  for (int i = 0; i < kMaxDim; ++i)
    if (i < d) {
      u = fmaf(w[i], xr[i], u);
      xm = fmaf(t.wa[i], xr[i], xm);
      ym = fmaf(t.wb[i], xr[i], ym);
    }
  float zr, zi, pr, pi;
  zpow(xm, ym, t.m, zr, zi, pr, pi);
  return fmaf(t.b, zi, fmaf(t.a, zr, u));
}

}  // namespace mfb
