// Fused linear projection + 2-D binning (separable Gaussian KDE deposit or exact histogram).
//
// Replaces (reference file:line, relative to mentflow/):
//   simulate/simulate.py:29-33, simulate/transform.py:67-68    u = x.clone() @ M_k^T
//   diagnostics/diagnostics.py:179-191                         u[:, axis] -> kde_histogram_2d
//   diagnostics/histogram.py:89-101, 47-74                     two (N,B) kernel matrices, Kx^T Ky SGEMM
//   diagnostics/diagnostics.py:192-201                         np.histogramdd on the host
//
// Design: one CTA = one screen x one contiguous block of particles; the screen's (Bx, By) bins
// live in shared memory.  Each particle deposits the (2R+1)^2 window of Kx_a * Ky_b around its
// image.  Deposits are accumulated as *fixed point* integers (44 fractional bits, split into
// two 22-bit halves held in two u32 tables) with native shared-memory integer atomics
// (ATOMS.ADD; on sm_100a both fp32 and 64-bit shared atomicAdd compile to CAS spin loops):
// integer addition is associative, so the result does not depend on the order of the atomics,
// the CTA decomposition, or the number of ranks (bit-reproducible).  44 bits keep the far
// Gaussian tails (6e-14 per deposit) that the KL's log(p + 1e-12) is sensitive to.  The per-CTA
// tables are flushed to 64-bit global accumulators before they could overflow.
#include "common.cuh"

namespace mfb {

constexpr int kHalfBits = MFB_KDE2D_FRAC_BITS / 2;  // 44 = 22 (high table) + 22 (low table)
constexpr float kHalfScale = 4194304.0f;            // 2^22
constexpr int k2dThreads = 256;
constexpr int kFlushParticles = 1024 - 256;         // 768 * 2^22 < 2^32, 768 * 2^21 < 2^31: no overflow

struct Axis {
  float c0, inv_delta, alpha, beta;  // beta = -delta / sigma^2
};

__device__ __forceinline__ Axis load_axis(const float* g) {
  Axis a;
  a.c0 = g[0];
  a.inv_delta = 1.0f / g[1];
  const float r = g[1] / g[2];
  a.alpha = -0.5f * r * r * kLog2e;
  a.beta = -g[1] / (g[2] * g[2]);
  return a;
}

template <int R>
__device__ __forceinline__ void window(const Axis& ax, float u, int nb, int& b0, float (&val)[2 * R + 1],
                                       float (&tt)[2 * R + 1]) {
  float a = (u - ax.c0) * ax.inv_delta;
  a = fminf(fmaxf(a, -(float)(R + 2)), (float)(nb + R + 1));
  const float fb = rintf(a);
  b0 = (int)fb;
  const float f = a - fb;
#pragma unroll
  for (int j = -R; j <= R; ++j) {
    const float t = f - (float)j;
    tt[j + R] = t;
    val[j + R] = fast_exp2(ax.alpha * t * t);
  }
}

// The same window by the tap recurrences of the 1-D kernels (kde1d.cu): the value at offset 0 is E = 2^(alpha f^2), the
// ratio from offset j-1 to j is 2^(alpha (2j - 1 - 2f)) = su c_j (up) and from -(j-1) to -j 2^(alpha (2j - 1 + 2f)) =
// sd c_j (down), su = 2^(alpha (1 - 2f)), sd = 2^(alpha (1 + 2f)), c_j = 2^(2 alpha (j - 1)).  |f| <= 1/2 keeps every
// factor <= 1, so nothing overflows at any bandwidth -- three MUFU per axis instead of 2R+1 --, the c_j do not depend on
// the particle (the compiler keeps them across the particles of a screen), and the nearest bin comes through the
// 1.5 * 2^23 rounding constant.
template <int R>
__device__ __forceinline__ void window_fact(const Axis& ax, float u, int nb, int& b0, float (&val)[2 * R + 1],
                                            float (&tt)[2 * R + 1]) {
  float a = (u - ax.c0) * ax.inv_delta;
  a = fminf(fmaxf(a, -(float)(R + 2)), (float)(nb + R + 1));
  const float shifted = a + 12582912.0f;
  const float fb = shifted - 12582912.0f;
  b0 = __float_as_int(shifted) - 0x4B400000;
  const float f = a - fb, af = ax.alpha * f;
  const float e0 = fast_exp2(af * f);
  const float su = fast_exp2(fmaf(-2.0f, af, ax.alpha)), sd = fast_exp2(fmaf(2.0f, af, ax.alpha));
  const float c2 = exp2f(2.0f * ax.alpha);
  val[R] = e0;
  tt[R] = f;
  float up = e0 * su, dn = e0 * sd, c = c2;
  val[R + 1] = up;
  val[R - 1] = dn;
  tt[R + 1] = f - 1.0f;
  tt[R - 1] = f + 1.0f;
#pragma unroll
  for (int j = 2; j <= R; ++j) {
    up *= su * c;
    dn *= sd * c;
    c *= c2;
    val[R + j] = up;
    val[R - j] = dn;
    tt[R + j] = f - (float)j;
    tt[R - j] = f + (float)j;
  }
}

template <int R>
__global__ void __launch_bounds__(k2dThreads)
kde2d_deposit_kernel(const float* __restrict__ x, int64_t n, int d, const float* __restrict__ proj,
                     const float* __restrict__ geom, int BX, int BY, int64_t chunk,
                     unsigned long long* __restrict__ acc /* [2][K][BX][BY]: high, low */, int64_t acc_len) {
  extern __shared__ __align__(16) unsigned int s_bins[];
  __shared__ float s_w[2 * kMaxDim];
  const int k = blockIdx.y;
  const int nbins = BX * BY;
  unsigned int* s_hi = s_bins;                              // units of 2^-22
  int* s_lo = reinterpret_cast<int*>(s_bins + nbins);       // signed, units of 2^-44
  for (int i = threadIdx.x; i < 2 * nbins; i += k2dThreads) s_bins[i] = 0u;
  if (threadIdx.x < 2 * d) s_w[threadIdx.x] = proj[(size_t)k * 2 * d + threadIdx.x];
  const Axis ax = load_axis(geom + (size_t)(2 * k) * MFB_GEOM_STRIDE);
  const Axis ay = load_axis(geom + (size_t)(2 * k + 1) * MFB_GEOM_STRIDE);
  __syncthreads();

  const int64_t first = (int64_t)blockIdx.x * chunk;
  int64_t last = first + chunk;
  if (last > n) last = n;
  unsigned long long* out = acc + (size_t)k * nbins;

  for (int64_t base = first; base < last; base += kFlushParticles) {
    int64_t stop = base + kFlushParticles;
    if (stop > last) stop = last;
    for (int64_t p = base + threadIdx.x; p < stop; p += k2dThreads) {
      float ux = 0.f, uy = 0.f;
      for (int i = 0; i < d; ++i) {
        const float xi = x[p * d + i];
        ux = fmaf(s_w[i], xi, ux);
        uy = fmaf(s_w[d + i], xi, uy);
      }
      int bx0, by0;
      float vx[2 * R + 1], vy[2 * R + 1], tx[2 * R + 1], ty[2 * R + 1];
      window<R>(ax, ux, BX, bx0, vx, tx);
      window<R>(ay, uy, BY, by0, vy, ty);
#pragma unroll
      for (int ja = 0; ja <= 2 * R; ++ja) {
        const int a = bx0 + ja - R;
        if ((unsigned)a < (unsigned)BX) {
          const float sx = vx[ja] * kHalfScale;
          const int rowoff = a * BY;
#pragma unroll
          for (int jb = 0; jb <= 2 * R; ++jb) {
            const int b = by0 + jb - R;
            // v * 2^44 = hi * 2^22 + lo with hi = rint(v 2^22), lo = rint((v 2^22 - hi) 2^22)
            const float v22 = sx * vy[jb];
            const float hif = rintf(v22);
            const int lo = __float2int_rn((v22 - hif) * kHalfScale);
            const unsigned int hi = (unsigned int)hif;
            if ((unsigned)b < (unsigned)BY) {
              if (hi) atomicAdd(s_hi + rowoff + b, hi);
              if (lo) atomicAdd(s_lo + rowoff + b, lo);
            }
          }
        }
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += k2dThreads) {
      const unsigned int h = s_hi[i];
      const int l = s_lo[i];
      if (h) {
        atomicAdd(out + i, (unsigned long long)h);
        s_hi[i] = 0u;
      }
      if (l) {
        atomicAdd(out + acc_len + i, (unsigned long long)(long long)l);
        s_lo[i] = 0;
      }
    }
    __syncthreads();
  }
}

__global__ void fixed_to_float_kernel(const unsigned long long* __restrict__ acc, int64_t len,
                                      float* __restrict__ sums) {
  const double sh = 1.0 / (double)(1ull << kHalfBits);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < len; i += (int64_t)gridDim.x * blockDim.x)
    sums[i] = (float)(((double)(long long)acc[i] + (double)(long long)acc[len + i] * sh) * sh);
}

// ---- normalisation P / (sum(P) dx dy + 1e-10) and its backward: one CTA per screen -------------
__device__ __forceinline__ float block_sum_2d(float v, float* red) {
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

__global__ void __launch_bounds__(256)
kde2d_normalize_kernel(const float* __restrict__ sums, const float* __restrict__ geom, int nbins,
                       float* __restrict__ prof) {
  __shared__ float red[33];
  const int k = blockIdx.x;
  const float dx = geom[(size_t)(2 * k) * MFB_GEOM_STRIDE + 3], dy = geom[(size_t)(2 * k + 1) * MFB_GEOM_STRIDE + 3];
  const float* s = sums + (size_t)k * nbins;
  float acc = 0.f;
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) acc += s[i] * dx * dy;
  const float z = block_sum_2d(acc, red) + 1.0e-10f;
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) prof[(size_t)k * nbins + i] = s[i] / z;
}

__global__ void __launch_bounds__(256)
kde2d_normalize_bwd_kernel(const float* __restrict__ sums, const float* __restrict__ geom, int nbins,
                           const float* __restrict__ gprof, float* __restrict__ gsums) {
  __shared__ float red[33];
  const int k = blockIdx.x;
  const float dx = geom[(size_t)(2 * k) * MFB_GEOM_STRIDE + 3], dy = geom[(size_t)(2 * k + 1) * MFB_GEOM_STRIDE + 3];
  const float* s = sums + (size_t)k * nbins;
  const float* gp = gprof + (size_t)k * nbins;
  float acc = 0.f;
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) acc += s[i] * dx * dy;
  const float z = block_sum_2d(acc, red) + 1.0e-10f;
  float dot = 0.f;
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) dot += gp[i] * (s[i] / z);
  const float g = block_sum_2d(dot, red);
  // p = S / Z, Z = dx dy sum S + eps  =>  dL/dS_i = gp_i / Z - dx dy (sum_j gp_j p_j) / Z
  for (int i = threadIdx.x; i < nbins; i += blockDim.x) gsums[(size_t)k * nbins + i] = gp[i] / z - dx * dy * g / z;
}

// ---- backward w.r.t. particles: CTA keeps its particles in registers, loops over screens --------
template <int R>
__global__ void __launch_bounds__(k2dThreads)
kde2d_bwd_kernel(const float* __restrict__ x, int64_t n, int d, const float* __restrict__ proj,
                 const float* __restrict__ geom, int K, int BX, int BY, const float* __restrict__ gsums,
                 float* __restrict__ gx, int accumulate) {
  // gradient table of the current screen with kPad zero bins around it: the (2R+1)^2 taps of a (clamped) particle never
  // need a bounds check
  constexpr int kPad = 2 * R + 2;
  extern __shared__ __align__(16) float s_g[];  // [BX + 2 kPad][BY + 2 kPad]
  __shared__ float s_w[2 * kMaxDim];
  __shared__ float s_geo[2 * MFB_GEOM_STRIDE];
  const int nbins = BX * BY, BYP = BY + 2 * kPad;
  for (int i = threadIdx.x; i < (BX + 2 * kPad) * BYP; i += k2dThreads) s_g[i] = 0.f;   // the pads stay zero
  // kPT particles per thread: a screen's gradient table (BX x BY floats, 29 KB at 85 x 85) is loaded into shared memory
  // once per kPT x 256 particles -- with one particle per thread the kernel was bound by re-reading the tables from
  // L2 (15 x 29 KB per 256 particles), not by its arithmetic
  constexpr int kPT = 4;
  for (int64_t p0 = (int64_t)blockIdx.x * (k2dThreads * kPT); p0 < n; p0 += (int64_t)gridDim.x * (k2dThreads * kPT)) {
    float xr[kPT][kMaxDim], g[kPT][kMaxDim];
    bool valid[kPT];
#pragma unroll
    for (int q = 0; q < kPT; ++q) {
      const int64_t p = p0 + q * k2dThreads + threadIdx.x;
      valid[q] = p < n;
#pragma unroll
      for (int i = 0; i < kMaxDim; ++i) {
        xr[q][i] = (valid[q] && i < d) ? x[p * d + i] : 0.f;
        g[q][i] = 0.f;
      }
    }
    for (int k = 0; k < K; ++k) {
      __syncthreads();
      for (int i = threadIdx.x; i < nbins; i += k2dThreads) {
        const int a = i / BY, b = i - a * BY;
        s_g[(a + kPad) * BYP + (b + kPad)] = gsums[(size_t)k * nbins + i];
      }
      if (threadIdx.x < 2 * d) s_w[threadIdx.x] = proj[(size_t)k * 2 * d + threadIdx.x];
      if (threadIdx.x < 2 * MFB_GEOM_STRIDE) s_geo[threadIdx.x] = geom[(size_t)(2 * k) * MFB_GEOM_STRIDE + threadIdx.x];
      __syncthreads();
      const Axis ax = load_axis(s_geo), ay = load_axis(s_geo + MFB_GEOM_STRIDE);
#pragma unroll 1
      for (int q = 0; q < kPT; ++q) {
        float ux = 0.f, uy = 0.f;
#pragma unroll
        for (int i = 0; i < kMaxDim; ++i)
          if (i < d) {
            ux = fmaf(s_w[i], xr[q][i], ux);
            uy = fmaf(s_w[d + i], xr[q][i], uy);
          }
        int bx0, by0;
        float vx[2 * R + 1], vy[2 * R + 1], tx[2 * R + 1], ty[2 * R + 1];
        window_fact<R>(ax, ux, BX, bx0, vx, tx);
        window_fact<R>(ay, uy, BY, by0, vy, ty);
        float gux = 0.f, guy = 0.f;
        const float* base = s_g + (bx0 - R + kPad) * BYP + (by0 - R + kPad);
#pragma unroll
        for (int ja = 0; ja <= 2 * R; ++ja) {
          const float* row = base + ja * BYP;
          float r0 = 0.f, r1 = 0.f;  // sum_b g_ab Ky_b  and  sum_b g_ab Ky_b ty_b
#pragma unroll
          for (int jb = 0; jb <= 2 * R; ++jb) {
            const float gv = row[jb] * vy[jb];
            r0 += gv;
            r1 = fmaf(gv, ty[jb], r1);
          }
          gux = fmaf(vx[ja] * tx[ja], r0, gux);
          guy = fmaf(vx[ja], r1, guy);
        }
        gux *= ax.beta;
        guy *= ay.beta;
#pragma unroll
        for (int i = 0; i < kMaxDim; ++i)
          if (i < d) g[q][i] = fmaf(s_w[i], gux, fmaf(s_w[d + i], guy, g[q][i]));
      }
    }
#pragma unroll
    for (int q = 0; q < kPT; ++q) {
      if (!valid[q]) continue;
      const int64_t p = p0 + q * k2dThreads + threadIdx.x;
#pragma unroll
      for (int i = 0; i < kMaxDim; ++i)
        if (i < d) {
          if (accumulate) gx[p * d + i] += g[q][i];
          else gx[p * d + i] = g[q][i];
        }
    }
  }
}

// ---- exact 2-D histogram ----------------------------------------------------------------------------
__device__ __forceinline__ int exact_bin(const float* E, int nb, float u) {
  // e[i] <= u < e[i+1], last bin closed; -1 if outside / NaN
  if (!(u >= E[0] && u <= E[nb])) return -1;
  int b = (int)((u - E[0]) * ((float)nb / (E[nb] - E[0])));
  b = min(max(b, 0), nb - 1);
  while (b > 0 && u < E[b]) --b;
  while (b < nb - 1 && u >= E[b + 1]) ++b;
  return b;
}

__global__ void __launch_bounds__(k2dThreads)
hist2d_deposit_kernel(const float* __restrict__ x, int64_t n, int d, const float* __restrict__ proj,
                      const float* __restrict__ edges_x, const float* __restrict__ edges_y, int BX, int BY,
                      int64_t chunk, unsigned long long* __restrict__ counts) {
  extern __shared__ __align__(16) unsigned int s_bins[];
  __shared__ float s_w[2 * kMaxDim];
  const int k = blockIdx.y;
  const int nbins = BX * BY;
  float* s_ex = reinterpret_cast<float*>(s_bins + nbins);
  float* s_ey = s_ex + BX + 1;
  for (int i = threadIdx.x; i < nbins; i += k2dThreads) s_bins[i] = 0u;
  for (int i = threadIdx.x; i <= BX; i += k2dThreads) s_ex[i] = edges_x[(size_t)k * (BX + 1) + i];
  for (int i = threadIdx.x; i <= BY; i += k2dThreads) s_ey[i] = edges_y[(size_t)k * (BY + 1) + i];
  if (threadIdx.x < 2 * d) s_w[threadIdx.x] = proj[(size_t)k * 2 * d + threadIdx.x];
  __syncthreads();
  const int64_t first = (int64_t)blockIdx.x * chunk;
  int64_t last = first + chunk;
  if (last > n) last = n;
  for (int64_t p = first + threadIdx.x; p < last; p += k2dThreads) {
    float ux = 0.f, uy = 0.f;
    for (int i = 0; i < d; ++i) {
      const float xi = x[p * d + i];
      ux = fmaf(s_w[i], xi, ux);
      uy = fmaf(s_w[d + i], xi, uy);
    }
    const int a = exact_bin(s_ex, BX, ux);
    const int b = exact_bin(s_ey, BY, uy);
    if (a >= 0 && b >= 0) atomicAdd(s_bins + a * BY + b, 1u);
  }
  __syncthreads();
  unsigned long long* out = counts + (size_t)k * nbins;
  for (int i = threadIdx.x; i < nbins; i += k2dThreads) {
    const unsigned int v = s_bins[i];
    if (v) atomicAdd(out + i, (unsigned long long)v);
  }
}

// particle block per CTA so that grid.x * K fills the machine a few times over
static int64_t plan_chunk(int64_t n, int k, int* grid_x) {
  const int sms = sm_count();
  int64_t want = ((int64_t)sms * 8 + k - 1) / k;  // CTAs along the particle axis
  if (want < 1) want = 1;
  int64_t chunk = (n + want - 1) / want;
  // keep chunks a multiple of the block size and below 2^31 particles
  chunk = ((chunk + k2dThreads - 1) / k2dThreads) * k2dThreads;
  if (chunk < k2dThreads) chunk = k2dThreads;
  if (chunk > (1ll << 30)) chunk = 1ll << 30;
  *grid_x = (int)((n + chunk - 1) / chunk);
  return chunk;
}

}  // namespace mfb

using namespace mfb;

static int radius2d(float hint) {
  double r = 8.85 * (hint > 0.f ? hint : 0.5) - 0.5;  // see kde1d.cu window_radius
  int ri = (int)r;
  if ((double)ri < r) ++ri;
  return ri < 1 ? 1 : ri;
}

// tensor-core path (kde2d_tc.cu): dense kernel rows as tcgen05 operands, screens up to 128 x 96 bins
namespace mfb {
bool kde2d_tc_supported(int64_t n, int d, int bx, int by);
int64_t kde2d_tc_partial_bytes(int k, int bx, int by);
int kde2d_tc_forward(const float* x, int64_t n, int d, const float* proj, const float* geom, int k, int bx, int by,
                     float* sums, unsigned long long* acc, float* partial, cudaStream_t st);
}  // namespace mfb

extern "C" {

int64_t mfb_kde2d_workspace_bytes(int64_t n, int d, int k, int bx, int by) {
  (void)n;
  (void)d;
  if (k < 1 || bx < 1 || by < 1) return 0;
  // two int64 planes (units 2^-22 and 2^-44) + the per-CTA partial screens of the tensor-core path
  return (int64_t)k * bx * by * 16 + kde2d_tc_partial_bytes(k, bx, by);
}

int mfb_kde2d_uses_tensor_cores(int64_t n, int d, int bx, int by, int flags) {
  return !(flags & MFB_FLAG_NO_TENSOR_CORES) && kde2d_tc_supported(n, d, bx, by) ? 1 : 0;
}

int mfb_project_kde2d_fwd(const float* x, int64_t n, int d, const float* proj, const float* geom, int k, int bx,
                          int by, float max_sigma_over_delta, float* sums, void* workspace,
                          int64_t workspace_bytes, int flags, void* stream) {
  MFB_CHECK_ARG(x && proj && geom && sums && workspace);
  MFB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim && k >= 1 && bx >= 2 && by >= 2);
  const int64_t len = (int64_t)k * bx * by;
  if (workspace_bytes < len * 16) return MFB_E_WORKSPACE;
  const size_t smem = (size_t)bx * by * 8;  // two u32 tables
  if (smem > 200 * 1024) return MFB_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* acc = (unsigned long long*)workspace;
  if (mfb_kde2d_uses_tensor_cores(n, d, bx, by, flags) &&
      workspace_bytes >= len * 16 + kde2d_tc_partial_bytes(k, bx, by)) {
    float* partial = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(workspace) + len * 16);
    return kde2d_tc_forward(x, n, d, proj, geom, k, bx, by, sums, acc, partial, st);
  }
  MFB_CUDA(cudaMemsetAsync(acc, 0, (size_t)len * 16, st));
  if (n > 0) {
    int gx;
    const int64_t chunk = plan_chunk(n, k, &gx);
    dim3 grid(gx, k);
    const int r = radius2d(max_sigma_over_delta);
    if (r <= 4) {
      MFB_CUDA(cudaFuncSetAttribute(kde2d_deposit_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kde2d_deposit_kernel<4><<<grid, k2dThreads, smem, st>>>(x, n, d, proj, geom, bx, by, chunk, acc, len);
    } else if (r <= 9) {
      MFB_CUDA(cudaFuncSetAttribute(kde2d_deposit_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kde2d_deposit_kernel<9><<<grid, k2dThreads, smem, st>>>(x, n, d, proj, geom, bx, by, chunk, acc, len);
    } else {
      return MFB_E_UNSUPPORTED;
    }
    int rc = launch_status();
    if (rc) return rc;
  }
  int fgrid = (int)((len + 255) / 256);
  if (fgrid > 4096) fgrid = 4096;
  fixed_to_float_kernel<<<fgrid, 256, 0, st>>>(acc, len, sums);
  return launch_status();
}

int mfb_kde2d_normalize(const float* sums, const float* geom, int k, int bx, int by, float* profiles, void* stream) {
  MFB_CHECK_ARG(sums && geom && profiles && k >= 1 && bx >= 2 && by >= 2);
  kde2d_normalize_kernel<<<k, 256, 0, (cudaStream_t)stream>>>(sums, geom, bx * by, profiles);
  return launch_status();
}

int mfb_kde2d_normalize_bwd(const float* sums, const float* geom, int k, int bx, int by, const float* gprof,
                            float* gsums, void* stream) {
  MFB_CHECK_ARG(sums && geom && gprof && gsums && k >= 1 && bx >= 2 && by >= 2);
  kde2d_normalize_bwd_kernel<<<k, 256, 0, (cudaStream_t)stream>>>(sums, geom, bx * by, gprof, gsums);
  return launch_status();
}

int mfb_project_kde2d_bwd(const float* x, int64_t n, int d, const float* proj, const float* geom, int k, int bx,
                          int by, float max_sigma_over_delta, const float* gsums, float* gx, int accumulate,
                          void* stream) {
  MFB_CHECK_ARG(x && proj && geom && gsums && gx);
  MFB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim && k >= 1 && bx >= 2 && by >= 2);
  if (n == 0) return 0;
  const int rr_ = radius2d(max_sigma_over_delta);
  const int pad = 2 * (rr_ <= 4 ? 4 : 9) + 2;                     // kPad of the template radius the launch picks
  const size_t smem = (size_t)(bx + 2 * pad) * (by + 2 * pad) * 4;
  if (smem > 200 * 1024) return MFB_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  int per_sm = (int)((200 * 1024) / (smem + 2048));
  if (per_sm < 1) per_sm = 1;
  if (per_sm > 6) per_sm = 6;
  int64_t grid = (int64_t)sm_count() * per_sm;
  const int64_t blocks = (n + 4 * k2dThreads - 1) / (4 * k2dThreads);   // four particles per thread (kPT)
  if (grid > blocks) grid = blocks;
  const int r = radius2d(max_sigma_over_delta);
  if (r <= 4) {
    MFB_CUDA(cudaFuncSetAttribute(kde2d_bwd_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kde2d_bwd_kernel<4><<<(int)grid, k2dThreads, smem, st>>>(x, n, d, proj, geom, k, bx, by, gsums, gx, accumulate);
  } else if (r <= 9) {
    MFB_CUDA(cudaFuncSetAttribute(kde2d_bwd_kernel<9>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kde2d_bwd_kernel<9><<<(int)grid, k2dThreads, smem, st>>>(x, n, d, proj, geom, k, bx, by, gsums, gx, accumulate);
  } else {
    return MFB_E_UNSUPPORTED;
  }
  return launch_status();
}

int mfb_project_hist2d(const float* x, int64_t n, int d, const float* proj, const float* edges_x,
                       const float* edges_y, int k, int bx, int by, int64_t* counts, void* stream) {
  MFB_CHECK_ARG(x && proj && edges_x && edges_y && counts);
  MFB_CHECK_ARG(n >= 0 && d >= 1 && d <= kMaxDim && k >= 1 && bx >= 1 && by >= 1);
  if (n == 0) return 0;
  const size_t smem = (size_t)bx * by * 4 + (size_t)(bx + by + 2) * 4;
  if (smem > 200 * 1024) return MFB_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  int gx;
  const int64_t chunk = plan_chunk(n, k, &gx);
  dim3 grid(gx, k);
  MFB_CUDA(cudaFuncSetAttribute(hist2d_deposit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  hist2d_deposit_kernel<<<grid, k2dThreads, smem, st>>>(x, n, d, proj, edges_x, edges_y, bx, by, chunk,
                                                       reinterpret_cast<unsigned long long*>(counts));
  return launch_status();
}

}  // extern "C"
