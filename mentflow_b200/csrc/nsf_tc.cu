// Neural spline flow layer on the 5th-generation tensor cores (tcgen05 + TMEM), sm_100a.
//
// Replaces, per autoregressive layer, the same reference work as nsf.cu (generate/flows/zuko.py:24-29
// -> zuko 1.3.1 MaskedMLP + MonotonicRQSTransform.call_and_ladj; SURVEY.md App. A): the four masked
// GEMMs of the conditioner run as tcgen05.mma tiles (M = 128 particles, fp32 inputs split into fp16
// (hi, lo) pairs, three MMAs per K step, fp32 accumulators in TMEM), and the rational-quadratic spline
// with its log|det J| is the epilogue of the output-layer tile: parameters go TMEM -> registers and
// never touch shared memory or HBM.
//
// CTA = 3 compute warpgroups + 1 MMA-issuer warpgroup (setmaxnreg: 160 / 32 registers), persistent,
// one CTA per SM.  The layer's weights live in shared memory as ready-made fp16 operand tiles (an
// "image" built by nsf_tc_prepare_kernel, loaded with one TMA bulk copy).  Every compute warpgroup owns
// one 128-particle tile at a time, its own A-operand buffer (activations, hi|lo) and its own 128 TMEM
// columns, and walks
//   v -> [L1 MMA] -> relu/split -> [L2 MMA] -> relu/split -> [L3 MMA] -> relu/split ->
//        per feature: [output MMA, N = 64] -> spline epilogue          (double buffered in TMEM)
// software-pipelined over its tiles (the chain of tile i+1 runs between the last splines of tile i);
// warp i of the issuer warpgroup issues the MMAs that compute warpgroup i requests through
// mbarriers.  Biases enter the accumulators through an extra "ones x bias" MMA.
//
// Mask awareness: hidden units are re-ordered by autoregressive class (a permutation of the hidden
// layer, applied when the image is built), which makes every masked weight matrix block lower
// triangular; K steps whose weights are all zero for a block of outputs are not issued (14 of 20
// output-layer K steps at D = 6).  The feature that is first in the layer's order has a bias-only
// spline: its knots are precomputed into a table in the image.
//
// Also in this file, on the same machinery: the backward variant of the layer kernel (kBwd: recompute + spline
// backward, writes the compact dL/dphi rows, ReLU masks and a bulk-copied mirror of the activation operand tiles for
// nsf_tc_bwd.cu), the forward variant's A hi operand in tensor memory (tcgen05.st + TMEM-A MMAs), programmatic
// dependent launch of consecutive layers, and nsf_tc_inverse_kernel (density direction: one conditioner pass plus a
// register-resident inverse spline per feature).
#include "nsf_spline_regs.cuh"
#include "nsf_tc_common.cuh"

namespace mfb {
namespace tc {


struct Meta {
  int slot_feature[kMaxDim];  // feature handled by output slot s (order > 0, ascending order)
  int slot_ksteps[kMaxDim];   // K steps (of 16 hidden units) with non-zero weights for slot s
  int hid_n0[4];              // hidden->hidden: first output row that reads K step s (multiple of 16)
  int const_feature;          // feature with order 0 (bias-only spline)
  int nslots;
  int perm[kH];               // original hidden unit at sorted position c (backward: global rows of the activations)
};

// pointers of the backward variant (recompute + spline backward).  Workspace matrices are tile-major:
// element (row r, particle p) of a matrix with R rows sits at ((p / 128) * R + r) * 128 + p % 128, so
// the rows of one 128-particle tile are contiguous (512 B each) and every row is a ready K-major
// operand row for the weight-gradient GEMMs.
struct BwdIO {
  const float* gy;      // [n][D] dL/dy
  const float* glogq;   // [n] dL/dlogq_out or null
  float* acts;          // per tile and hidden layer: the 32 KB (hi, lo) fp16 operand tile of the post-ReLU activations
                        // ([128 particles][64 units in sorted order], SWIZZLE_128B) -- see store_hidden
  float* gphi;          // D*kGRows rows: dL/d(raw conditioner output), compact (nsf_tc_common.cuh)
  uint32_t* masks;      // 3 x 2 rows: ReLU masks of the hidden layers (bit c of word w = unit perm[32 w + c] is active)
  float* gvd;           // [n][D] direct dL/dv through the spline (+ base density term)
  float* gmax;          // [n] max |gphi| of the particle
  int* gmaxes;          // [0]: batch maximum of |gphi| (float bits, atomicMax)
};

struct PrepMeta {             // per layer: which feature each output slot serves
  int slot_feature[kMaxDim];
  int const_feature;
  int nslots;
};
constexpr int kMaxPrepLayers = 16;
struct PrepArgs {             // by-value kernel argument (no host->device copy, graph-capturable)
  int perm[kH];               // perm[p] = original hidden unit stored at sorted position p (same for every layer)
  PrepMeta layer[kMaxPrepLayers];
};

// ---- image layout (bytes) -------------------------------------------------------------------
// "k tile" = one MMA K step of an operand: rows x 32 B, SWIZZLE_32B (umma::sw32_offset), 2 KB for 64 rows.
//   [ones: 128-row k tile, row = (1, 1, 0...)]                                   A operand of the bias MMAs
//   [B1: k tile (W1hi | W1hi | b1hi | b1lo), k tile (W1lo)]                      first layer, bias folded in
//   [hid l: hi 8K | lo 8K] x (L-1)                                               64 x 64, SWIZZLE_128B
//   [bias k tiles: (L-1) hidden, S slots: row n = (b_hi, b_lo, 0...)]            B operand of the bias MMAs
//   [slot s: (hi, lo) k tiles of its slot_nk(D, s) non-zero K steps]             output layer, x log2 e
//   [const tables [6][kCT] fp32]
// Hidden units of class c = 1 + h % (D-1) may feed outputs of order >= c; sorted by class, the first
// cnt_le(o) units are the ones an output of order o reads.
constexpr int kKTile = 2048;
__host__ __device__ constexpr int cnt_le(int D, int o) {   // hidden units with class <= o
  return o >= D - 1 ? kH : o * (kH / (D - 1)) + (o < kH % (D - 1) ? o : kH % (D - 1));
}
__host__ __device__ constexpr int slot_nk(int D, int s) { return (cnt_le(D, s + 1) + 15) / 16; }   // slot s has order s+1
__host__ __device__ constexpr int slot_koff(int D, int s) {
  int k = 0;
  for (int i = 0; i < s; ++i) k += slot_nk(D, i);
  return k;
}
__host__ __device__ constexpr int off_ones() { return 0; }
__host__ __device__ constexpr int off_b1() { return 2 * kKTile; }
__host__ __device__ constexpr int off_hid(int l) { return 4 * kKTile + l * 2 * kTileBytes; }
__host__ __device__ constexpr int off_bias(int L, int i) { return off_hid(L - 1) + i * kKTile; }   // i < L-1: hidden, then slots
__host__ __device__ constexpr int off_slot(int D, int L, int s, int ks, int half) {
  return off_bias(L, (L - 1) + (D - 1)) + ((slot_koff(D, s) + ks) * 2 + half) * kKTile;
}
__host__ __device__ constexpr int off_f32(int D, int L) { return off_slot(D, L, D - 1, 0, 0); }
__host__ __device__ constexpr int image_bytes(int D, int L) { return (off_f32(D, L) + 4 * kConstFloats + 1023) & ~1023; }

__device__ __forceinline__ void store_ktile_row(unsigned char* tile, int row, const __half (&v)[16]) {
  *reinterpret_cast<uint4*>(tile + umma::sw32_offset(row, 0)) = reinterpret_cast<const uint4*>(v)[0];
  *reinterpret_cast<uint4*>(tile + umma::sw32_offset(row, 1)) = reinterpret_cast<const uint4*>(v)[1];
}

// grid (layers, kPrepSlices): the rows of a layer's image are dealt out over kPrepSlices blocks (a single
// block took 28 us per layer, which a training step pays per layer and per step).  The image must have
// been zeroed before the launch (padding rows / columns are exact zeros): the launchers do that with a
// memset node.  params = packed fp32 block of nsf_common.cuh (pre-masked, [in][out])
constexpr int kPrepSlices = 8;
__global__ void __launch_bounds__(256)
nsf_tc_prepare_kernel(const float* __restrict__ params_all, int64_t layer_stride, int D, int L, int nb,
                      const __grid_constant__ PrepArgs args, int layer0, unsigned char* __restrict__ images,
                      int img_bytes) {
  const int layer = layer0 + blockIdx.x;
  const float* par = params_all + (size_t)layer * layer_stride;
  const PrepMeta& pm = args.layer[blockIdx.x];
  const int* perm = args.perm;
  unsigned char* img = images + (size_t)layer * img_bytes;
  const int S = pm.nslots;
  const float* W1t = par;
  const float* b1 = W1t + D * kH;
  const float* hid = b1 + kH;
  const float* Wout = hid + (size_t)(L - 1) * (kH * kH + kH);
  const float* bout = Wout + (size_t)D * kH * kPP;
  float* f32 = reinterpret_cast<float*>(img + off_f32(D, L));
  const __half zero = __float2half_rn(0.f), one = __float2half_rn(1.0f);

  // tasks: 128 ones rows | 64 first-layer rows | (L-1) x 64 x 8 hidden chunks | (L-1+S) x 64 bias rows |
  //        sum_s nk(s) x 64 slot rows
  const int n_ones = 128, n_b1 = kH, n_hid = (L - 1) * kH * 8, n_bias = (L - 1 + S) * kH;
  const int n_slot = slot_koff(D, S) * kH;
  const int ntask = n_ones + n_b1 + n_hid + n_bias + n_slot;
  for (int task = blockIdx.y * blockDim.x + threadIdx.x; task < ntask; task += blockDim.x * gridDim.y) {
    int t2 = task;
    if (t2 < n_ones) {
      __align__(16) __half v[16];
      for (int e = 0; e < 16; ++e) v[e] = e < 2 ? one : zero;
      store_ktile_row(img + off_ones(), t2, v);
      continue;
    }
    t2 -= n_ones;
    if (t2 < n_b1) {
      // first layer, row n: K step 0 = [W1hi (D) | W1hi (D) | b1hi | b1lo | 0], K step 1 = [W1lo (D) | 0]
      const int n = t2, o = perm[n];
      __align__(16) __half k0[16], k1[16];
      for (int e = 0; e < 16; ++e) k0[e] = k1[e] = zero;
      for (int i = 0; i < D; ++i) {
        __half hi, lo;
        umma::split_f16(W1t[i * kH + o], hi, lo);
        k0[i] = hi;
        k0[D + i] = hi;
        k1[i] = lo;
      }
      umma::split_f16(b1[o], k0[2 * D], k0[2 * D + 1]);
      store_ktile_row(img + off_b1(), n, k0);
      store_ktile_row(img + off_b1() + kKTile, n, k1);
      continue;
    }
    t2 -= n_b1;
    if (t2 < n_hid) {
      const int l = t2 / (kH * 8), n = (t2 / 8) % kH, c = t2 % 8;
      const float* wt = hid + (size_t)l * (kH * kH + kH);
      float x[8];
      for (int e = 0; e < 8; ++e) x[e] = wt[perm[c * 8 + e] * kH + perm[n]];
      store_split8(img + off_hid(l), img + off_hid(l) + kTileBytes, n, c, x);
      continue;
    }
    t2 -= n_hid;
    if (t2 < n_bias) {
      const int i = t2 / kH, n = t2 % kH;
      float bv;
      if (i < L - 1) {
        bv = hid[(size_t)i * (kH * kH + kH) + kH * kH + perm[n]];
      } else {
        bv = (n < 3 * nb - 1) ? bout[pm.slot_feature[i - (L - 1)] * kPP + n] * kLog2e : 0.f;
      }
      __align__(16) __half v[16];
      for (int e = 0; e < 16; ++e) v[e] = zero;
      umma::split_f16(bv, v[0], v[1]);
      store_ktile_row(img + off_bias(L, i), n, v);
      continue;
    }
    t2 -= n_bias;
    {
      // slot rows: find (slot, K step) of this row
      const int kk = t2 / kH, q = t2 % kH;
      int sl = 0;
      while (sl + 1 < S && slot_koff(D, sl + 1) <= kk) ++sl;
      const int ks = kk - slot_koff(D, sl);
      const float* wf = Wout + (size_t)pm.slot_feature[sl] * kH * kPP;
      __align__(16) __half hi[16], lo[16];
      for (int e = 0; e < 16; ++e) {
        const float w = (q < 3 * nb - 1) ? wf[perm[16 * ks + e] * kPP + q] * kLog2e : 0.f;
        umma::split_f16(w, hi[e], lo[e]);
      }
      store_ktile_row(img + off_slot(D, L, sl, ks, 0), q, hi);
      store_ktile_row(img + off_slot(D, L, sl, ks, 1), q, lo);
    }
  }
  // constant feature: knots of its bias-only spline, evaluated in double (once per layer and image) and
  // rounded to fp32 at the end; the left knot in x is stored as (hi, lo)
  if (threadIdx.x == 0 && blockIdx.y == gridDim.y - 1) {
    float* ct = f32;
    const float* bf = bout + pm.const_feature * kPP;
    double ew[32], eh[32];
    double sw = 0.0, sh = 0.0;
    for (int j = 0; j < nb; ++j) {
      const double w = bf[j], h = bf[nb + j];
      ew[j] = exp(w / (1.0 + (double)kClipW * fabs(w)));
      eh[j] = exp(h / (1.0 + (double)kClipW * fabs(h)));
      sw += ew[j];
      sh += eh[j];
    }
    double cw = 0.0, ch = 0.0;
    for (int j = 0; j < nb; ++j) {
      const double wj = ew[j] / sw, hj = eh[j] / sh;
      double dl = 1.0, dr = 1.0;
      if (j > 0) {
        const double r = bf[2 * nb + j - 1];
        dl = exp(r / (1.0 + (double)kClipD * fabs(r)));
      }
      if (j < nb - 1) {
        const double r = bf[2 * nb + j];
        dr = exp(r / (1.0 + (double)kClipD * fabs(r)));
      }
      const double x0 = 2.0 * kBound * cw - kBound;
      const float x0f = (float)x0;
      ct[0 * kCT + j] = x0f;                                         // left knot x
      ct[1 * kCT + j] = (float)(2.0 * kBound * wj);                  // bin width
      ct[2 * kCT + j] = (float)(2.0 * kBound * ch - kBound);         // left knot y
      ct[3 * kCT + j] = (float)(2.0 * kBound * hj);                  // bin height
      ct[4 * kCT + j] = (float)dl;
      ct[5 * kCT + j] = (float)dr;
      ct[6 * kCT + j] = (float)(x0 - (double)x0f);
      cw += wj;
      ch += hj;
    }
    for (int j = 0; j < kPP; ++j) ct[kConstRows * kCT + j] = (j < 3 * nb - 1) ? bf[j] * kLog2e : 0.f;   // backward only
  }
}

// =============================================================================================
// device helpers
// =============================================================================================
#ifdef MFB_TC_TRACE
__device__ long long g_trace[4 * 1024];
__device__ __forceinline__ void trace_event(int& pos, int warp, int id) {
  if ((threadIdx.x & 31) == 0 && blockIdx.x == 0 && pos < 1024) {
    g_trace[warp * 1024 + pos] = ((long long)id << 48) | (clock64() & 0xFFFFFFFFFFFFll);
    ++pos;
  }
}
#define TRACE(id) trace_event(trace_pos, (int)(threadIdx.x >> 5), id)
#else
#define TRACE(id)
#endif
__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// relu + (hi, lo) fp16 split of two activations with the ReLU folded into the conversions:
// hi = rz(max(x, 0)) (truncated, so the residual of a positive x is never negative),
// lo = rn(max(x - hi, 0)) (x < 0: hi = 0 and the residual x is clamped to 0).  hi + lo = relu(x) to 2^-22.
__device__ __forceinline__ void split_relu_pair(float x0, float x1, uint32_t& hi, uint32_t& lo) {
#ifdef MFB_TC_RNSPLIT
  x0 = fmaxf(x0, 0.f);
  x1 = fmaxf(x1, 0.f);
  const __half2 h2 = __floats2half2_rn(x0, x1);
  const float2 h2f = __half22float2(h2);
  const __half2 l2 = __floats2half2_rn(x0 - h2f.x, x1 - h2f.y);
  hi = *reinterpret_cast<const uint32_t*>(&h2);
  lo = *reinterpret_cast<const uint32_t*>(&l2);
  return;
#endif
  asm("cvt.rz.relu.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
  const __half2 h = *reinterpret_cast<const __half2*>(&hi);
  const float2 hf = __half22float2(h);
  float r0, r1;
  add2(x0, x1, -hf.x, -hf.y, r0, r1);     // exact residuals, one packed subtraction
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(r1), "f"(r0));
}

// relu(acc) -> (hi, lo) fp16 rows of the A operand tile (row = particle); the bias is already in acc
__device__ __forceinline__ void store_hidden(const float (&acc)[64], unsigned char* a_hi, unsigned char* a_lo, int row) {
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) split_relu_pair(acc[8 * c + 2 * e], acc[8 * c + 2 * e + 1], hi[e], lo[e]);
    const uint32_t off = umma::sw128_offset(row, c);
    *reinterpret_cast<uint4*>(a_hi + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(a_lo + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// Forward variant: the hi half of the A operand lives in TENSOR MEMORY (32 packed columns per warpgroup, written by
// the thread that owns the row with one tcgen05.st), only the lo half goes through shared memory.  Two of the three
// MMAs of a K step then read A from TMEM: per K step the tensor core fetches 10 KB from shared memory instead of 18 KB
// (an N = 64 MMA with both operands in shared memory is bound by that fetch, 48 cycles against the 32 of the math).
#ifndef MFB_TC_TS
#define MFB_TC_TS 1
#endif
// The forward variant converts its accumulator in two pieces of 32 columns (chunks 4 piece .. 4 piece + 3 of the
// row), so that only half of it is live in registers; kTS: the hi half goes to tensor memory (the caller waits for
// the tcgen05.st after the last piece).
template <bool kTS>
__device__ __forceinline__ void store_hidden_piece(const float (&acc)[32], int piece, uint32_t tmem_a_hi,
                                                   unsigned char* a_hi, unsigned char* a_lo, int row) {
#pragma unroll
  for (int c2 = 0; c2 < 2; ++c2) {   // two 16-byte chunks = eight packed columns at a time: few registers in flight
    uint32_t hi[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int cl = 2 * c2 + h, c = 4 * piece + cl;
      uint32_t lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) split_relu_pair(acc[8 * cl + 2 * e], acc[8 * cl + 2 * e + 1], hi[4 * h + e], lo[e]);
      *reinterpret_cast<uint4*>(a_lo + umma::sw128_offset(row, c)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      if constexpr (!kTS)
        *reinterpret_cast<uint4*>(a_hi + umma::sw128_offset(row, c)) = make_uint4(hi[4 * h], hi[4 * h + 1], hi[4 * h + 2], hi[4 * h + 3]);
    }
    if constexpr (kTS) umma::tmem_st8(tmem_a_hi + 8 * (2 * piece + c2), hi);
  }
}

// Backward variant: the rows a warp has just written to the A tile (32 rows x 128 B = 4 KB of the hi plane and 4 KB
// of the lo plane, contiguous: the swizzle only permutes 16-byte chunks inside a row) go to HBM as they are, with two
// bulk copies issued by one lane.  The weight-gradient kernel reads the 32 KB tile back with one bulk copy and uses it
// as an MN-major operand (units contiguous, K = particles): no conversion pass on either side, no store instructions.
__device__ __forceinline__ void mirror_rows(const unsigned char* a_hi, unsigned char* g_img, int warp_in_wg) {
  __syncwarp();
  if ((threadIdx.x & 31) == 0) {
    const uint32_t off = (uint32_t)warp_in_wg * 4096u;
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 4096;" ::"l"(g_img + off), "r"(smem_u32(a_hi + off)) : "memory");
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], 4096;" ::"l"(g_img + kABytes / 2 + off),
                 "r"(smem_u32(a_hi + kABytes / 2 + off))
                 : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  }
}
// ... and before the rows are written again, the copies must have read them
__device__ __forceinline__ void mirror_wait() {
  if ((threadIdx.x & 31) == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  __syncwarp();
}

// output-layer tile of one feature: nk K steps, N = 64
__device__ __forceinline__ void mma_slot(uint32_t tmem_d, uint64_t a_hi, uint64_t a_lo, uint64_t b_hi, uint64_t b_lo,
                                         int nk, uint32_t idesc) {
  for (int ks = 0; ks < nk; ++ks) mma_cross(tmem_d, a_hi, a_lo, b_hi, b_lo, ks, idesc, ks > 0);
  for (int ks = 0; ks < nk; ++ks) mma_main(tmem_d, a_hi, b_hi, ks, idesc);
}

// =============================================================================================
// the layer kernel
// =============================================================================================
// kBwd = false: forward layer (y, log q).  kBwd = true: the first stage of the backward of the same
// layer -- conditioner recomputed, then spline forward + backward per feature: writes the post-ReLU
// activations, dL/dphi, the direct dL/dv and the gradient maxima of BwdIO; y / log q are not written.
#ifndef MFB_TC_PDL
#define MFB_TC_PDL 1
#endif
template <int D, int L, int NB, bool kBwd>
__global__ void __launch_bounds__(kThreads, 1)
nsf_tc_layer_kernel(const float* __restrict__ v, int64_t n, const unsigned char* __restrict__ image,
                    const __grid_constant__ Meta meta,
                    const float* __restrict__ logq_in, int first_layer, float* __restrict__ y,
                    float* __restrict__ logq_out, const __grid_constant__ BwdIO bio) {
  constexpr int S = D - 1;
  constexpr int kImg = image_bytes(D, L);
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // keeps the shared address space
  unsigned char* img = smem;
  unsigned char* a_all = smem + kImg;
  // mbarriers: [0] image; [1 + 2*wg + b] "MMA into TMEM buffer b of wg complete" (count 1, tcgen05.commit);
  // [1 + 2*kWG + 3*wg + r] requests of wg to the issuer (count 4): r = 0 conditioner chain, 1 / 2 = slot
  // buffer 0 / 1 has been read
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_all + kWG * kABytes);
  uint64_t* reqs = bars + 1 + 2 * kWG;
  uint64_t* sbars = reqs + 3 * kWG;            // [wg][2]: particle rows of a tile have landed (TMA, count 1)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sbars + 2 * kWG);
  float* stage_all = reinterpret_cast<float*>(a_all + kWG * kABytes + 256);   // [wg][2][128][D]

  const int tid = threadIdx.x;
  // warp-uniform by construction (shuffle from lane 0): lets the MMA descriptors live in uniform registers
  const int wg = __shfl_sync(0xffffffffu, tid >> 7, 0);   // kWG = the issuer warp
  const int t = tid & 127;
  if (tid == 0) {
    for (int i = 0; i < 1 + 2 * kWG; ++i) mbar_init(&bars[i], 1);
    for (int i = 0; i < 3 * kWG; ++i) mbar_init(&reqs[i], 4);
    for (int i = 0; i < 2 * kWG; ++i) mbar_init(&sbars[i], 1);
    fence_mbar_init();
  }
  if (tid < 32) umma::tmem_alloc(tmem_slot, 512);
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  if (tid == 0) {
    mbar_expect_tx(&bars[0], (uint32_t)kImg);
    tma_load_1d(img, image, (uint32_t)kImg, &bars[0]);
  }
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
#if MFB_TC_PDL
  // Programmatic dependent launch: the layers of a flow are launched back to back, and the next layer's CTA may take
  // this SM as soon as the current layer's CTA has left it -- set-up and the 111 KB operand image (written by the
  // prepare kernel, which never triggers early, so it is complete before any layer kernel starts) are loaded while
  // the slower SMs of the previous layer finish their last tiles.  Everything the previous layer wrote (v, log q) is
  // read only after griddepcontrol.wait.
  asm volatile("griddepcontrol.launch_dependents;");
  asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
  mbar_wait_bounded(&bars[0], 0);

  // TMEM buffers of a warpgroup: slot s lands in buffer s & 1; the hidden chain of the NEXT tile
  // runs in the buffer that frees first (the one of slot S-2) while the last splines are computed.
  constexpr int kHB = (S >= 2) ? ((S - 2) & 1) : 1;
  constexpr int kFork = (S >= 2) ? S - 2 : 0;   // slot after whose TMEM load the next tile starts
  const int64_t ntiles = (n + 127) / 128;
  const int64_t tstride = (int64_t)gridDim.x * kWG;
  const uint32_t idesc64 = umma::make_idesc_f16(128, 64);
  constexpr bool kTS = MFB_TC_TS && !kBwd;   // the backward variant mirrors the whole A tile from shared memory

  if (wg == kWG) {
    // =========================================================================================
    // MMA issuers: warp i of this warpgroup (one thread of it) serves compute warpgroup i.  The
    // requests of a warpgroup come in a fixed order -- per tile: slots 2..S-1 as the TMEM buffers are
    // read, then the conditioner chain of the next tile (first layer, two hidden GEMMs, output slots
    // 0 and 1) -- so the issuer simply polls the next request barrier (test_wait + a short nanosleep,
    // which keeps it off the issue port of the compute warps on its scheduler).
    // =========================================================================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsIssuer));
    const int w = __shfl_sync(0xffffffffu, (tid - kWG * 128) >> 5, 0);
    if (w < kWG) {   // the whole warp walks the schedule; one elected lane issues
      const int64_t first = first_tile_of(w);
      const int cnt = first < ntiles ? (int)((ntiles - first + tstride - 1) / tstride) : 0;
      uint64_t* req_chain = &reqs[3 * w];
      uint64_t* wbar = &bars[1 + 2 * w];
      uint32_t rp = 0, rq0 = 0, rq1 = 0;
      unsigned char* wa_hi = a_all + w * kABytes;
      const uint64_t dA_hi = umma::make_desc_sw128(smem_u32(wa_hi));
      const uint64_t dA_lo = umma::make_desc_sw128(smem_u32(wa_hi + kABytes / 2));
      const uint64_t dOnes = umma::make_desc_sw32(smem_u32(img + off_ones()));
      const uint64_t dB1 = umma::make_desc_sw32(smem_u32(img + off_b1()));
      const uint32_t col0 = tmem_base + (uint32_t)(w * 128);
      const uint32_t tA = tmem_base + (uint32_t)(kWG * 128 + w * 32);   // A hi in tensor memory: K step ks = columns 8 ks ..
      // output-layer tile of slot `slot`: bias (ones x bias tile), then the cross terms of all its
      // non-zero K steps, then the hi*hi terms (see mma_cross)
      auto issue_slot = [&](int slot) {
        const int bsel = slot & 1;
        if (elect_one()) {
          const uint32_t dcol = col0 + bsel * 64;
          int koff = 0;
          for (int i = 0; i < slot; ++i) koff += meta.slot_ksteps[i];
          const uint32_t tiles = smem_u32(img + off_slot(D, L, 0, 0, 0)) + (uint32_t)(koff * 2 * kKTile);
          const int nk = meta.slot_ksteps[slot];
          umma::mma_f16_ss(dcol, dOnes, umma::make_desc_sw32(smem_u32(img + off_bias(L, (L - 1) + slot))), idesc64, 0);
          for (int ks = 0; ks < nk; ++ks) {
            const uint64_t dBh = umma::make_desc_sw32(tiles + (uint32_t)(ks * 2 * kKTile));
            const uint64_t dBl = umma::make_desc_sw32(tiles + (uint32_t)(ks * 2 * kKTile + kKTile));
            if constexpr (kTS) umma::mma_f16_ts(dcol, tA + 8 * ks, dBl, idesc64, 1);
            else umma::mma_f16_ss(dcol, umma::desc_advance_k(dA_hi, ks), dBl, idesc64, 1);
            umma::mma_f16_ss(dcol, umma::desc_advance_k(dA_lo, ks), dBh, idesc64, 1);
          }
          for (int ks = 0; ks < nk; ++ks) {
            const uint64_t dBh = umma::make_desc_sw32(tiles + (uint32_t)(ks * 2 * kKTile));
            if constexpr (kTS) umma::mma_f16_ts(dcol, tA + 8 * ks, dBh, idesc64, 1);
            else umma::mma_f16_ss(dcol, umma::desc_advance_k(dA_hi, ks), dBh, idesc64, 1);
          }
          umma::commit(wbar + bsel);
        }
        __syncwarp();
      };
      auto chain = [&]() {
        // first masked layer (K = 16, bias folded into the weights' spare K columns)
        mbar_wait_polite(req_chain, rp);
        rp ^= 1;
        umma::fence_after_sync();
        if (elect_one()) {
          umma::mma_f16_ss(col0 + kHB * 64, dA_hi, dB1, idesc64, 0);
          umma::mma_f16_ss(col0 + kHB * 64, dA_hi, dB1 + (uint64_t)(kKTile >> 4), idesc64, 1);
          umma::commit(wbar + kHB);
        }
        __syncwarp();
        // hidden -> hidden
#pragma unroll 1
        for (int l = 0; l < L - 1; ++l) {
          mbar_wait_polite(req_chain, rp);
          rp ^= 1;
          umma::fence_after_sync();
          const uint64_t dBh = umma::make_desc_sw128(smem_u32(img + off_hid(0) + l * 2 * kTileBytes));
          const uint64_t dBl = umma::make_desc_sw128(smem_u32(img + off_hid(0) + l * 2 * kTileBytes + kTileBytes));
          if (elect_one()) {
          umma::mma_f16_ss(col0 + kHB * 64, dOnes, umma::make_desc_sw32(smem_u32(img + off_bias(L, 0) + l * kKTile)),
                           idesc64, 0);
#pragma unroll
          for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              // outputs below hid_n0[ks] have all-zero weights for this K step: skip those rows
              const int n0 = meta.hid_n0[ks];
              const uint32_t idesc = umma::make_idesc_f16(128, 64 - n0);
              const uint64_t boff = (uint64_t)((n0 * 128) >> 4);
              if constexpr (kTS) {
                const uint32_t dd = col0 + kHB * 64 + n0;
                if (pass == 0) {
                  umma::mma_f16_ts(dd, tA + 8 * ks, umma::desc_advance_k(dBl + boff, ks), idesc, 1);
                  umma::mma_f16_ss(dd, umma::desc_advance_k(dA_lo, ks), umma::desc_advance_k(dBh + boff, ks), idesc, 1);
                } else {
                  umma::mma_f16_ts(dd, tA + 8 * ks, umma::desc_advance_k(dBh + boff, ks), idesc, 1);
                }
              } else if (pass == 0)
                mma_cross(col0 + kHB * 64 + n0, dA_hi, dA_lo, dBh + boff, dBl + boff, ks, idesc, 1);
              else
                mma_main(col0 + kHB * 64 + n0, dA_hi, dBh + boff, ks, idesc);
            }
          }
          umma::commit(wbar + kHB);
          }
          __syncwarp();
        }
        // output layer: slots 0 and 1 into the two TMEM buffers
        mbar_wait_polite(req_chain, rp);
        rp ^= 1;
        umma::fence_after_sync();
        issue_slot(0);
        if (S > 1) issue_slot(1);
      };
      if (cnt > 0) chain();
#pragma unroll 1
      for (int i = 0; i < cnt; ++i) {
#pragma unroll 1
        for (int sq = 0; sq + 2 < S; ++sq) {
          if ((sq & 1) == 0) {
            mbar_wait_polite(req_chain + 1, rq0);
            rq0 ^= 1;
          } else {
            mbar_wait_polite(req_chain + 2, rq1);
            rq1 ^= 1;
          }
          umma::fence_after_sync();
          issue_slot(sq + 2);
        }
        if (i + 1 < cnt) chain();
      }
    }
    __syncwarp();
  } else {
  // ===========================================================================================
  // compute warpgroups
  // ===========================================================================================
  asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsCompute));
  unsigned char* a_hi = a_all + wg * kABytes;
  unsigned char* a_lo = a_hi + kABytes / 2;
  uint64_t* bar0 = &bars[1 + 2 * wg];
  uint64_t* bar1 = bar0 + 1;
  uint64_t* req_chain = &reqs[3 * wg];
  uint32_t ph0 = 0, ph1 = 0;
  const uint32_t lane_sel = (uint32_t)((t >> 5) * 32) << 16;
  const uint32_t col0 = tmem_base + (uint32_t)(wg * 128);
  const uint32_t ta_hi = tmem_base + (uint32_t)(kWG * 128 + wg * 32);   // this warpgroup's A hi columns (forward variant)
  const float* ctab = reinterpret_cast<const float*>(img + off_f32(D, L));

#ifdef MFB_TC_TRACE
  int trace_pos = 0;
#endif
  auto wait_buf = [&](int bsel) {
    TRACE(1);
    if (bsel == 0) {
      mbar_wait_bounded(bar0, ph0);
      ph0 ^= 1;
    } else {
      mbar_wait_bounded(bar1, ph1);
      ph1 ^= 1;
    }
    umma::fence_after_sync();
    TRACE(2);
  };
  // first masked layer of a tile: A row = [v_hi (D) | v_lo (D) | 1 | 1 | 0 ...] (K = 16)
  auto start_tile = [&](const float* vv, uint64_t* landed, uint32_t parity) {
    mbar_wait_bounded(landed, parity);   // the TMA copy of this tile's particle rows has landed
    if constexpr (kBwd) mirror_wait();   // the copy of the previous chain's last activations has read the A rows
    __align__(16) __half row[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) row[e] = __float2half_rn(0.f);
#pragma unroll
    for (int i = 0; i < D; ++i) umma::split_f16(vv[i], row[i], row[D + i]);
    row[2 * D] = __float2half_rn(1.0f);
    row[2 * D + 1] = __float2half_rn(1.0f);
    *reinterpret_cast<uint4*>(a_hi + umma::sw128_offset(t, 0)) = reinterpret_cast<const uint4*>(row)[0];
    *reinterpret_cast<uint4*>(a_hi + umma::sw128_offset(t, 1)) = reinterpret_cast<const uint4*>(row)[1];
    fence_proxy_async();
    request_arrive(req_chain);
    TRACE(3);
  };
  int64_t next_p = 0;        // particle of this thread in the tile whose chain is running (backward variant)
  bool next_valid = false;
  // hidden step l (0..L-1): accumulator -> relu -> (hi, lo) rows of A, then ask for the next masked
  // GEMM (l < L-1) or the first two output-layer tiles (l == L-1)
  auto hidden_step = [&](int l) {
    wait_buf(kHB);
    // biases are already in the accumulator (bias MMA)
    float acc[kBwd ? 64 : 1];
    if constexpr (kBwd) {
      tmem_ld64(col0 + (uint32_t)(kHB * 64) + lane_sel, acc);
      mirror_wait();
      store_hidden(acc, a_hi, a_lo, t);
    } else {
#pragma unroll
      for (int piece = 0; piece < 2; ++piece) {
        float part[32];
        tmem_ld_cols(col0 + (uint32_t)(kHB * 64 + 32 * piece) + lane_sel, part);
        store_hidden_piece<kTS>(part, piece, ta_hi + lane_sel, a_hi, a_lo, t);
      }
      if constexpr (kTS) umma::tmem_wait_st();
    }
    fence_proxy_async();
    umma::fence_before_sync();
    request_arrive(req_chain);
    if constexpr (kBwd) {
      // post-ReLU activations of the tile being started (= next tile) for the weight gradients: the operand tile
      // itself, columns in the SORTED unit order of the operand images (column c = unit meta.perm[c]; the
      // weight-gradient reduce maps back).  Rows beyond n hold the activations of zero input (prefetch below).
      mirror_rows(a_hi, reinterpret_cast<unsigned char*>(bio.acts) + ((size_t)(next_p >> 7) * L + l) * kABytes, t >> 5);
      // ReLU masks for the data-gradient chain: bit c of word w = unit at sorted position 32 w + c is active
      if (next_valid) {
        uint32_t m0 = 0, m1 = 0;
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          if (c < 32) m0 |= (acc[c] > 0.f ? 1u : 0u) << c;
          else m1 |= (acc[c] > 0.f ? 1u : 0u) << (c - 32);
        }
        uint32_t* mk = bio.masks + ((size_t)(next_p >> 7) * (L * 2) + l * 2) * 128 + t;
        mk[0] = m0;
        mk[128] = m1;
      }
    }
    TRACE(4 + l);
  };

  // Particles are staged through shared memory ([128][D] per tile, two buffers per warpgroup): the
  // rows of the NEXT tile come in with one TMA bulk copy issued a few splines ahead (no registers
  // held, no exposed global-load latency), each spline reads its v_f from the thread's row and writes
  // y_f back in place, and the finished row goes out from there.
  float* stage0 = stage_all + ((size_t)(wg * 2) * 128 + t) * D;
  float* stage1 = stage0 + 128 * D;
  uint64_t* sbar = sbars + 2 * wg;
  auto prefetch = [&](int64_t tl, int buf) {   // one thread of the warpgroup
    if (tl >= ntiles) return;
    int64_t rows = n - tl * 128;
    if (rows > 128) rows = 128;
    float* dst = stage_all + (size_t)(wg * 2 + buf) * 128 * D;
    const float* src = v + tl * 128 * D;
    const uint32_t bytes = (uint32_t)(rows * D * 4), bulk = bytes & ~15u;
    for (uint32_t i = bulk / 4; i < bytes / 4; ++i) dst[i] = src[i];   // ragged tail (< 16 B)
    for (uint32_t i = bytes / 4; i < 128u * D; ++i) dst[i] = 0.f;      // rows beyond n: defined (finite) input
    mbar_expect_tx(&sbar[buf], bulk);
    if (bulk) tma_load_1d(dst, src, bulk, &sbar[buf]);
  };

  int64_t tile = first_tile_of(wg);
  // Software-pipelined over the tiles of this warpgroup: iteration i computes the splines of tile i
  // ("cur") and, interleaved with its last splines, the conditioner chain of tile i+1 ("next"), so
  // every MMA has a spline's worth of CUDA-core work to hide behind.  The first iteration has no
  // current tile (cur = false): it only runs the chain of the first tile, through the same code.
  bool cur = false;
  bool has_next = tile < ntiles;   // uniform over the warpgroup
  float* sc = stage0;              // this thread's row of the current tile
  float* sn = stage1;              // ... of the next tile
  int nbuf = 1;                    // staging buffer of the next tile
  uint32_t sph0 = 0, sph1 = 0;     // phases of the two "landed" barriers
  float jac_carry = 1.0f, ss_carry = 0.f;
  if (t == 0) prefetch(tile, nbuf);
  tile -= tstride;
  while (cur || has_next) {
    const int64_t p = tile * 128 + t;
    const bool valid = cur && p < n;
    if (cur) has_next = tile + tstride < ntiles;
    next_p = (tile + tstride) * 128 + t;
    next_valid = has_next && next_p < n;
    float jac = jac_carry;   // Jacobian of the bias-only feature, computed at the end of the previous iteration
    float ss = ss_carry;     // |v|^2 for the base density of the first layer
    float lq_in = 0.f;       // loaded a tile's worth of work before it is needed
    if (!kBwd && cur && valid && logq_out && !first_layer) lq_in = logq_in[p];
    // backward variant: upstream gradients of this particle, running maximum of |dL/dphi|
    float gyr[D] = {}, glq = 0.f, amax = 0.f;
    if constexpr (kBwd) {
#pragma unroll
      for (int i = 0; i < D; ++i) gyr[i] = valid ? bio.gy[p * D + i] : 0.f;
      glq = (valid && bio.glogq) ? bio.glogq[p] : 0.f;
    }
    // one feature of the backward variant: spline forward + backward from the raw parameters in acc,
    // dL/dphi rows out, direct dL/dv into the staging row in place of v_f
    auto feature_bwd = [&](float (&acc)[64], int f) {
      const float vf = sc[f];
      float gyf = gyr[0];
#pragma unroll
      for (int i = 1; i < D; ++i) gyf = (f == i) ? gyr[i] : gyf;
      // logq_out = logq_in - ladj  =>  dL/d(ladj) = -dL/dlogq
      KnotGrad kg;
      float gvf = rq_spline_regs_bwd<NB>(acc, vf, gyf, -glq, &kg);
      if (first_layer) gvf -= glq * vf;   // d/dv of log N(v; 0, I)
      sc[f] = gvf;
      if (valid) {
        float* gp = bio.gphi + ((size_t)tile * (D * kGRows) + f * kGRows) * 128 + t;
#pragma unroll
        for (int j = 0; j < 2 * NB; ++j) {
          gp[j * 128] = acc[j];
          amax = fmaxf(amax, fabsf(acc[j]));
        }
        gp[(2 * NB) * 128] = kg.left;
        gp[(2 * NB + 1) * 128] = kg.right;
        gp[(2 * NB + 2) * 128] = (float)kg.bin;
        amax = fmaxf(amax, fmaxf(fabsf(kg.left), fabsf(kg.right)));
      }
    };
    // backward variant: the bias-only feature is iteration s = -1 of the same loop (its raw parameters
    // come from the constant table instead of TMEM), so the spline code exists once -- the kernel is
    // large enough for instruction-cache misses to show up as a stall reason
#pragma unroll 1
    for (int s = kBwd ? -1 : 0; s < S; ++s) {
      const int b = s & 1;
      // after slot kFork's accumulator has been read: the chain of the next tile may start (it runs in that buffer)
      auto fork = [&]() {
        if (cur && S >= 2) wait_buf((S - 1) & 1);   // every output-layer MMA of this tile is done: A is free
        if (has_next) {
          if (nbuf == 0) {
            start_tile(sn, &sbar[0], sph0);
            sph0 ^= 1;
          } else {
            start_tile(sn, &sbar[1], sph1);
            sph1 ^= 1;
          }
        }
      };
      // the last slot was already waited for at kFork; slot 0 is complete => every warp is past its last read of
      // the other staging buffer
      auto slot_ready = [&]() {
        if (!(S >= 2 && s == S - 1)) wait_buf(b);
        if (s == 0 && t == 0 && has_next) prefetch(tile + tstride, nbuf);
      };
      if constexpr (kBwd) {
        float acc[64];
        if (s < 0) {
          if (cur) {
            const float4* cb = reinterpret_cast<const float4*>(ctab + kConstRows * kCT);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float4 q4 = cb[i];
              acc[4 * i] = q4.x; acc[4 * i + 1] = q4.y; acc[4 * i + 2] = q4.z; acc[4 * i + 3] = q4.w;
            }
          }
        } else if (cur) {
          slot_ready();
          tmem_ld64(col0 + (uint32_t)(b * 64) + lane_sel, acc);
          umma::fence_before_sync();
          if (s + 2 < S) request_arrive(req_chain + 1 + b);
          TRACE(10 + s);
        }
        if (s == kFork) fork();
        if (cur) {
          feature_bwd(acc, s < 0 ? meta.const_feature : meta.slot_feature[s < 0 ? 0 : s]);
          TRACE(20 + s);
        }
      } else if (cur) {
        // the spline reads the accumulator in two pieces; after the second the buffer is released
        slot_ready();
        const int f = meta.slot_feature[s];
        const float vf = sc[f];
        ss = fmaf(vf, vf, ss);
        sc[f] = rq_spline_regs_ld<NB>(
            [&](int col, auto& dst) {
              tmem_ld_cols(col0 + (uint32_t)(b * 64 + col) + lane_sel, dst);
              if (col == 0) return;
              umma::fence_before_sync();
              if (s + 2 < S) request_arrive(req_chain + 1 + b);
              TRACE(10 + s);
              if (s == kFork) fork();
            },
            vf, jac);
        TRACE(20 + s);
      } else if (s == kFork) {
        fork();
      }
      if (has_next) {
        if (s == kFork) hidden_step(0);
        if (S >= 2 && s == S - 1) hidden_step(1);
      }
    }
    if (S == 1 && has_next) hidden_step(1);
    if constexpr (kBwd) {
      if (valid) {
#pragma unroll
        for (int i = 0; i < D; ++i) bio.gvd[p * D + i] = sc[i];
        bio.gmax[p] = amax;
      }
      if (cur) {   // batch maximum of |dL/dphi|: one atomic per warp (non-negative floats order like ints)
        float wm = valid ? amax : 0.f;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) wm = fmaxf(wm, __shfl_xor_sync(0xffffffffu, wm, o));
        if ((t & 31) == 0) atomicMax(bio.gmaxes, __float_as_int(wm));
      }
      if (has_next) hidden_step(2);
    } else {
      if (valid) {
#pragma unroll
        for (int i = 0; i < D; ++i) y[p * D + i] = sc[i];
        if (logq_out) {
          const float base = first_layer ? -0.5f * ss - (float)D * kHalfLog2Pi : lq_in;
          logq_out[p] = fmaf(-0.69314718055994531f, fast_lg2(jac), base);
        }
      }
      if (has_next) {
        // bias-only feature of the NEXT tile here: CUDA-core work between the request for the third
        // GEMM of its chain and the wait for it
        const float vf = sn[meta.const_feature];
        ss_carry = vf * vf;
        jac_carry = 1.0f;
        sn[meta.const_feature] = rq_spline_const<NB>(ctab, vf, jac_carry);
        hidden_step(2);
      }
    }
    float* tmp = sc;
    sc = sn;
    sn = tmp;
    nbuf ^= 1;
    cur = has_next;
    has_next = false;   // recomputed at the top of the next iteration
    tile += tstride;
  }
    if constexpr (kBwd) {   // the last activation tiles are in HBM before the CTA gives up its shared memory
      if ((threadIdx.x & 31) == 0) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
      __syncwarp();
    }
  }  // compute warpgroups
  umma::fence_before_sync();
  __syncthreads();
  if (tid < 32) umma::tmem_dealloc(tmem_base, 512);
}

// =============================================================================================
// Density direction on the same machinery: v = A^-1(y), one layer per launch (generate/flows/zuko.py:21-22,31-32,
// 43-50: log_prob / inverse / inverse_steps).  The autoregressive inverse is sequential in the features: the feature
// that is first in the layer's order inverts its bias-only spline, then every further feature needs the conditioner
// of the values found so far -- first layer, two hidden GEMMs, ONE output-feature tile -- followed by the inverse
// spline in registers (rq_spline_regs_inv).  Per 128-particle tile a warpgroup therefore makes S x 4 round trips to
// the tensor core; the three warpgroups of a CTA run their tiles independently, so the issuer warps interleave them.
// Same operand image, TMEM layout and hand-off as the forward kernel; one accumulator buffer, nothing pipelined inside
// a tile (each step depends on the one before).  Replaces D full sweeps of the CUDA-core kernel (nsf_inv.cu).
// =============================================================================================
template <int D, int L, int NB>
__global__ void __launch_bounds__(kThreads, 1)
nsf_tc_inverse_kernel(const float* __restrict__ y, int64_t n, const unsigned char* __restrict__ image,
                      const __grid_constant__ Meta meta, const float* __restrict__ ladj_in, int last_layer,
                      float* __restrict__ v_out, float* __restrict__ ladj_out) {
  static_assert(L == 3, "compiled for three hidden layers");
  constexpr int S = D - 1;
  constexpr int kImg = image_bytes(D, L);
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  unsigned char* img = smem;
  unsigned char* a_all = smem + kImg;
  uint64_t* bars = reinterpret_cast<uint64_t*>(a_all + kWG * kABytes);   // [0] image, [1 + wg] MMA done, [1 + kWG + wg] request
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 1 + 2 * kWG);

  const int tid = threadIdx.x;
  const int wg = __shfl_sync(0xffffffffu, tid >> 7, 0);
  const int t = tid & 127;
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    for (int i = 0; i < kWG; ++i) {
      mbar_init(&bars[1 + i], 1);
      mbar_init(&bars[1 + kWG + i], 4);
    }
    fence_mbar_init();
  }
  if (tid < 32) umma::tmem_alloc(tmem_slot, 256);
  umma::fence_before_sync();
  __syncthreads();
  umma::fence_after_sync();
  if (tid == 0) {
    mbar_expect_tx(&bars[0], (uint32_t)kImg);
    tma_load_1d(img, image, (uint32_t)kImg, &bars[0]);
  }
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);
  mbar_wait_bounded(&bars[0], 0);

  const int64_t ntiles = (n + 127) / 128;
  const int64_t tstride = (int64_t)gridDim.x * kWG;
  const uint32_t idesc64 = umma::make_idesc_f16(128, 64);

  if (wg == kWG) {
    // ===== issuers: warp i serves warpgroup i; per tile and slot: first layer, two hidden GEMMs, the slot's tile =====
    asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kRegsIssuer));
    const int w = __shfl_sync(0xffffffffu, (tid - kWG * 128) >> 5, 0);
    if (w < kWG) {
      uint64_t* done = &bars[1 + w];
      uint64_t* req = &bars[1 + kWG + w];
      uint32_t rp = 0;
      unsigned char* wa_hi = a_all + w * kABytes;
      const uint64_t dA_hi = umma::make_desc_sw128(smem_u32(wa_hi));
      const uint64_t dA_lo = umma::make_desc_sw128(smem_u32(wa_hi + kABytes / 2));
      const uint64_t dOnes = umma::make_desc_sw32(smem_u32(img + off_ones()));
      const uint64_t dB1 = umma::make_desc_sw32(smem_u32(img + off_b1()));
      const uint32_t dcol = tmem_base + (uint32_t)(w * 64);
      auto wait_req = [&]() {
        mbar_wait_polite(req, rp);
        rp ^= 1;
        umma::fence_after_sync();
      };
      for (int64_t tile = first_tile_of(w); tile < ntiles; tile += tstride) {
#pragma unroll 1
        for (int slot = 0; slot < S; ++slot) {
          // first masked layer (K = 16, bias folded into the weights' spare K columns)
          wait_req();
          if (elect_one()) {
            umma::mma_f16_ss(dcol, dA_hi, dB1, idesc64, 0);
            umma::mma_f16_ss(dcol, dA_hi, dB1 + (uint64_t)(kKTile >> 4), idesc64, 1);
            umma::commit(done);
          }
          __syncwarp();
          // hidden -> hidden
#pragma unroll 1
          for (int l = 0; l < L - 1; ++l) {
            wait_req();
            const uint64_t dBh = umma::make_desc_sw128(smem_u32(img + off_hid(0) + l * 2 * kTileBytes));
            const uint64_t dBl = umma::make_desc_sw128(smem_u32(img + off_hid(0) + l * 2 * kTileBytes + kTileBytes));
            if (elect_one()) {
              umma::mma_f16_ss(dcol, dOnes, umma::make_desc_sw32(smem_u32(img + off_bias(L, 0) + l * kKTile)), idesc64, 0);
#pragma unroll
              for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                  const int n0 = meta.hid_n0[ks];
                  const uint32_t idesc = umma::make_idesc_f16(128, 64 - n0);
                  const uint64_t boff = (uint64_t)((n0 * 128) >> 4);
                  if (pass == 0) mma_cross(dcol + n0, dA_hi, dA_lo, dBh + boff, dBl + boff, ks, idesc, 1);
                  else mma_main(dcol + n0, dA_hi, dBh + boff, ks, idesc);
                }
              }
              umma::commit(done);
            }
            __syncwarp();
          }
          // the output-feature tile of this slot
          wait_req();
          if (elect_one()) {
            int koff = 0;
            for (int i = 0; i < slot; ++i) koff += meta.slot_ksteps[i];
            const uint32_t tiles = smem_u32(img + off_slot(D, L, 0, 0, 0)) + (uint32_t)(koff * 2 * kKTile);
            const int nk = meta.slot_ksteps[slot];
            umma::mma_f16_ss(dcol, dOnes, umma::make_desc_sw32(smem_u32(img + off_bias(L, (L - 1) + slot))), idesc64, 0);
            for (int ks = 0; ks < nk; ++ks) {
              const uint64_t dBh = umma::make_desc_sw32(tiles + (uint32_t)(ks * 2 * kKTile));
              const uint64_t dBl = umma::make_desc_sw32(tiles + (uint32_t)(ks * 2 * kKTile + kKTile));
              umma::mma_f16_ss(dcol, umma::desc_advance_k(dA_hi, ks), dBl, idesc64, 1);
              umma::mma_f16_ss(dcol, umma::desc_advance_k(dA_lo, ks), dBh, idesc64, 1);
            }
            for (int ks = 0; ks < nk; ++ks)
              umma::mma_f16_ss(dcol, umma::desc_advance_k(dA_hi, ks), umma::make_desc_sw32(tiles + (uint32_t)(ks * 2 * kKTile)),
                               idesc64, 1);
            umma::commit(done);
          }
          __syncwarp();
        }
      }
    }
    __syncwarp();
  } else {
    // ===== compute warpgroups: thread = particle row =====
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kRegsCompute));
    unsigned char* a_hi = a_all + wg * kABytes;
    unsigned char* a_lo = a_hi + kABytes / 2;
    uint64_t* done = &bars[1 + wg];
    uint64_t* req = &bars[1 + kWG + wg];
    uint32_t ph = 0;
    const uint32_t taddr = tmem_base + (uint32_t)(wg * 64) + ((uint32_t)((t >> 5) * 32) << 16);
    const float* ctab = reinterpret_cast<const float*>(img + off_f32(D, L));
    auto hand_off = [&]() {
      fence_proxy_async();
      umma::fence_before_sync();
      request_arrive(req);
    };
    auto wait_done = [&]() {
      mbar_wait_bounded(done, ph);
      ph ^= 1;
      umma::fence_after_sync();
    };
    for (int64_t tile = first_tile_of(wg); tile < ntiles; tile += tstride) {
      const int64_t p = tile * 128 + t;
      const bool valid = p < n;
      float yy[D], vv[D];
#pragma unroll
      for (int i = 0; i < D; ++i) {
        yy[i] = valid ? y[p * D + i] : 0.f;
        vv[i] = yy[i];        // features not found yet: any finite value (their weights are masked)
      }
      const float la_in = (valid && ladj_in) ? ladj_in[p] : 0.f;
      float jac = 1.0f;
      {
        float yc = yy[0];
#pragma unroll
        for (int i = 1; i < D; ++i) yc = (meta.const_feature == i) ? yy[i] : yc;
        const float vc = rq_spline_const_inv<NB>(ctab, yc, jac);
#pragma unroll
        for (int i = 0; i < D; ++i) vv[i] = (meta.const_feature == i) ? vc : vv[i];
      }
#pragma unroll 1
      for (int slot = 0; slot < S; ++slot) {
        const int f = meta.slot_feature[slot];
        {   // first layer: A row = [v_hi (D) | v_lo (D) | 1 | 1 | 0 ...]
          __align__(16) __half row[16];
#pragma unroll
          for (int e = 0; e < 16; ++e) row[e] = __float2half_rn(0.f);
#pragma unroll
          for (int i = 0; i < D; ++i) umma::split_f16(vv[i], row[i], row[D + i]);
          row[2 * D] = __float2half_rn(1.0f);
          row[2 * D + 1] = __float2half_rn(1.0f);
          *reinterpret_cast<uint4*>(a_hi + umma::sw128_offset(t, 0)) = reinterpret_cast<const uint4*>(row)[0];
          *reinterpret_cast<uint4*>(a_hi + umma::sw128_offset(t, 1)) = reinterpret_cast<const uint4*>(row)[1];
          hand_off();
        }
        float acc[64];
#pragma unroll 1
        for (int l = 0; l < L; ++l) {
          wait_done();
          tmem_ld64(taddr, acc);
          store_hidden(acc, a_hi, a_lo, t);
          hand_off();
        }
        wait_done();
        tmem_ld64(taddr, acc);
        umma::fence_before_sync();
        float yf = yy[0];
#pragma unroll
        for (int i = 1; i < D; ++i) yf = (f == i) ? yy[i] : yf;
        const float vf = rq_spline_regs_inv<NB>(acc, yf, jac);
#pragma unroll
        for (int i = 0; i < D; ++i) vv[i] = (f == i) ? vf : vv[i];
      }
      if (valid) {
#pragma unroll
        for (int i = 0; i < D; ++i) v_out[p * D + i] = vv[i];
        if (ladj_out) {
          float tot = fmaf(0.69314718055994531f, fast_lg2(jac), la_in);
          if (last_layer) {   // log q(x) = log N(z; 0, I) - sum of the forward log-Jacobians
            float ss = 0.f;
#pragma unroll
            for (int i = 0; i < D; ++i) ss = fmaf(vv[i], vv[i], ss);
            tot = -0.5f * ss - (float)D * kHalfLog2Pi - tot;
          }
          ladj_out[p] = tot;
        }
      }
    }
  }
  umma::fence_before_sync();
  __syncthreads();
  if (tid < 32) umma::tmem_dealloc(tmem_base, 256);
}

// ---- host side ----------------------------------------------------------------------------
static void make_meta(int d, const int32_t* order, Meta* m, PrepMeta* pm) {
  int cls[kH], perm[kH];
  hidden_classes(d, cls, perm);
  int cnt_le[kMaxDim + 2] = {0};  // cnt_le[c] = #hidden units with class <= c
  for (int c = 1; c <= d; ++c) {
    cnt_le[c] = cnt_le[c - 1];
    for (int h = 0; h < kH; ++h) cnt_le[c] += (cls[h] == c);
  }
  int slots = 0, cfeat = 0;
  int feat_of_order[kMaxDim];
  for (int i = 0; i < d; ++i) feat_of_order[order[i]] = i;
  cfeat = feat_of_order[0];
  Meta mm = {};
  PrepMeta pp = {};
  for (int o = 1; o < d; ++o) {
    const int f = feat_of_order[o];
    mm.slot_feature[slots] = f;
    mm.slot_ksteps[slots] = slot_nk(d, slots);
    pp.slot_feature[slots] = f;
    ++slots;
  }
  for (int ks = 0; ks < 4; ++ks) {
    const int cmin = cls[perm[16 * ks]];   // smallest class among the inputs of this K step
    const int first = cnt_le[cmin - 1];    // outputs with class >= cmin start here (sorted order)
    mm.hid_n0[ks] = (first / 16) * 16;
  }
  mm.const_feature = cfeat;
  mm.nslots = slots;
  for (int h = 0; h < kH; ++h) mm.perm[h] = perm[h];
  pp.const_feature = cfeat;
  pp.nslots = slots;
  if (m) *m = mm;
  if (pm) *pm = pp;
}

static bool valid_order(int d, const int32_t* order) {
  int seen = 0;
  for (int i = 0; i < d; ++i) {
    if (order[i] < 0 || order[i] >= d) return false;
    seen |= 1 << order[i];
  }
  return seen == (1 << d) - 1;
}

template <int D>
static int launch_layer(const float* v, int64_t n, const unsigned char* image, const Meta& meta, const float* logq_in,
                        int first, float* y, float* logq_out, cudaStream_t st) {
  constexpr int L = 3, NB = 20;
  const size_t smem = (size_t)image_bytes(D, L) + kWG * kABytes + 256 + (size_t)kWG * 2 * 128 * D * 4 + 1024;
  auto kern = nsf_tc_layer_kernel<D, L, NB, false>;
  MFB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (n + 127) / 128;
  int64_t grid = sm_count();
  if (grid * kWG > ntiles) grid = (ntiles + kWG - 1) / kWG;
#if MFB_TC_PDL
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  MFB_CUDA(cudaLaunchKernelEx(&cfg, kern, v, n, image, meta, logq_in, first, y, logq_out, BwdIO{}));
#else
  kern<<<(int)grid, kThreads, smem, st>>>(v, n, image, meta, logq_in, first, y, logq_out, BwdIO{});
#endif
  return launch_status();
}

template <int D>
static int launch_layer_bwd(const float* v, int64_t n, const unsigned char* image, const Meta& meta, int first,
                            const BwdIO& bio, cudaStream_t st) {
  constexpr int L = 3, NB = 20;
  const size_t smem = (size_t)image_bytes(D, L) + kWG * kABytes + 256 + (size_t)kWG * 2 * 128 * D * 4 + 1024;
  auto kern = nsf_tc_layer_kernel<D, L, NB, true>;
  MFB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (n + 127) / 128;
  int64_t grid = sm_count();
  if (grid * kWG > ntiles) grid = (ntiles + kWG - 1) / kWG;
  kern<<<(int)grid, kThreads, smem, st>>>(v, n, image, meta, nullptr, first, nullptr, nullptr, bio);
  return launch_status();
}

template <int D>
static int launch_inverse(const float* y, int64_t n, const unsigned char* image, const Meta& meta, const float* ladj_in,
                          int last, float* v, float* ladj_out, cudaStream_t st) {
  constexpr int L = 3, NB = 20;
  const size_t smem = (size_t)image_bytes(D, L) + kWG * kABytes + 256 + 1024;
  auto kern = nsf_tc_inverse_kernel<D, L, NB>;
  MFB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int64_t ntiles = (n + 127) / 128;
  int64_t grid = sm_count();
  if (grid * kWG > ntiles) grid = (ntiles + kWG - 1) / kWG;
  kern<<<(int)grid, kThreads, smem, st>>>(y, n, image, meta, ladj_in, last, v, ladj_out);
  return launch_status();
}

}  // namespace tc

int nsf_tc_check(int d, int hidden_layers, int bins, const void* image, const int32_t* order, const void* rows) {
  if (!(d >= 2 && d <= 6 && hidden_layers == 3 && bins == 20)) return MFB_E_UNSUPPORTED;
  if (!tc::valid_order(d, order)) return MFB_E_BADARG;
  if ((reinterpret_cast<uintptr_t>(image) & 15u) != 0) return MFB_E_BADARG;   // loaded with a bulk copy
  if ((reinterpret_cast<uintptr_t>(rows) & 15u) != 0) return MFB_E_BADARG;    // tiles of rows: bulk copies too
  return 0;
}

int nsf_tc_fwd(const float* v, int64_t n, int d, int hidden_layers, int bins, const void* image,
               const int32_t* order, const float* logq_in, int first_layer, float* y, float* logq_out,
               cudaStream_t st) {
  const int rc = nsf_tc_check(d, hidden_layers, bins, image, order, v);
  if (rc || n == 0) return rc;
  tc::Meta meta;
  tc::make_meta(d, order, &meta, nullptr);
  const unsigned char* img = reinterpret_cast<const unsigned char*>(image);
  switch (d) {
    case 2: return tc::launch_layer<2>(v, n, img, meta, logq_in, first_layer, y, logq_out, st);
    case 3: return tc::launch_layer<3>(v, n, img, meta, logq_in, first_layer, y, logq_out, st);
    case 4: return tc::launch_layer<4>(v, n, img, meta, logq_in, first_layer, y, logq_out, st);
    case 5: return tc::launch_layer<5>(v, n, img, meta, logq_in, first_layer, y, logq_out, st);
    case 6: return tc::launch_layer<6>(v, n, img, meta, logq_in, first_layer, y, logq_out, st);
    default: return MFB_E_UNSUPPORTED;
  }
}

int nsf_tc_inv(const float* y, int64_t n, int d, int hidden_layers, int bins, const void* image,
               const int32_t* order, const float* ladj_in, int last_layer, float* v, float* ladj_out,
               cudaStream_t st) {
  const int rc = nsf_tc_check(d, hidden_layers, bins, image, order, nullptr);   // y is read row by row
  if (rc || n == 0) return rc;
  tc::Meta meta;
  tc::make_meta(d, order, &meta, nullptr);
  const unsigned char* img = reinterpret_cast<const unsigned char*>(image);
  switch (d) {
    case 2: return tc::launch_inverse<2>(y, n, img, meta, ladj_in, last_layer, v, ladj_out, st);
    case 3: return tc::launch_inverse<3>(y, n, img, meta, ladj_in, last_layer, v, ladj_out, st);
    case 4: return tc::launch_inverse<4>(y, n, img, meta, ladj_in, last_layer, v, ladj_out, st);
    case 5: return tc::launch_inverse<5>(y, n, img, meta, ladj_in, last_layer, v, ladj_out, st);
    case 6: return tc::launch_inverse<6>(y, n, img, meta, ladj_in, last_layer, v, ladj_out, st);
    default: return MFB_E_UNSUPPORTED;
  }
}

int nsf_tc_spline_bwd(const float* v, const float* gy, const float* glogq, int64_t n, int d, const void* image,
                      const int32_t* order, int first_layer, float* acts, float* gphi, uint32_t* masks, float* gvd,
                      float* gmax, int* gmaxes, cudaStream_t st) {
  tc::Meta meta;
  tc::make_meta(d, order, &meta, nullptr);
  const unsigned char* img = reinterpret_cast<const unsigned char*>(image);
  const tc::BwdIO bio = {gy, glogq, acts, gphi, masks, gvd, gmax, gmaxes};
  switch (d) {
    case 2: return tc::launch_layer_bwd<2>(v, n, img, meta, first_layer, bio, st);
    case 3: return tc::launch_layer_bwd<3>(v, n, img, meta, first_layer, bio, st);
    case 4: return tc::launch_layer_bwd<4>(v, n, img, meta, first_layer, bio, st);
    case 5: return tc::launch_layer_bwd<5>(v, n, img, meta, first_layer, bio, st);
    case 6: return tc::launch_layer_bwd<6>(v, n, img, meta, first_layer, bio, st);
    default: return MFB_E_UNSUPPORTED;
  }
}

}  // namespace mfb

using namespace mfb;

extern "C" {

#ifdef MFB_TC_TRACE
int mfb_debug_copy_trace(long long* host) {
  return (int)cudaMemcpyFromSymbol(host, tc::g_trace, sizeof(long long) * 4 * 1024);
}
#endif

int mfb_nsf_tc_supported(int d, int hidden_units, int hidden_layers, int bins) {
  return (d >= 2 && d <= 6 && hidden_units == kH && hidden_layers == 3 && bins == 20) ? 1 : 0;
}

int64_t mfb_nsf_tc_image_bytes(int d, int hidden_layers) {
  if (d < 2 || d > 6 || hidden_layers < 1 || hidden_layers > 3) return 0;
  return tc::image_bytes(d, hidden_layers);
}

int mfb_nsf_tc_prepare(const float* params, int64_t layer_stride_floats, int n_layers, int d, int hidden_units,
                       int hidden_layers, int bins, const int32_t* orders_host, void* images, void* stream) {
  MFB_CHECK_ARG(params && orders_host && images && n_layers > 0);
  if (!mfb_nsf_tc_supported(d, hidden_units, hidden_layers, bins)) return MFB_E_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int img_bytes = tc::image_bytes(d, hidden_layers);
  for (int l0 = 0; l0 < n_layers; l0 += tc::kMaxPrepLayers) {
    const int nl = n_layers - l0 < tc::kMaxPrepLayers ? n_layers - l0 : tc::kMaxPrepLayers;
    tc::PrepArgs args = {};
    int cls[kH];
    tc::hidden_classes(d, cls, args.perm);
    for (int l = 0; l < nl; ++l) {
      if (!tc::valid_order(d, orders_host + (size_t)(l0 + l) * d)) return MFB_E_BADARG;
      tc::make_meta(d, orders_host + (size_t)(l0 + l) * d, nullptr, &args.layer[l]);
    }
    MFB_CUDA(cudaMemsetAsync(reinterpret_cast<unsigned char*>(images) + (size_t)l0 * img_bytes, 0,
                             (size_t)nl * img_bytes, st));
    tc::nsf_tc_prepare_kernel<<<dim3(nl, tc::kPrepSlices), 256, 0, st>>>(
        params, layer_stride_floats, d, hidden_layers, bins, args, l0, reinterpret_cast<unsigned char*>(images),
        img_bytes);
    const int rc = launch_status();
    if (rc) return rc;
  }
  return 0;
}

}  // extern "C"
