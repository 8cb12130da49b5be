// Register-resident rational-quadratic spline of the tcgen05 flow kernels (forward, forward + backward,
// bias-only table form).  Kept in a header of its own, written against MFB_HD helpers, so that the very
// same source also compiles for the HOST: tests/csrc/spline_host.cu builds it with the approximate
// MUFU operations replaced by libm calls and checks the arithmetic against the float64 oracle on a
// machine without a GPU (tests/test_spline_host.py).  Reference: zuko 1.3.1 MonotonicRQSTransform as
// called from generate/flows/zuko.py:24-29 (SURVEY.md App. A.3).
#pragma once
#include <math.h>

#include "nsf_common.cuh"

#define MFB_HD __host__ __device__ __forceinline__

namespace mfb {
namespace tc {

constexpr int kCT = 24;              // stride of the constant-feature tables (floats)
constexpr int kConstRows = 7;        // x0 | dx | y0 | dy | d0 | d1 | x0 - fl(x0)
constexpr int kConstFloats = kConstRows * kCT + kPP;   // knot tables + the raw parameters (x log2 e) of the bias-only feature

MFB_HD float sp_exp2(float x) {
#ifdef __CUDA_ARCH__
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return exp2f(x);
#endif
}
MFB_HD float sp_rcp(float x) {
#ifdef __CUDA_ARCH__
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
#else
  return 1.0f / x;
#endif
}
MFB_HD float sp_add(float a, float b) {
#ifdef __CUDA_ARCH__
  return __fadd_rn(a, b);
#else
  volatile float s = a + b;
  return s;
#endif
}

// MUFU reciprocal + one Newton step (the raw approximation's 1 ulp is amplified by the
// ill-conditioned knot sums; with the step the spline is as accurate as a divide)
MFB_HD float rcp_nr(float x) {
  const float r = sp_rcp(x);
  return fmaf(r, fmaf(-x, r, 1.0f), r);
}

// soft clip + exp of two raw (log2e-scaled) parameters with one reciprocal:
//   e = 2^(t / (1 + c |t|))
MFB_HD void clip_exp2_pair(float t0, float t1, float c, float& e0, float& e1) {
  const float d0 = fmaf(fabsf(t0), c, 1.0f), d1 = fmaf(fabsf(t1), c, 1.0f);
#ifdef MFB_TC_EXACT
  e0 = exp2f(t0 / d0);
  e1 = exp2f(t1 / d1);
#else
  const float r = sp_rcp(d0 * d1);
  e0 = sp_exp2(t0 * (r * d1));
  e1 = sp_exp2(t1 * (r * d0));
#endif
}

// Packed fp32 pairs (Blackwell FMUL2 / FADD2 / FFMA2: two IEEE round-to-nearest lanes for ONE issue slot -- the flow
// kernel is bound by issue slots, not by the FMA pipe; scripts/micro/ffma2_bench.cu).  Lane results are bit-identical
// to the scalar operations, so the host build (and the parity statistics) see the same arithmetic.
#ifndef MFB_F32X2
#define MFB_F32X2 1
#endif
MFB_HD void mul2(float a0, float a1, float b0, float b1, float& c0, float& c1) {
#if defined(__CUDA_ARCH__) && MFB_F32X2
  unsigned long long a, b, c;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(c) : "l"(a), "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(c0), "=f"(c1) : "l"(c));
#else
  c0 = a0 * b0;
  c1 = a1 * b1;
#endif
}
MFB_HD void add2(float a0, float a1, float b0, float b1, float& c0, float& c1) {
#if defined(__CUDA_ARCH__) && MFB_F32X2
  unsigned long long a, b, c;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(c) : "l"(a), "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(c0), "=f"(c1) : "l"(c));
#else
  c0 = sp_add(a0, b0);
  c1 = sp_add(a1, b1);
#endif
}

// the same for four parameters with ONE reciprocal (the spline phases are bound by the MUFU pipe:
// 8 issue slots per MUFU instruction, so three extra multiplies per quad are the cheaper side)
MFB_HD void clip_exp2_quad(float t0, float t1, float t2, float t3, float c, float& e0, float& e1,
                                               float& e2, float& e3) {
  const float d0 = fmaf(fabsf(t0), c, 1.0f), d1 = fmaf(fabsf(t1), c, 1.0f);
  const float d2 = fmaf(fabsf(t2), c, 1.0f), d3 = fmaf(fabsf(t3), c, 1.0f);
  // packed where the operands are pairs already: (t0, t1) and (t2, t3) are neighbours in the tcgen05.ld result
  float p01, p23, x0, x1, x2, x3;
  mul2(d0, d2, d1, d3, p01, p23);
  const float r = sp_rcp(p01 * p23);
  const float r01 = r * p23, r23 = r * p01;   // 1 / (d0 d1), 1 / (d2 d3)
  mul2(t0, t1, r01 * d1, r01 * d0, x0, x1);
  mul2(t2, t3, r23 * d3, r23 * d2, x2, x3);
  e0 = sp_exp2(x0);
  e1 = sp_exp2(x1);
  e2 = sp_exp2(x2);
  e3 = sp_exp2(x3);
}

// error-free addition (Knuth): s = fl(a + b), err = (a + b) - s exactly
MFB_HD void two_sum(float a, float b, float& s, float& err) {
  s = sp_add(a, b);
  const float bb = sp_add(s, -a);
  err = sp_add(sp_add(a, -sp_add(s, -bb)), sp_add(b, -bb));
}

#ifndef MFB_SPLINE_COMP
#define MFB_SPLINE_COMP 1   // 0: plain fp32 group prefixes; 1: widths carried as (hi, lo); 2: widths and heights
#endif

// Rational-quadratic spline of one feature from the raw conditioner outputs a[0..3NB-2] (already
// multiplied by log2 e through the weights, bias included by the bias MMA).  Works in
// un-normalised softmax units: bin width / height come from e_k directly (no differencing of knots).
// The search is two-level -- which group of four bins, then which bin of the group -- with
// predicated selects, so that nothing is indexed dynamically and everything stays in registers.
//
// Where the rounding goes (scripts/emul_spline.py, measured against float64 on the benchmark's
// weights): everything that decides the position inside the bin is formed as a DIFFERENCE FROM THE
// CENTRE of the knot array, rounded once at its own (small) magnitude:
//     numer = u * sum + (sum / 2 - P_g) - (running sum inside the group),   u = v / 2B
// with one fused multiply-add, instead of target = (v + B) / 2B * sum (three roundings at the
// magnitude of the sum) minus a running sum that was itself rounded at every step; the left knot in y
// likewise as (Q_g - sumh / 2 + inside) / sumh.  v and u are exact inputs, so particles near the
// centre -- most of them -- see knots accurate to an ulp of their own distance from it.  This puts
// the fp32 result at the accuracy of the reference's own fp32 evaluation (fraction of log q beyond
// 1e-4 of float64: 1.0-1.2x torch-fp32's, was 4x).  MFB_SPLINE_COMP additionally carries the group
// prefixes as (hi, lo) pairs (0.3-0.9x torch-fp32's).
// Multiplies jac by dy/dv (1 outside [-B, B]) and returns y.
//
// The raw parameters come in two pieces through load(col, float (&dst)[N]) = columns [col, col + N): the NB
// widths first, then the NB heights and NB - 1 derivatives (plus one padding column) once the widths are reduced
// to the few values the search keeps.  The flow kernel reads them from tensor memory that way, so that at most
// 2 NB of the 64 accumulator columns are live in registers; the loader sees the second piece last and may
// release the accumulator after it.
template <int NB, class Load>
MFB_HD float rq_spline_regs_ld(Load&& load, float v, float& jac) {
  static_assert(NB % 4 == 0 && NB >= 8, "bins are searched in groups of four");
  constexpr int G = NB / 4;
  constexpr float cW = kClipW / kLog2e, cD = kClipD / kLog2e;
  // ---- widths: e_j, sums of the groups of four and their prefixes P_g (short dependency chains)
  float e[NB], pre[G + 1], plo[G + 1];
  {
    float aw[NB];
    load(0, aw);
#pragma unroll
    for (int j = 0; j < NB; j += 4) {
      clip_exp2_quad(aw[j], aw[j + 1], aw[j + 2], aw[j + 3], cW, e[j], e[j + 1], e[j + 2], e[j + 3]);
    }
  }
  pre[0] = 0.f;
  plo[0] = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float s01, s23;
    add2(e[4 * g], e[4 * g + 2], e[4 * g + 1], e[4 * g + 3], s01, s23);
    const float gs = s01 + s23;
    if (MFB_SPLINE_COMP >= 1 && g > 0) {
      float err;
      two_sum(pre[g], gs, pre[g + 1], err);
      plo[g + 1] = plo[g] + err;
    } else {
      pre[g + 1] = pre[g] + gs;
      plo[g + 1] = 0.f;
    }
  }
  const float sum = pre[G], half = 0.5f * sum;
  const float u = v * (0.5f / kBound);
  const float target = fmaf(u, sum, half);
  // level 1: pg[g] <=> the bin of v lies beyond group g (monotone in g)
  bool pg[G - 1];
#pragma unroll
  for (int g = 0; g < G - 1; ++g) pg[g] = pre[g + 1] < target;
  float q0 = e[0], q1 = e[1], q2 = e[2], q3 = e[3], xg = 0.f, xgl = 0.f;
#pragma unroll
  for (int g = 1; g < G; ++g) {
    q0 = pg[g - 1] ? e[4 * g] : q0;
    q1 = pg[g - 1] ? e[4 * g + 1] : q1;
    q2 = pg[g - 1] ? e[4 * g + 2] : q2;
    q3 = pg[g - 1] ? e[4 * g + 3] : q3;
    xg = pg[g - 1] ? pre[g] : xg;
    if (MFB_SPLINE_COMP >= 1) xgl = pg[g - 1] ? plo[g] : xgl;
  }
  // level 2: what is left of the target inside the group, then the bin of the group
  float cen = half - xg;
  if (MFB_SPLINE_COMP >= 1) cen += fmaf(0.5f, plo[G], -xgl);
  const float rem = fmaf(u, sum, cen);
  const float i1 = q0 + q1, i2 = i1 + q2;
  const bool r0 = q0 < rem, r1 = i1 < rem, r2 = i2 < rem;
  const float numer = rem - (r2 ? i2 : (r1 ? i1 : (r0 ? q0 : 0.f)));
  const float ek = r2 ? q3 : (r1 ? q2 : (r0 ? q1 : q0));
  float a[2 * NB];   // a[j] = raw parameter NB + j: heights, then derivatives
  load(NB, a);
  // ---- heights, one group at a time
  float run = 0.f, runl = 0.f, yg = 0.f, ygl = 0.f, h0s = 0.f, h1s = 0.f, h2s = 0.f, h3s = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    float h0, h1, h2, h3;
    clip_exp2_quad(a[4 * g], a[4 * g + 1], a[4 * g + 2], a[4 * g + 3], cW, h0, h1, h2, h3);
    const bool take = g == 0 ? true : pg[g > 0 ? g - 1 : 0];
    h0s = take ? h0 : h0s;
    h1s = take ? h1 : h1s;
    h2s = take ? h2 : h2s;
    h3s = take ? h3 : h3s;
    yg = take ? run : yg;
    float s01, s23;
    add2(h0, h2, h1, h3, s01, s23);
    const float gs = s01 + s23;
    if (MFB_SPLINE_COMP >= 2 && g > 0) {
      ygl = take ? runl : ygl;
      float err;
      two_sum(run, gs, run, err);
      runl += err;
    } else {
      run += gs;
    }
  }
  const float sumh = run;
  const float j1h = h0s + h1s, j2h = j1h + h2s;
  float ycen = (yg - 0.5f * sumh) + (r2 ? j2h : (r1 ? j1h : (r0 ? h0s : 0.f)));   // left knot of the bin from the centre
  if (MFB_SPLINE_COMP >= 2) ycen += fmaf(-0.5f, runl, ygl);
  const float hk = r2 ? h3s : (r1 ? h2s : (r0 ? h1s : h0s));
  // ---- derivatives at the two knots of the bin (raw 0 -> slope 1 at the outer knots):
  //      u[-1..3] = raw parameters of the knots around the group's four bins
  float um = 0.f, u0 = 0.f, u1 = 0.f, u2 = 0.f, u3 = 0.f, prev = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    const float t0 = a[NB + 4 * g], t1 = a[NB + 4 * g + 1], t2 = a[NB + 4 * g + 2];
    const float t3 = (4 * g + 3 < NB - 1) ? a[NB + 4 * g + 3] : 0.f;
    const bool take = g == 0 ? true : pg[g > 0 ? g - 1 : 0];
    um = take ? prev : um;
    u0 = take ? t0 : u0;
    u1 = take ? t1 : u1;
    u2 = take ? t2 : u2;
    u3 = take ? t3 : u3;
    prev = t3;
  }
  const float tl = r2 ? u2 : (r1 ? u1 : (r0 ? u0 : um));
  const float tr = r2 ? u3 : (r1 ? u2 : (r0 ? u1 : u0));
  float d0, d1;
  clip_exp2_pair(tl, tr, cD, d0, d1);
  // ---- rational quadratic
  const float r_e = rcp_nr(ek), r_sh = rcp_nr(sumh);
  float t = numer * r_e;
  t = fminf(fmaxf(t, 0.0f), 1.0f);
  const float hn = hk * r_sh;                 // normalised bin height / 2B
  const float s = hn * sum * r_e;             // dy / dx
  const float omt = 1.0f - t, tomt = t * omt;
  const float den = fmaf(d0 + d1 - 2.0f * s, tomt, s);
  const float r_den = rcp_nr(den);
  const float y0 = 2.0f * kBound * (ycen * r_sh);
  const float y = fmaf(2.0f * kBound * hn * (s * t * t + d0 * tomt), r_den, y0);
  const float j1 = s * s * (2.0f * s * tomt + d0 * omt * omt + d1 * t * t) * r_den * r_den;
  const bool inside = (v > -kBound) && (v <= kBound);
  jac *= inside ? j1 : 1.0f;
  return inside ? y : v;
}
// ... from all raw parameters at once
template <int NB>
MFB_HD float rq_spline_regs(const float (&a)[64], float v, float& jac) {
  return rq_spline_regs_ld<NB>(
      [&](int col, auto& dst) {
        for (int j = 0; j < (int)(sizeof(dst) / sizeof(dst[0])); ++j) dst[j] = a[col + j];
      },
      v, jac);
}

// soft clip + exp of four parameters like clip_exp2_quad; additionally returns 1 / (1 + c |t_j|) in place
// of t_j: the derivative of the clip is its square
MFB_HD void clip_exp2_quad_bwd(float& t0, float& t1, float& t2, float& t3, float c, float& e0,
                                                   float& e1, float& e2, float& e3) {
  const float d0 = fmaf(fabsf(t0), c, 1.0f), d1 = fmaf(fabsf(t1), c, 1.0f);
  const float d2 = fmaf(fabsf(t2), c, 1.0f), d3 = fmaf(fabsf(t3), c, 1.0f);
  const float p01 = d0 * d1, p23 = d2 * d3;
  const float r = sp_rcp(p01 * p23);
  const float r01 = r * p23, r23 = r * p01;
  const float i0 = r01 * d1, i1 = r01 * d0, i2 = r23 * d3, i3 = r23 * d2;
  e0 = sp_exp2(t0 * i0);
  e1 = sp_exp2(t1 * i1);
  e2 = sp_exp2(t2 * i2);
  e3 = sp_exp2(t3 * i3);
  t0 = i0; t1 = i1; t2 = i2; t3 = i3;
}

// Spline forward + backward of one feature in registers (backward variant of rq_spline_regs; the
// formulas are those of rq_spline_backward in nsf_bwd.cu, prototype scripts/proto_spline_bwd.py).
// a[]: raw parameters (x log2 e) in, dL/d(raw natural parameter) out (j < 3NB-1).  gy = dL/dy,
// gl = dL/d(log dy/dv).  Returns the direct dL/dv.
struct KnotGrad {   // the derivative block of dL/dphi has two non-zero entries: knots k-1 and k of the particle's bin k
  float left, right;
  int bin;
};
template <int NB>
MFB_HD float rq_spline_regs_bwd(float (&a)[64], float v, float gy, float gl, KnotGrad* kg = nullptr) {
  static_assert(NB % 4 == 0 && NB >= 8, "bins are searched in groups of four");
  constexpr int G = NB / 4;
  constexpr float cW = kClipW / kLog2e, cD = kClipD / kLog2e;
  float e[NB], h[NB], pre[G + 1], preh[G + 1];
#pragma unroll
  for (int j = 0; j < NB; j += 4) {
    clip_exp2_quad_bwd(a[j], a[j + 1], a[j + 2], a[j + 3], cW, e[j], e[j + 1], e[j + 2], e[j + 3]);
    clip_exp2_quad_bwd(a[NB + j], a[NB + j + 1], a[NB + j + 2], a[NB + j + 3], cW, h[j], h[j + 1], h[j + 2], h[j + 3]);
  }
  pre[0] = 0.f;
  preh[0] = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    pre[g + 1] = pre[g] + ((e[4 * g] + e[4 * g + 1]) + (e[4 * g + 2] + e[4 * g + 3]));
    preh[g + 1] = preh[g] + ((h[4 * g] + h[4 * g + 1]) + (h[4 * g + 2] + h[4 * g + 3]));
  }
  const float sum = pre[G], sumh = preh[G];
  const float half = 0.5f * sum, u = v * (0.5f / kBound);
  const float target = fmaf(u, sum, half);
  // two-level search as in the forward pass (same centred differences), plus the integer bin index
  // for the scatter below
  int gsel = 0;
  float q0 = e[0], q1 = e[1], q2 = e[2], q3 = e[3], xg = 0.f;
  float h0s = h[0], h1s = h[1], h2s = h[2], h3s = h[3], yg = 0.f;
  // raw derivative parameters of the knots around the group's four bins (u[-1..3], raw 0 at the outer
  // knots), selected with the same predicates: nothing is indexed dynamically, so a[] stays in registers
  float um = 0.f, u0 = a[2 * NB], u1 = a[2 * NB + 1], u2 = a[2 * NB + 2], u3 = a[2 * NB + 3];
#pragma unroll
  for (int g = 1; g < G; ++g) {
    const bool pgm = pre[g] < target;
    gsel += pgm ? 1 : 0;
    um = pgm ? a[2 * NB + 4 * g - 1] : um;
    u0 = pgm ? a[2 * NB + 4 * g] : u0;
    u1 = pgm ? a[2 * NB + 4 * g + 1] : u1;
    u2 = pgm ? a[2 * NB + 4 * g + 2] : u2;
    u3 = pgm ? ((4 * g + 3 < NB - 1) ? a[2 * NB + 4 * g + 3] : 0.f) : u3;
    q0 = pgm ? e[4 * g] : q0;
    q1 = pgm ? e[4 * g + 1] : q1;
    q2 = pgm ? e[4 * g + 2] : q2;
    q3 = pgm ? e[4 * g + 3] : q3;
    xg = pgm ? pre[g] : xg;
    h0s = pgm ? h[4 * g] : h0s;
    h1s = pgm ? h[4 * g + 1] : h1s;
    h2s = pgm ? h[4 * g + 2] : h2s;
    h3s = pgm ? h[4 * g + 3] : h3s;
    yg = pgm ? preh[g] : yg;
  }
  const float rem = fmaf(u, sum, half - xg);
  const float i1 = q0 + q1, i2 = i1 + q2;
  const bool r0 = q0 < rem, r1 = i1 < rem, r2 = i2 < rem;
  const int k = 4 * gsel + (r0 ? 1 : 0) + (r1 ? 1 : 0) + (r2 ? 1 : 0);
  const float inner = r2 ? i2 : (r1 ? i1 : (r0 ? q0 : 0.f));
  const float numer = rem - inner;
  const float x0c = xg + inner;
  const float ek = r2 ? q3 : (r1 ? q2 : (r0 ? q1 : q0));
  const float j1h = h0s + h1s, j2h = j1h + h2s;
  const float y0c = yg + (r2 ? j2h : (r1 ? j1h : (r0 ? h0s : 0.f)));
  const float hk = r2 ? h3s : (r1 ? h2s : (r0 ? h1s : h0s));
  // derivative parameters at the two knots of bin k (raw 0 at the outer knots)
  const float tl = r2 ? u2 : (r1 ? u1 : (r0 ? u0 : um));
  const float tr = r2 ? u3 : (r1 ? u2 : (r0 ? u1 : u0));
  const float dd0 = fmaf(fabsf(tl), cD, 1.0f), dd1 = fmaf(fabsf(tr), cD, 1.0f);
  const float rdd = sp_rcp(dd0 * dd1);
  const float ri0 = rdd * dd1, ri1 = rdd * dd0;
  const float d0 = sp_exp2(tl * ri0), d1 = sp_exp2(tr * ri1);
  // forward quantities in natural units
  const float inv_s = rcp_nr(sum), inv_sh = rcp_nr(sumh);
  const float wk = ek * inv_s, hn = hk * inv_sh;
  const float cumw = x0c * inv_s, cumh = y0c * inv_sh;
  const float dx = 2.0f * kBound * wk, dy = 2.0f * kBound * hn;
  const float r_wk = rcp_nr(wk), r_dx = rcp_nr(dx);
  const float s = hn * r_wk;
  float t = numer * rcp_nr(ek);
  t = fminf(fmaxf(t, 0.0f), 1.0f);
  const float omt = 1.0f - t, q = t * omt;
  const float A = d0 + d1 - 2.0f * s;
  const float den = fmaf(A, q, s);
  const float n1 = s * t * t + d0 * q;
  const float n2 = 2.0f * s * q + d0 * omt * omt + d1 * t * t;
  const float dq_dt = 1.0f - 2.0f * t;
  const float dden_dt = A * dq_dt, dden_ds = 1.0f - 2.0f * q, dden_dd = q;
  const float inv_den = rcp_nr(den), inv_n2 = rcp_nr(n2);
  const float r1q = n1 * inv_den;
  const float dy_dt = dy * (2.0f * s * t + d0 * dq_dt - r1q * dden_dt) * inv_den;
  const float dy_ds = dy * (t * t - r1q * dden_ds) * inv_den;
  const float dy_dd0 = dy * (q - r1q * dden_dd) * inv_den;
  const float dy_dd1 = dy * (-r1q * dden_dd) * inv_den;
  const float dl_dt = (2.0f * s * dq_dt - 2.0f * d0 * omt + 2.0f * d1 * t) * inv_n2 - 2.0f * dden_dt * inv_den;
  const float dl_ds = 2.0f * rcp_nr(s) + 2.0f * q * inv_n2 - 2.0f * dden_ds * inv_den;
  const float dl_dd0 = omt * omt * inv_n2 - 2.0f * dden_dd * inv_den;
  const float dl_dd1 = t * t * inv_n2 - 2.0f * dden_dd * inv_den;
  const float g_t = gy * dy_dt + gl * dl_dt;
  const float g_s = gy * dy_ds + gl * dl_ds;
  const float g_d0 = gy * dy_dd0 + gl * dl_dd0;
  const float g_d1 = gy * dy_dd1 + gl * dl_dd1;
  const float g_dy = gy * r1q;
  const float gv = g_t * r_dx;
  const float g_dx = -g_t * t * r_dx;
  const float gW_lo = -2.0f * kBound * gv;
  const float gW_k = 2.0f * kBound * g_dx - g_s * s * r_wk;
  const float gH_lo = 2.0f * kBound * gy;
  const float gH_k = 2.0f * kBound * g_dy + g_s * r_wk;
  const float dotW = gW_lo * cumw + gW_k * wk;
  const float dotH = gH_lo * cumh + gH_k * hn;
  const bool inside = (v > -kBound) && (v <= kBound);
  const float live = inside ? 1.0f : 0.0f;   // identity outside the spline box: no parameter gradient
  const float ws = inv_s * live, hs = inv_sh * live;
#pragma unroll
  for (int j = 0; j < NB; ++j) {
    const float gw = (j < k ? gW_lo : (j == k ? gW_k : 0.f)) - dotW;
    const float gh = (j < k ? gH_lo : (j == k ? gH_k : 0.f)) - dotH;
    a[j] = (e[j] * ws) * gw * (a[j] * a[j]);                  // softmax Jacobian, then the clip derivative
    a[NB + j] = (h[j] * hs) * gh * (a[NB + j] * a[NB + j]);
  }
  const float gd0 = g_d0 * d0 * ri0 * ri0 * live, gd1 = g_d1 * d1 * ri1 * ri1 * live;
#pragma unroll
  for (int j = 0; j < NB - 1; ++j) a[2 * NB + j] = (j == k - 1) ? gd0 : ((j == k) ? gd1 : 0.f);
  if (kg) {   // the outer knots (k - 1 = -1, k = NB - 1) have fixed slope 1: no parameter
    kg->left = k > 0 ? gd0 : 0.f;
    kg->right = k < NB - 1 ? gd1 : 0.f;
    kg->bin = k;
  }
  return inside ? gv : gy;
}

// Inverse of the same spline (density direction, generate/flows/zuko.py:21-22,31-32,43-50): returns v with RQS(v) = y
// and multiplies jac by dy/dv at v (the forward Jacobian log_prob needs).  The bin is searched over the HEIGHT
// prefixes with the same centred differences as the forward search over the widths; inside the bin, with
// eta = (y - y0) / dy in [0, 1]:  a = (s - d0) + eta A,  b = d0 - eta A,  c = -s eta,  A = d0 + d1 - 2 s,
// z = 2 c / (-b - sqrt(b^2 - 4 a c))  (zuko's numerically stable root), v = x0 + z dx.
template <int NB>
MFB_HD float rq_spline_regs_inv(const float (&a)[64], float y, float& jac) {
  static_assert(NB % 4 == 0 && NB >= 8, "bins are searched in groups of four");
  constexpr int G = NB / 4;
  constexpr float cW = kClipW / kLog2e, cD = kClipD / kLog2e;
  float e[NB], h[NB], pre[G + 1], preh[G + 1];
#pragma unroll
  for (int j = 0; j < NB; j += 4) {
    clip_exp2_quad(a[j], a[j + 1], a[j + 2], a[j + 3], cW, e[j], e[j + 1], e[j + 2], e[j + 3]);
    clip_exp2_quad(a[NB + j], a[NB + j + 1], a[NB + j + 2], a[NB + j + 3], cW, h[j], h[j + 1], h[j + 2], h[j + 3]);
  }
  pre[0] = 0.f;
  preh[0] = 0.f;
#pragma unroll
  for (int g = 0; g < G; ++g) {
    pre[g + 1] = pre[g] + ((e[4 * g] + e[4 * g + 1]) + (e[4 * g + 2] + e[4 * g + 3]));
    preh[g + 1] = preh[g] + ((h[4 * g] + h[4 * g + 1]) + (h[4 * g + 2] + h[4 * g + 3]));
  }
  const float sum = pre[G], sumh = preh[G];
  const float halfh = 0.5f * sumh, uy = y * (0.5f / kBound);
  const float targeth = fmaf(uy, sumh, halfh);
  float q0 = e[0], q1 = e[1], q2 = e[2], q3 = e[3], xg = 0.f;
  float h0s = h[0], h1s = h[1], h2s = h[2], h3s = h[3], yg = 0.f;
  float um = 0.f, u0 = a[2 * NB], u1 = a[2 * NB + 1], u2 = a[2 * NB + 2], u3 = a[2 * NB + 3];
#pragma unroll
  for (int g = 1; g < G; ++g) {
    const bool pgm = preh[g] < targeth;
    um = pgm ? a[2 * NB + 4 * g - 1] : um;
    u0 = pgm ? a[2 * NB + 4 * g] : u0;
    u1 = pgm ? a[2 * NB + 4 * g + 1] : u1;
    u2 = pgm ? a[2 * NB + 4 * g + 2] : u2;
    u3 = pgm ? ((4 * g + 3 < NB - 1) ? a[2 * NB + 4 * g + 3] : 0.f) : u3;
    q0 = pgm ? e[4 * g] : q0;
    q1 = pgm ? e[4 * g + 1] : q1;
    q2 = pgm ? e[4 * g + 2] : q2;
    q3 = pgm ? e[4 * g + 3] : q3;
    xg = pgm ? pre[g] : xg;
    h0s = pgm ? h[4 * g] : h0s;
    h1s = pgm ? h[4 * g + 1] : h1s;
    h2s = pgm ? h[4 * g + 2] : h2s;
    h3s = pgm ? h[4 * g + 3] : h3s;
    yg = pgm ? preh[g] : yg;
  }
  const float remh = fmaf(uy, sumh, halfh - yg);
  const float j1 = h0s + h1s, j2 = j1 + h2s;
  const bool r0 = h0s < remh, r1 = j1 < remh, r2 = j2 < remh;
  const float numer = remh - (r2 ? j2 : (r1 ? j1 : (r0 ? h0s : 0.f)));       // (y - y0) in un-normalised height units
  const float hk = r2 ? h3s : (r1 ? h2s : (r0 ? h1s : h0s));
  const float i1 = q0 + q1, i2 = i1 + q2;
  const float xcen = (xg - 0.5f * sum) + (r2 ? i2 : (r1 ? i1 : (r0 ? q0 : 0.f)));   // left knot of the bin from the centre
  const float ek = r2 ? q3 : (r1 ? q2 : (r0 ? q1 : q0));
  const float tl = r2 ? u2 : (r1 ? u1 : (r0 ? u0 : um));
  const float tr = r2 ? u3 : (r1 ? u2 : (r0 ? u1 : u0));
  float d0, d1;
  clip_exp2_pair(tl, tr, cD, d0, d1);
  const float r_s = rcp_nr(sum), r_hk = rcp_nr(hk);
  float eta = numer * r_hk;
  eta = fminf(fmaxf(eta, 0.0f), 1.0f);
  const float s = (hk * rcp_nr(sumh)) * sum * rcp_nr(ek);   // dy / dx
  const float A = d0 + d1 - 2.0f * s;
  const float qa = fmaf(eta, A, s - d0), qb = fmaf(-eta, A, d0), qc = -s * eta;
  const float disc = fmaxf(fmaf(qb, qb, -4.0f * qa * qc), 0.0f);
  float z = (2.0f * qc) * rcp_nr(-qb - sqrtf(disc));
  z = fminf(fmaxf(z, 0.0f), 1.0f);
  const float omz = 1.0f - z, zomz = z * omz;
  const float den = fmaf(A, zomz, s);
  const float r_den = rcp_nr(den);
  const float jj = s * s * (2.0f * s * zomz + d0 * omz * omz + d1 * z * z) * r_den * r_den;
  const float v = 2.0f * kBound * (fmaf(z, ek, xcen) * r_s);
  const bool inside = (y > -kBound) && (y <= kBound);
  jac *= inside ? jj : 1.0f;
  return inside ? v : y;
}

// ... and of the bias-only spline from the knot tables
template <int NB>
MFB_HD float rq_spline_const_inv(const float* __restrict__ ct, float y, float& jac) {
  int k = 0;
#pragma unroll
  for (int j = 1; j < NB; ++j) k += (ct[2 * kCT + j] < y) ? 1 : 0;
  const float x0 = ct[k], dx = ct[kCT + k], y0 = ct[2 * kCT + k], dy = ct[3 * kCT + k];
  const float d0 = ct[4 * kCT + k], d1 = ct[5 * kCT + k];
  const float s = dy * rcp_nr(dx);
  float eta = (y - y0) * rcp_nr(dy);
  eta = fminf(fmaxf(eta, 0.0f), 1.0f);
  const float A = d0 + d1 - 2.0f * s;
  const float qa = fmaf(eta, A, s - d0), qb = fmaf(-eta, A, d0), qc = -s * eta;
  const float disc = fmaxf(fmaf(qb, qb, -4.0f * qa * qc), 0.0f);
  float z = (2.0f * qc) * rcp_nr(-qb - sqrtf(disc));
  z = fminf(fmaxf(z, 0.0f), 1.0f);
  const float omz = 1.0f - z, zomz = z * omz;
  const float den = fmaf(A, zomz, s);
  const float r_den = rcp_nr(den);
  const float jj = s * s * (2.0f * s * zomz + d0 * omz * omz + d1 * z * z) * r_den * r_den;
  const float v = fmaf(z, dx, x0) + ct[6 * kCT + k];
  const bool inside = (y > -kBound) && (y <= kBound);
  jac *= inside ? jj : 1.0f;
  return inside ? v : y;
}

// bias-only spline from the precomputed knot tables (shared memory, broadcast reads)
template <int NB>
MFB_HD float rq_spline_const(const float* __restrict__ ct, float v, float& jac) {
  int k = 0;
#pragma unroll
  for (int j = 1; j < NB; ++j) k += (ct[j] < v) ? 1 : 0;
  const float x0 = ct[k], dx = ct[kCT + k], y0 = ct[2 * kCT + k], dy = ct[3 * kCT + k];
  const float d0 = ct[4 * kCT + k], d1 = ct[5 * kCT + k];
  const float r_dx = rcp_nr(dx);
  const float s = dy * r_dx;
  float t = ((v - x0) - ct[6 * kCT + k]) * r_dx;
  t = fminf(fmaxf(t, 0.0f), 1.0f);
  const float omt = 1.0f - t, tomt = t * omt;
  const float den = fmaf(d0 + d1 - 2.0f * s, tomt, s);
  const float r_den = rcp_nr(den);
  const float y = fmaf(dy * (s * t * t + d0 * tomt), r_den, y0);
  const float j1 = s * s * (2.0f * s * tomt + d0 * omt * omt + d1 * t * t) * r_den * r_den;
  const bool inside = (v > -kBound) && (v <= kBound);
  jac *= inside ? j1 : 1.0f;
  return inside ? y : v;
}

}  // namespace tc
}  // namespace mfb
