// bean_math.cuh -- in-register special functions for the bean SVI kernels (sm_100a).
//
// These replace the torch.lgamma / torch.digamma / erf sweeps behind pyro's
// DirichletMultinomial.log_prob, its backward and get_std_normal_prob
// (reference call sites: bean/model/model.py:138-164, :531-547; bean/model/utils.py:34-76).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace bean {

// MUFU reciprocal / log2 in their flush-to-zero form.  Without -ftz nvcc wraps every `__fdividef` / `__logf` in denormal
// pre-scaling (FSETP + FMUL 2^24 + FSEL ... ~4 extra instructions each); their arguments here are never denormal
// (concentrations >= 1e-5, counts, sums of those), and an issue-bound kernel pays for every instruction: this removed
// a fifth of the per-bin instruction count.
__device__ __forceinline__ float rcp_ftz(float x) {
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float log_ftz(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r * 0.69314718055994530942f;
}

// Asynchronous global -> shared copies (LDGSTS): the data of the NEXT replicate is put in flight while the current one is
// evaluated, without holding registers for it.  Each thread copies and later reads only its own slots, so no CTA barrier is
// involved: cp.async.wait_group orders the thread's own copies.
__device__ __forceinline__ void cp_async_16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_8(void* smem, const void* gmem) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(smem)), "l"(gmem));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// Library functions with long bodies are called through ONE out-of-line copy each: the SVI kernel is bound by
// instruction issue AND by its instruction-cache footprint, and a call costs far less than a duplicated body.
static __device__ __noinline__ float ool_logf(float x) { return logf(x); }
static __device__ __noinline__ float ool_log1pf(float x) { return log1pf(x); }
static __device__ __noinline__ float ool_powf(float x, float y) { return powf(x, y); }
static __device__ __noinline__ float ool_erfcf(float x) { return erfcf(x); }
static __device__ __noinline__ double ool_log(double x) { return ::log(x); }

template <typename real> struct Num;
template <> struct Num<float> {
  static __device__ __forceinline__ float log(float x) { return ool_logf(x); }
  static __device__ __forceinline__ float exp(float x) { return expf(x); }
  static __device__ __forceinline__ float erf(float x) { return erff(x); }
  static __device__ __forceinline__ float sqrt(float x) { return sqrtf(x); }
  static __device__ __forceinline__ float lgamma(float x) { return lgammaf(x); }
  static __device__ __forceinline__ float pow(float x, float y) { return ool_powf(x, y); }
  static __device__ __forceinline__ float log1p(float x) { return ool_log1pf(x); }
  static __device__ __forceinline__ float log1p_inl(float x) { return log1pf(x); }
  static __device__ __forceinline__ float fmax(float a, float b) { return fmaxf(a, b); }
  static __device__ __forceinline__ float fabs(float a) { return fabsf(a); }
  static __device__ __forceinline__ float fmin(float a, float b) { return fminf(a, b); }
  static __device__ __forceinline__ float rcp(float x) { return rcp_ftz(x); }  // MUFU.RCP, ~1 ulp
  // 2-ulp division (MUFU.RCP + FMUL) for quantities whose own rounding already dominates
  static __device__ __forceinline__ float div(float a, float b) { return a * rcp_ftz(b); }
  // 3-ulp log (MUFU.LG2 + FMUL): only where the value is multiplied by O(1) factors
  static __device__ __forceinline__ float flog(float x) { return log_ftz(x); }
};
template <> struct Num<double> {
  static __device__ __forceinline__ double log(double x) { return ool_log(x); }
  static __device__ __forceinline__ double exp(double x) { return ::exp(x); }
  static __device__ __forceinline__ double erf(double x) { return ::erf(x); }
  static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
  static __device__ __forceinline__ double lgamma(double x) { return ::lgamma(x); }
  static __device__ __forceinline__ double pow(double x, double y) { return ::pow(x, y); }
  static __device__ __forceinline__ double log1p(double x) { return ::log1p(x); }
  static __device__ __forceinline__ double log1p_inl(double x) { return ::log1p(x); }
  static __device__ __forceinline__ double fmax(double a, double b) { return ::fmax(a, b); }
  static __device__ __forceinline__ double fabs(double a) { return ::fabs(a); }
  static __device__ __forceinline__ double fmin(double a, double b) { return ::fmin(a, b); }
  static __device__ __forceinline__ double rcp(double x) { return 1.0 / x; }
  static __device__ __forceinline__ double div(double a, double b) { return a / b; }
  static __device__ __forceinline__ double flog(double x) { return ::log(x); }
};

// ---- Gamma-function corrections to the Stirling main part, z > 0 ---------------------------------
// gamma_corr(z) returns
//   cv = lgamma(z)  - [(z - 1/2) ln z - z + ln(2 pi)/2]      (Binet's function)
//   dl = digamma(z) - ln z
//   iz = 1 / z                                                (a by-product every caller needs)
// The Dirichlet-Multinomial row is assembled from these in "KL form" (bean_row.cuh): every large
// z ln z product cancels ANALYTICALLY and only logs of near-1 ratios remain, so float keeps ~1e-6
// absolute accuracy on a row whose individual lgamma terms are O(1e3..1e4) (a float lgamma(300) alone
// is already off by 1e-4, which is the noise floor of the reference's own fp32 torch.lgamma path).
//
// float: Binet's function is exactly odd in w = 1/z (mu(z) = 2 int_0^inf atan(t w) / (e^{2 pi t} - 1) dt) and
// dl + w/2 is w^2 times an even function, so on z >= 1
//   cv = w Q(w^2),   dl = -w/2 - w^2 R(w^2)
// with degree-6 polynomials fitted on w^2 in [0, 1] (tools/fit_gamma_corr.py: 1.2e-8 / 4.2e-8 absolute in float
// arithmetic).  ONE uniform path -- 1 MUFU + 17 FP32 instructions -- replaces round 1's 4-term asymptotic series
// (z >= 4) / 4-step product recurrence (z < 4, 3 MUFU.RCP + 2 MUFU.LG2 + ~40 FP32), whose two branches nearly every
// warp executed one after the other.  z < 1 (concentrations of low-depth guides) takes one recurrence step first:
//   cv(z) = cv(z+1) + (z + 1/2) ln(1 + 1/z) - 1,   dl(z) = dl(z+1) + ln(1 + 1/z) - 1/z.
__device__ __forceinline__ void gamma_corr(float z, float& cv, float& dl, float& iz) {
  const bool small = z < 1.0f;
  const float zs = small ? z + 1.0f : z;
  const float w = rcp_ftz(zs);
  const float s = w * w;
  float q = -4.973261975e-05f, r = 3.128883582e-04f;
  r = fmaf(r, s, -1.310639309e-03f);
  q = fmaf(q, s, 2.012484825e-04f);   r = fmaf(r, s, 2.468633250e-03f);
  q = fmaf(q, s, -4.087322828e-04f);  r = fmaf(r, s, -3.093881036e-03f);
  q = fmaf(q, s, 7.606665913e-04f);   r = fmaf(r, s, 3.831227344e-03f);
  q = fmaf(q, s, -2.775296125e-03f);  r = fmaf(r, s, -8.325798381e-03f);
  q = fmaf(q, s, 8.333329976e-02f);   r = fmaf(r, s, 8.333325842e-02f);
  cv = w * q;
  dl = fmaf(-s, r, -0.5f * w);
  iz = w;
  if (small) {
    iz = rcp_ftz(z);
    const float ls = log_ftz(zs * iz);  // ln(1 + 1/z) >= ln 2: the MUFU log's absolute error is relative here
    cv += fmaf(z + 0.5f, ls, -1.0f);
    dl += ls - iz;
  }
}
__device__ __forceinline__ void gamma_corr(float z, float& cv, float& dl) {
  float iz;
  gamma_corr(z, cv, dl, iz);
}

// log1p(y) for the ratio arguments of the KL-form row, y > -1.  1 + y in [0.4, 2.5] (every bin whose posterior and prior
// fractions are within a factor 2.5 of each other -- all but outlier bins):
//   log1p(y) = 2 atanh(s) = 2 s + s^3 P(s^2),  s = y / (2 + y),  |s| <= 3/7,
// P of degree 4 (tools/fit_log1p_ratio.py: 8.8e-9 truncation, 1.6e-7 in float arithmetic = the rounding of the division):
// 1 MUFU + 10 FP32 instructions against ~26 for log1pf.  The argument itself carries ~3 ulp (a product of two MUFU
// reciprocals), so nothing is lost against log1pf.  Outside that range: MUFU lg2 of the rounded 1 + y plus the
// first-order term of the rounding residue; |log| >= ln 2.5 there, so lg2's 2^-22 ABSOLUTE error is ~2e-7 relative.
__device__ __forceinline__ bool log1p_ratio_in_range(float y) { return y > -0.6f && y < 1.5f; }
__device__ __forceinline__ float log1p_ratio_series(float y) {
  const float d = 2.0f + y;
  const float s = y * rcp_ftz(d);
  const float t = s * s;
  float p = 2.757020617e-01f;
  p = fmaf(p, t, 2.058080059e-01f);
  p = fmaf(p, t, 2.868322504e-01f);
  p = fmaf(p, t, 3.999738930e-01f);
  p = fmaf(p, t, 6.666667629e-01f);
  return fmaf(s * t, p, s + s);
}
// y = ratio - 1 where the caller also knows `ratio` as a PRODUCT of positive factors (no cancellation): outside the series'
// range the log of that product is taken directly -- exact also where 1 + y would round to 0 (y within 3e-8 of -1: a bin whose
// concentration is clamped at 1e-5 inside a row of total concentration > 300).
__device__ __forceinline__ float log1p_ratio(float y, float ratio) {
  return log1p_ratio_in_range(y) ? log1p_ratio_series(y) : log_ftz(ratio);
}

// ---- the same two functions on PAIRS, through Blackwell's packed FP32 instructions ---------------------------------------
// sm_100 has FFMA2 / FMUL2 / FADD2 (PTX fma.rn.f32x2 ...): one issue slot, two IEEE-rounded FP32 operations on a 64-bit
// register pair.  The SVI guide kernel is bound by instruction ISSUE (profiles/), and its row maths comes in natural
// pairs -- gamma_corr of (a_b, x_b + a_b) and of (A, N + A), the two log1p of a bin -- so each pair's Horner chains run
// as one chain of packed instructions.  Results are bit-identical to the scalar functions above (same operations, same
// rounding), which is what the CPU-side emulation in tests/ checks them against.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{.reg .b64 ra, rb, rc, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\t"
      "mov.b64 {%0, %1}, rd;}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  float2 d;
  asm("{.reg .b64 ra, rb, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "mul.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 d;
  asm("{.reg .b64 ra, rb, rd;\n\t"
      "mov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t"
      "add.rn.f32x2 rd, ra, rb;\n\t"
      "mov.b64 {%0, %1}, rd;}"
      : "=f"(d.x), "=f"(d.y) : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return d;
}
__device__ __forceinline__ float2 splat2(float c) { return make_float2(c, c); }

// (cv, dl, 1/z) of z.x and z.y
__device__ __forceinline__ void gamma_corr2(float2 z, float2& cv, float2& dl, float2& iz) {
  // z + [z < 1] as a float (FSET.BF) and ONE packed add, instead of add + compare + select per component
  const float bx = z.x < 1.0f ? 1.0f : 0.0f, by = z.y < 1.0f ? 1.0f : 0.0f;
  const float2 zs = add2(z, make_float2(bx, by));
  const bool sx = bx != 0.0f, sy = by != 0.0f;
  const float2 w = make_float2(rcp_ftz(zs.x), rcp_ftz(zs.y));
  const float2 s = mul2(w, w);
  float2 q = splat2(-4.973261975e-05f), r = splat2(3.128883582e-04f);
  r = fma2(r, s, splat2(-1.310639309e-03f));
  q = fma2(q, s, splat2(2.012484825e-04f));   r = fma2(r, s, splat2(2.468633250e-03f));
  q = fma2(q, s, splat2(-4.087322828e-04f));  r = fma2(r, s, splat2(-3.093881036e-03f));
  q = fma2(q, s, splat2(7.606665913e-04f));   r = fma2(r, s, splat2(3.831227344e-03f));
  q = fma2(q, s, splat2(-2.775296125e-03f));  r = fma2(r, s, splat2(-8.325798381e-03f));
  q = fma2(q, s, splat2(8.333329976e-02f));   r = fma2(r, s, splat2(8.333325842e-02f));
  cv = mul2(w, q);
  dl = fma2(make_float2(-s.x, -s.y), r, mul2(w, splat2(-0.5f)));
  iz = w;
  if (sx | sy) {  // one recurrence step for arguments below 1 (see gamma_corr)
    if (sx) {
      iz.x = rcp_ftz(z.x);
      const float ls = log_ftz(zs.x * iz.x);
      cv.x += fmaf(z.x + 0.5f, ls, -1.0f);
      dl.x += ls - iz.x;
    }
    if (sy) {
      iz.y = rcp_ftz(z.y);
      const float ls = log_ftz(zs.y * iz.y);
      cv.y += fmaf(z.y + 0.5f, ls, -1.0f);
      dl.y += ls - iz.y;
    }
  }
}

// both components inside the series' range (-0.6, 1.5)  <=>  max |y - 0.45| < 1.05: one packed add, one max of absolute
// values, one compare
__device__ __forceinline__ bool log1p_ratio_in_range2(float2 y) {
  const float2 d = add2(y, splat2(-0.45f));
  return fmaxf(fabsf(d.x), fabsf(d.y)) < 1.05f;
}

// series of (log1p(y.x), log1p(y.y)); the caller replaces out-of-range components by the log of the ratio itself
__device__ __forceinline__ float2 log1p_ratio_series2(float2 y) {
  const float2 d = add2(y, splat2(2.0f));
  const float2 s = mul2(y, make_float2(rcp_ftz(d.x), rcp_ftz(d.y)));
  const float2 t = mul2(s, s);
  float2 p = splat2(2.757020617e-01f);
  p = fma2(p, t, splat2(2.058080059e-01f));
  p = fma2(p, t, splat2(2.868322504e-01f));
  p = fma2(p, t, splat2(3.999738930e-01f));
  p = fma2(p, t, splat2(6.666667629e-01f));
  return fma2(mul2(s, t), p, add2(s, s));
}

__device__ __forceinline__ double digamma_f64(double z) {
  // Cephes psi for z > 0 -- recurrence up to 10, then the asymptotic series with 7 Bernoulli terms -- summed IN THE ORDER
  // torch's CPU digamma sums it (the negative recurrence terms first, then + log - 1/2x - series, left to right).  The order is
  // part of fp64 parity: for the ~1e-7 concentrations of non-existent tiling alleles psi is ~ -1e7 (ulp 1.9e-9) and the
  // reference's pathwise Dirichlet derivative forms psi(a) + 1/a from it (model.py:937-938 through torch._dirichlet_grad), so
  // a differently ordered -- even a more accurate -- sum moves alpha_pi's gradient by ~2e-9.
  double result = 0.0, x = z;
  // bounded: a concentration is > 0 (at most 10 terms), but -inf or a huge negative argument would never reach 10
  for (int k = 0; x < 10.0 && k < 64; ++k) {
    result -= 1.0 / x;
    x += 1.0;
  }
  if (x == 10.0) return result + 2.25175258906672110764;
  const double r2 = 1.0 / (x * x);
  double poly = 1.0 / 12;
  poly = poly * r2 + (-691.0 / 32760);
  poly = poly * r2 + (1.0 / 132);
  poly = poly * r2 + (-1.0 / 240);
  poly = poly * r2 + (1.0 / 252);
  poly = poly * r2 + (-1.0 / 120);
  poly = poly * r2 + (1.0 / 12);
  return result + ::log(x) - (0.5 / x) - r2 * poly;
}

__device__ __forceinline__ void gamma_corr(double z, double& cv, double& dl) {
  const double lz = ::log(z);
  cv = ::lgamma(z) - ((z - 0.5) * lz - z + 0.91893853320467274178);
  dl = digamma_f64(z) - lz;
}
__device__ __forceinline__ void gamma_corr(double z, double& cv, double& dl, double& iz) {
  gamma_corr(z, cv, dl);
  iz = 1.0 / z;
}
__device__ __forceinline__ double log1p_ratio(double y, double /*ratio*/) { return ::log1p(y); }

// full lgamma / digamma of one argument (off the hot row loop: Dirichlet normalisers).  The out-of-line body returns its
// two results BY VALUE, in registers: with reference parameters (stack slots in the caller's frame) the float build of
// surv_guide_kernel was observed on B200 to hand the first call's digamma slot the lgamma of the same call once two more calls
// were added to the kernel (psi of the abundance site): nvcc 12.9, sm_100a, profiles/README.md "aliasing of out-parameters".
template <typename real> struct LgDg { real lg, dg; };
template <typename real>
__device__ __noinline__ LgDg<real> lgamma_digamma_value(real z) {
  real cv, dl;
  gamma_corr(z, cv, dl);
  const real lz = Num<real>::log(z);
  LgDg<real> out;
  out.lg = (z - real(0.5)) * lz - z + real(0.91893853320467274178) + cv;
  out.dg = lz + dl;
  return out;
}
template <typename real>
__device__ __forceinline__ void lgamma_digamma(real z, real& lg, real& dg) {
  const LgDg<real> v = lgamma_digamma_value(z);
  lg = v.lg;
  dg = v.dg;
}

// ---- Normal CDF pieces ----------------------------------------------------------------------------
template <typename real>
__device__ __forceinline__ real std_normal_pdf(real z) {
  return real(0.39894228040143267794) * Num<real>::exp(real(-0.5) * z * z);
}

// Probability mass of one sorting bin and its derivatives w.r.t. (mu, sd).
// thr_u = +inf / thr_l = -inf encode quantile 1 / 0 (model/utils.py:48-54, :60-72).
// double: exactly the reference expression, Normal.cdf = 0.5 (1 + erf(z / sqrt 2)).
__device__ __forceinline__ void bin_prob_sorting(double thr_u, double thr_l, double mu, double sd, double& P,
                                                 double& dP_dmu, double& dP_dsd) {
  const double rs = 1.0 / sd;
  double cu = 1.0, fu = 0.0, zfu = 0.0, cl = 0.0, fl = 0.0, zfl = 0.0;
  if (!isinf(thr_u)) {
    const double z = (thr_u - mu) * rs;
    cu = 0.5 * (1.0 + ::erf(z * 0.70710678118654752440));
    fu = std_normal_pdf(z);
    zfu = z * fu;
  }
  if (!isinf(thr_l)) {
    const double z = (thr_l - mu) * rs;
    cl = 0.5 * (1.0 + ::erf(z * 0.70710678118654752440));
    fl = std_normal_pdf(z);
    zfl = z * fl;
  }
  P = cu - cl;
  dP_dmu = -(fu - fl) * rs;
  dP_dsd = -(zfu - zfl) * rs;
}

// float: the same mass written with erfc on the tail side, Q(z) = erfc(z / sqrt 2) / 2, so that a bin far
// in a tail keeps its RELATIVE accuracy (0.5 (1 + erf) in float loses it below ~1e-3 and that error is
// amplified by a0 / sum(p) downstream).
static __device__ __noinline__ void bin_prob_sorting(float thr_u, float thr_l, float mu, float sd, float& P,
                                                 float& dP_dmu, float& dP_dsd) {
  const float rs = 1.0f / sd;
  const bool hu = !isinf(thr_u), hl = !isinf(thr_l);
  const float zu = hu ? (thr_u - mu) * rs : INFINITY;
  const float zl = hl ? (thr_l - mu) * rs : -INFINITY;
  const float k = 0.70710678118654752440f;
  if (zl > 0.0f)
    P = 0.5f * (ool_erfcf(zl * k) - ool_erfcf(zu * k));
  else
    P = 0.5f * (ool_erfcf(-zu * k) - ool_erfcf(-zl * k));
  const float fu = hu ? std_normal_pdf(zu) : 0.0f, fl = hl ? std_normal_pdf(zl) : 0.0f;
  const float zfu = hu ? zu * fu : 0.0f, zfl = hl ? zl * fl : 0.0f;
  dP_dmu = -(fu - fl) * rs;
  dP_dsd = -(zfu - zfl) * rs;
}

// The same split in two: the mass alone (prologue of the SVI guide kernel) and its (mu, sd) derivatives alone (epilogue).
__device__ __forceinline__ double bin_mass_sorting(double thr_u, double thr_l, double mu, double sd) {
  double P, a, b;
  bin_prob_sorting(thr_u, thr_l, mu, sd, P, a, b);
  return P;
}
static __device__ __noinline__ float bin_mass_sorting(float thr_u, float thr_l, float mu, float sd) {
  const float rs = 1.0f / sd;
  const float zu = !isinf(thr_u) ? (thr_u - mu) * rs : INFINITY;
  const float zl = !isinf(thr_l) ? (thr_l - mu) * rs : -INFINITY;
  const float k = 0.70710678118654752440f;
  if (zl > 0.0f) return 0.5f * (ool_erfcf(zl * k) - ool_erfcf(zu * k));
  return 0.5f * (ool_erfcf(-zu * k) - ool_erfcf(-zl * k));
}
template <typename real>
__device__ __forceinline__ void bin_mass_grad_sorting(real thr_u, real thr_l, real mu, real sd, real& dP_dmu, real& dP_dsd) {
  const real rs = real(1) / sd;
  const bool hu = !isinf(thr_u), hl = !isinf(thr_l);
  const real zu = hu ? (thr_u - mu) * rs : real(0), zl = hl ? (thr_l - mu) * rs : real(0);
  const real fu = hu ? std_normal_pdf(zu) : real(0), fl = hl ? std_normal_pdf(zl) : real(0);
  dP_dmu = -(fu - fl) * rs;
  dP_dsd = -(zu * fu - zl * fl) * rs;
}

// Bin masses of consecutive sorting bins.  float: every finite threshold is turned into (z, tail mass erfc(|z| / sqrt 2) / 2)
// ONCE -- adjacent bins share a threshold (the upper quantile of one is the lower quantile of the next), infinite ones need no
// erfc at all -- and a mass is a difference of tail masses on the side where both are small (relative accuracy in the tails):
// 4 erfc calls per guide instead of 8 for the usual four bins.  double: the reference expression, bin by bin.
template <typename real> struct BinMasses;
template <> struct BinMasses<float> {
  float mu, rs, z_prev, c_prev;
  __device__ __forceinline__ BinMasses(float mu_, float sd) : mu(mu_), rs(1.0f / sd), z_prev(0.0f), c_prev(0.0f) {}
  __device__ __forceinline__ void tail(float thr, float& z, float& c) const {
    if (isinf(thr)) {
      z = thr;
      c = 0.0f;
    } else {
      z = (thr - mu) * rs;
      c = 0.5f * ool_erfcf(fabsf(z) * 0.70710678118654752440f);
    }
  }
  __device__ __forceinline__ float next(float thr_u, float thr_l, bool shares_lower) {
    float zl, cl, zu, cu;
    if (shares_lower) {
      zl = z_prev;
      cl = c_prev;
    } else {
      tail(thr_l, zl, cl);
    }
    tail(thr_u, zu, cu);
    z_prev = zu;
    c_prev = cu;
    if (zl > 0.0f) return cl - cu;
    if (zu < 0.0f) return cu - cl;
    return 1.0f - cl - cu;
  }
};
template <> struct BinMasses<double> {
  double mu, sd;
  __device__ __forceinline__ BinMasses(double mu_, double sd_) : mu(mu_), sd(sd_) {}
  __device__ __forceinline__ double next(double thr_u, double thr_l, bool) { return bin_mass_sorting(thr_u, thr_l, mu, sd); }
};

// log of a probability c in (0, 1]: series on c - 1 (exact subtraction) near 1, MUFU log below 0.4 (|log| > 0.9 there, so its
// absolute error is relative); ~12 instructions against ~45 through the out-of-line logf
__device__ __forceinline__ float log_unit(float c) { return c > 0.4f ? log1p_ratio_series(c - 1.0f) : log_ftz(c); }
__device__ __forceinline__ double log_unit(double c) { return ::log(c); }
// log of any positive float, inline: the series of log1p_ratio around 1, the MUFU log elsewhere (absolute error 2^-22 ln 2 of
// |log| >= 0.9: <= 2e-7 relative)
__device__ __forceinline__ float log_pos(float x) { return (x > 0.4f && x < 2.5f) ? log1p_ratio_series(x - 1.0f) : log_ftz(x); }
__device__ __forceinline__ double log_pos(double x) { return ::log(x); }

// ---- block reduction of a double (deterministic order) ------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// all threads must call; result valid in thread 0.  blockDim.x <= 1024.
__device__ __forceinline__ double block_sum(double v, double* smem32) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  v = warp_sum(v);
  if (lane == 0) smem32[wid] = v;
  __syncthreads();
  double r = 0.0;
  if (wid == 0) {
    const int nw = (blockDim.x + 31) >> 5;
    r = lane < nw ? smem32[lane] : 0.0;
    r = warp_sum(r);
  }
  __syncthreads();
  return r;
}

}  // namespace bean
