// kidmp_math.cuh - arithmetic helpers of the column kernels.
//
// Parity contract (DESIGN.md "Arithmetic"): the reference (M: = module_mp_thompson09n.f90) mixes
// default REAL (f32) and DOUBLE PRECISION (f64) and the result of many expressions steers a
// discontinuous table index or threshold.  The kernels therefore
//   * are compiled with -fmad=false, IEEE division and square root, no flush-to-zero, so every
//     + - * / sqrt rounds exactly like the Fortran expression it restates;
//   * evaluate every transcendental whose result is stored as f32 in f64 and round once, which
//     is within one f32 ulp of any faithful libm (gfortran calls glibc powf/expf/logf/log10f);
//   * keep f64 where the reference has DOUBLE PRECISION, with x**y as exp(y*log(x)) (error below
//     3 (1 + |y log x|) ulp, see kidmp_fastmath.h; invisible once the rates are narrowed to the f32
//     tendencies) and the
//     PARAMETER exponents of the scheme (mu_r = mu_g = mu_i = 0, bm_r = bm_g = bm_i = 3,
//     bv_r = bv_i = 1, M:56-111) strength-reduced to products and square roots.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include "kidmp_fastmath.h"

namespace kidmp {

// node tables of kidmp_fastmath.h, filled by kidmp_init (read-only afterwards, L1-resident)
__device__ double g_exp_tab[KFM_N];
__device__ LogNode g_log_tab[KFM_N];

// One copy of the f64 logarithm / exponential / power in the kernel image: the column kernel has ~130
// call sites and its working set must stay near the instruction cache (profiles/r01: inlining them made
// a 254 KB kernel that stalled 13 cycles per issue on instruction fetch).  The bodies are the
// table-driven algorithms of kidmp_fastmath.h with the polynomial coefficients read straight from the
// constant bank (no immediate materialisation) and, for x**y, one fused routine (one call, one
// descriptor set-up, no intermediate special-case test).
__constant__ double c_fm[16] = {
    184.6649652337873,            // 0  128/ln2
    6755399441055744.0,           // 1  1.5*2^52
    -0.005415212333900854,        // 2  -ln2/128 hi
    -1.4223718738313642e-11,      // 3  -ln2/128 lo
    8.3333333333333332e-03,       // 4  1/120
    4.1666666666666664e-02,       // 5  1/24
    1.6666666666666666e-01,       // 6  1/6
    1.4285714285714285e-01,       // 7  1/7
    -1.6666666666666666e-01,      // 8  -1/6
    0.2,                          // 9
    3.3333333333333331e-01,       // 10
    6.9314718055989033e-01,       // 11 ln2 hi
    5.4979230187083712e-14,       // 12 ln2 lo
    0.0, 0.0, 0.0};

__device__ __forceinline__ double fm_exp_core(double x) {          // |x| < 704
  const double kd0 = x * c_fm[0] + c_fm[1];
  const int k = __double2loint(kd0);
  const double kd = kd0 - c_fm[1];
  double r = fma(kd, c_fm[2], x);
  r = fma(kd, c_fm[3], r);
  const double r2 = r * r;
  double p = fma(r, c_fm[4], c_fm[5]);
  const double q = fma(r, c_fm[6], 0.5);
  p = fma(r2, p, q);
  p = fma(r2, p, r);
  const double t = __ldg(g_exp_tab + (k & (KFM_N - 1)));
  const double s = __hiloint2double(__double2hiint(t) + ((k >> 7) << 20), __double2loint(t));
  return fma(s, p, s);
}
__device__ __forceinline__ double fm_log_core(double x) {          // x positive, normal, finite
  const int hx = __double2hiint(x);
  const int tmp = hx - 0x3fe60000;
  const int i = (tmp >> 13) & (KFM_N - 1);
  const double z = __hiloint2double(hx - (tmp & (int)0xfff00000), __double2loint(x));
  const double2 nd = __ldg(reinterpret_cast<const double2*>(g_log_tab) + i);
  const double r = fma(z, nd.x, -1.0);
  const double kd = (double)(tmp >> 20);
  double p = fma(r, c_fm[7], c_fm[8]);
  p = fma(r, p, c_fm[9]);
  p = fma(r, p, -0.25);
  p = fma(r, p, c_fm[10]);
  p = fma(r, p, -0.5);
  const double hi = fma(kd, c_fm[11], nd.y);
  const double lo = fma(kd, c_fm[12], r);
  return hi + fma(r * r, p, lo);
}
__device__ __forceinline__ bool fm_log_fast(double x) { return (unsigned)(__double2hiint(x) - 0x00100000) < 0x7fe00000u; }
__device__ __forceinline__ bool fm_exp_fast(double x) { return (__double2hiint(x) & 0x7fffffff) < 0x40860000; }

#ifndef KIDMP_MATH_FN
#define KIDMP_MATH_FN __device__ __noinline__
#endif
#ifndef KIDMP_SAT_FN
#define KIDMP_SAT_FN __device__ __forceinline__      // measured: the two saturation polynomials are better in line (-1.4 %)
#endif
KIDMP_MATH_FN double dlog(double x) { return fm_log_fast(x) ? fm_log_core(x) : log(x); }
KIDMP_MATH_FN double dexp(double x) { return fm_exp_fast(x) ? fm_exp_core(x) : exp(x); }
// x**y = exp(y*log(x)) for x > 0 (x = 0 gives 0 for y > 0, NaN propagates), f64
KIDMP_MATH_FN double dpow(double x, double y) {
  if (fm_log_fast(x)) {
    const double e = y * fm_log_core(x);
    if (fm_exp_fast(e)) return fm_exp_core(e);
    return exp(e);
  }
  // x = 0 (a rate or a content that is exactly zero) is the one special base the step meets in numbers: log(0) = -inf,
  // so exp(y * log(0)) is 0 for y > 0, +inf for y < 0 and NaN for y = 0 - without the two library calls
  if (x == 0.0) return y > 0.0 ? 0.0 : (y < 0.0 ? __longlong_as_double(0x7ff0000000000000LL) : __longlong_as_double(0x7ff8000000000000LL));
  return exp(y * log(x));
}
__device__ __forceinline__ double pow_d(double x, double y) { return dpow(x, y); }
#ifdef KIDMP_NATIVE_F32
// EXPERIMENT ONLY (tools/variants.py "native32", never the shipped build): the f32 transcendentals on the special-function
// unit (ex2 / lg2, ~2 ulp) instead of rule 2 of DESIGN.md section 4 - measures what bit-exactness costs and how many cells flip.
__device__ __forceinline__ float pow_f(float x, float y) { return x == 0.f ? (y > 0.f ? 0.f : __powf(x, y)) : exp2f(y * __log2f(x)); }
__device__ __forceinline__ float exp_f(float x) { return __expf(x); }
__device__ __forceinline__ float log10_f(float x) { return __log10f(x); }
__device__ __forceinline__ float pow10_f(float y) { return exp2f(y * 3.3219280948873623f); }
#else
// f32 result: REAL ** REAL of the reference (a libm powf call under gfortran)
__device__ __forceinline__ float pow_f(float x, float y) { return (float)dpow((double)x, (double)y); }
__device__ __forceinline__ float exp_f(float x) { return (float)dexp((double)x); }
__device__ __forceinline__ float log10_f(float x) { return (float)(dlog((double)x) * 0.43429448190325182765); }
// 10.**y with REAL y (M:1560, M:1646, M:2242 ...)
__device__ __forceinline__ float pow10_f(float y) { return (float)dexp((double)y * 2.302585092994046); }
#endif
__device__ __forceinline__ float cube_f(float x) { double d = x; return (float)(d * d * d); }   // x**bm_r etc.
__device__ __forceinline__ double cube_d(double x) { return x * x * x; }
__device__ __forceinline__ double sq_d(double x) { return x * x; }

__device__ __forceinline__ int nint_f(float x) { return (int)lroundf(x); }     // NINT: half away from zero
__device__ __forceinline__ int nint_d(double x) { return (int)lround(x); }

// RSLF / RSIF, M:4656-4717 (Flatau et al. polynomials, Horner form, f32)
KIDMP_SAT_FN float rslf(float P, float T) {
  const float C0 = .611583699E03f, C1 = .444606896E02f, C2 = .143177157E01f, C3 = .264224321E-1f,
              C4 = .299291081E-3f, C5 = .203154182E-5f, C6 = .702620698E-8f, C7 = .379534310E-11f,
              C8 = -.321582393E-13f;
  float X = fmaxf(-80.f, T - 273.16f);
  float ESL = C0 + X * (C1 + X * (C2 + X * (C3 + X * (C4 + X * (C5 + X * (C6 + X * (C7 + X * C8)))))));
  ESL = fminf(ESL, P * 0.15f);
  return .622f * ESL / (P - ESL);
}
KIDMP_SAT_FN float rsif(float P, float T) {
  const float C0 = .609868993E03f, C1 = .499320233E02f, C2 = .184672631E01f, C3 = .402737184E-1f,
              C4 = .565392987E-3f, C5 = .521693933E-5f, C6 = .307839583E-7f, C7 = .105785160E-9f,
              C8 = .161444444E-12f;
  float X = fmaxf(-80.f, T - 273.16f);
  float ESI = C0 + X * (C1 + X * (C2 + X * (C3 + X * (C4 + X * (C5 + X * (C6 + X * (C7 + X * C8)))))));
  ESI = fminf(ESI, P * 0.15f);
  return .622f * ESI / (P - ESI);
}

}  // namespace kidmp
