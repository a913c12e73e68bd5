// kidmp_fastmath.h - table-driven f64 exp and log for the column kernels (host + device).
//
// Half of the dynamic instructions of the column-physics kernel were CUDA's generic f64 log/exp
// (profiles/r01): ~40-50 instructions each with no table.  These versions use the classic
// reduce-to-a-table-node scheme (as in glibc / ARM optimized-routines; restated here from the
// published method, not copied): 128-entry tables, degree-5 / degree-7 polynomials on |r| < 2^-7,
// ~16 and ~24 instructions.  Accuracy (tests/test_device_math.py, against long double / mpmath):
//   exp   < 1 ulp of f64 for |x| < 704;
//   log   < 1.5 ulp where |log x| > 0.1 (1.42 measured, 1.10 below |log x| = 700); near 1 the error is
//         absolute, < 1.5e-17 where |log x| <= 0.1 (up to ~1e4 ulps of a result next to 0);
//   exp(y*log(x))  < 3 (1 + |y log x|) ulp, plus |y| * 1.5e-17 relative where |log x| <= 0.1.
// They are only ever used under an f32 rounding or inside f64 rates that are narrowed to f32
// tendencies, so this is far inside the parity budget (DESIGN.md section 4).
//
// Arguments outside the fast range (x <= 0, inf, nan, subnormal for log; |x| >= 704 or nan for exp)
// take the library function.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define KFM_HD __host__ __device__ __forceinline__
#else
#define KFM_HD inline
#endif

namespace kidmp {

enum { KFM_N = 128 };
struct LogNode { double invc, logc; };

KFM_HD int kfm_hi(double x) {
#if defined(__CUDA_ARCH__)
  return __double2hiint(x);
#else
  int64_t b; memcpy(&b, &x, 8); return (int)(b >> 32);
#endif
}
KFM_HD int kfm_lo(double x) {
#if defined(__CUDA_ARCH__)
  return __double2loint(x);
#else
  int64_t b; memcpy(&b, &x, 8); return (int)(b & 0xffffffff);
#endif
}
KFM_HD double kfm_make(int hi, int lo) {
#if defined(__CUDA_ARCH__)
  return __hiloint2double(hi, lo);
#else
  int64_t b = ((int64_t)hi << 32) | (uint32_t)lo; double x; memcpy(&x, &b, 8); return x;
#endif
}

// exp(x) = 2^(k/128) * exp(r),  k = round(x*128/ln2),  r = x - k*ln2/128, |r| <= ln2/256
KFM_HD double kfm_exp(double x, const double* __restrict__ tab) {
  const int hx = kfm_hi(x) & 0x7fffffff;
  if (hx >= 0x40860000) return exp(x);                        // |x| >= 704, inf, nan
  const double shift = 6755399441055744.0;                    // 1.5 * 2^52
  const double kd0 = x * 184.6649652337873 + shift;           // 128/ln2
  const int k = kfm_lo(kd0);
  const double kd = kd0 - shift;
  double r = fma(kd, -0.005415212333900854, x);               // ln2/128 high part (24 trailing zero bits: kd*hi exact)
  r = fma(kd, -1.4223718738313642e-11, r);                    // low part
  const double r2 = r * r;
  double p = fma(r, 8.3333333333333332e-03, 4.1666666666666664e-02);   // 1/120, 1/24
  const double q = fma(r, 1.6666666666666666e-01, 0.5);       // 1/6, 1/2
  p = fma(r2, p, q);
  p = fma(r2, p, r);                                          // exp(r) - 1
#if defined(__CUDA_ARCH__)
  const double t = __ldg(tab + (k & (KFM_N - 1)));
#else
  const double t = tab[k & (KFM_N - 1)];
#endif
  const double s = kfm_make(kfm_hi(t) + ((k >> 7) << 20), kfm_lo(t));   // t * 2^(k>>7), normal range guaranteed by |x| < 704
  return fma(s, p, s);
}

// log(x) = k*ln2 + log(c) + log1p(r),  z = x/2^k in [0.6875, 1.375),  r = z/c - 1
KFM_HD double kfm_log(double x, const LogNode* __restrict__ tab) {
  const int hx = kfm_hi(x);
  if ((unsigned)(hx - 0x00100000) >= 0x7fe00000u) return log(x);        // x <= 0, subnormal, inf, nan
  const int tmp = hx - 0x3fe60000;
  const int i = (tmp >> 13) & (KFM_N - 1);
  const int k = tmp >> 20;
  const double z = kfm_make(hx - (tmp & (int)0xfff00000), kfm_lo(x));
#if defined(__CUDA_ARCH__)
  const double2 nd = __ldg(reinterpret_cast<const double2*>(tab) + i);
  const double invc = nd.x, logc = nd.y;
#else
  const double invc = tab[i].invc, logc = tab[i].logc;
#endif
  const double r = fma(z, invc, -1.0);
  const double kd = (double)k;
  // log1p(r) = r - r^2/2 + r^3/3 - r^4/4 + r^5/5 - r^6/6 + r^7/7,  |r| < 2^-7.4
  double p = fma(r, 1.4285714285714285e-01, -1.6666666666666666e-01);
  p = fma(r, p, 0.2);
  p = fma(r, p, -0.25);
  p = fma(r, p, 3.3333333333333331e-01);
  p = fma(r, p, -0.5);
  const double r2 = r * r;
  const double hi = fma(kd, 6.9314718055989033e-01, logc);              // ln2 high part (low bits zero: k*hi exact)
  const double lo = fma(kd, 5.4979230187083712e-14, r);                 // ln2 low part + r
  return hi + fma(r2, p, lo);
}

// ---- host: build the tables (long double; x87 64-bit mantissa is plenty for a double table) ----------
inline void kfm_build_tables(double* exp_tab, LogNode* log_tab) {
  for (int j = 0; j < KFM_N; ++j) exp_tab[j] = (double)exp2l((long double)j / (long double)KFM_N);
  for (int i = 0; i < KFM_N; ++i) {
    const int64_t off = 0x3fe6000000000000LL;
    int64_t blo = off + ((int64_t)i << 45), bhi = off + ((int64_t)(i + 1) << 45);
    double lo, hi;
    memcpy(&lo, &blo, 8); memcpy(&hi, &bhi, 8);
    // z of node i always has the exponent of `lo`'s binade after the reduction; the node centre:
    const long double c = ((long double)lo + (long double)hi) * 0.5L;
    const double invc = (double)(1.0L / c);
    log_tab[i].invc = invc;
    log_tab[i].logc = (double)(-logl((long double)invc));      // log of the centre actually used (1/invc)
  }
}

}  // namespace kidmp
