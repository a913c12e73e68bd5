// kidmp_column.cuh - the column-shaped parts of the Thompson step on the device, one thread per column.
//
// Replaces the body of `do i = 1, nx` around `call mp_thompson` (I:54-246) together with kidmp_cells.cuh, which
// holds the physics of one cell (S1..S13 of M:1156-3688).  Data layout: every field is [nz][ld] f32 (columns
// fastest), so the 32 lanes of a warp read 128 contiguous bytes per level.
//
// Kernels of this file (DESIGN.md section 3):
//   k_classify     one bottom-up read of the ten fields decides `no_micro` (M:1396-1521, the early RETURN
//                  at M:1540); clear-sky columns only get back the species <= R1 that the reference
//                  zeroes in the caller's arrays (M:1412-1489) and are done.  Every cell gets its class byte
//                  (which species it holds, whether it is supersaturated, which cell kernel takes it).
//   k_list_scan /  the ballots of the cloudy lanes become a compacted work list in column order.
//   k_list_fill
//   finish_level   the last sedimentation sub-step of a level + S15 + S16 (used by k_finish, kidmp_cells.cuh)
//   k_diag_columns the eight domain sums in column order (bitwise reproducible), k_diag_reduce adds the blocks.
#pragma once
#include "kidmp_internal.h"
#include "kidmp_math.cuh"

namespace kidmp {

// The f64 logarithm / exponential / power stay out of line (kidmp_math.cuh): ~130 call sites, and in line they made a
// kernel whose instruction fetch was the limit (profiles/r01; still 6 % slower in line under the lockstep barriers).
// The small helpers below are in line again since the lockstep blocks share their instruction-cache lines: measured
// 2 % faster than out of line (a call costs two branch latencies on a path that is latency-bound).
#ifndef KIDMP_HELPER
#define KIDMP_HELPER __device__ __forceinline__
#endif

#define R1 KP_R1
#define R2 KP_R2
#define EPSF KP_EPS
#define T_0 KP_T_0
#define D0r KP_D0R
#define D0c KP_D0C
#define D0s KP_D0S
#define D0g KP_D0G

// Field et al. (2005) moment relation coefficients, M:305-312
__device__ __constant__ float c_sa[11] = {0, 5.065339f, -0.062659f, -3.032362f, 0.029469f, -0.000285f,
                                          0.31255f, 0.000204f, 0.003199f, 0.0f, -0.015952f};
__device__ __constant__ float c_sb[11] = {0, 0.476221f, -0.015896f, 0.165977f, 0.007468f, -0.000141f,
                                          0.060366f, 0.000079f, 0.000594f, 0.0f, -0.003577f};

// loga_/b_ for moment order c at tc0, M:1590-1599 (term order kept)
__device__ __forceinline__ void field_ab(float tc0, float c, float& loga_, float& b_) {
  const float* sa = c_sa; const float* sb = c_sb;
  loga_ = sa[1] + sa[2] * tc0 + sa[3] * c + sa[4] * tc0 * c + sa[5] * tc0 * tc0 + sa[6] * c * c
          + sa[7] * tc0 * tc0 * c + sa[8] * tc0 * c * c + sa[9] * tc0 * tc0 * tc0 + sa[10] * c * c * c;
  b_ = sb[1] + sb[2] * tc0 + sb[3] * c + sb[4] * tc0 * c + sb[5] * tc0 * tc0 + sb[6] * c * c
       + sb[7] * tc0 * tc0 * c + sb[8] * tc0 * c * c + sb[9] * tc0 * tc0 * tc0 + sb[10] * c * c * c;
}
KIDMP_HELPER float field_moment(float tc0, float c, float smo2) {
  float loga_, b_;
  field_ab(tc0, c, loga_, b_);
  return pow10_f(loga_) * pow_f(smo2, b_);
}

// decade-mantissa table index, M:1762-1774 (f32) / M:1824-1833 (f64 argument).  The reference
// starts its three-candidate search at NINT(log10 x); the candidate that matches does not depend
// on how that logarithm rounds (SURVEY.md appendix A), so a bit-level estimate is enough.
__device__ __forceinline__ int decade_guess(float x) {
  const int b = __float_as_int(x);
  const float l2 = (float)((b >> 23) - 127) + __int_as_float((b & 0x007fffff) | 0x3f800000) - 1.0f;
  return __float2int_rn(l2 * 0.30103f);
}
// When x / 10.**n0 is well inside [1, 10) no other candidate can match (x / 10.**(n0-1) is ten times larger, x / 10.**(n0+1)
// ten times smaller, and a division is off by half an ulp at most), so the search of the reference is only walked,
// in its own order, when the quotient is within 1e-5 of a decade boundary or the guess is a decade off.
KIDMP_HELPER int decade_idx_f(const KConst& ck, float x, int n2, int ntb) {
  const int n0 = decade_guess(x);
  const float q0 = x / ck.p10[n0 + 32];
  int n = n0;
  float qn = q0;
  if (!(q0 > 1.00001f && q0 < 9.9999f)) {
    n = n0 + 1;
#pragma unroll
    for (int nn = -1; nn <= 1; ++nn) {
      const float q = x / ck.p10[n0 + nn + 32];
      if (q >= 1.0f && q < 10.0f) { n = n0 + nn; break; }
    }
    qn = x / ck.p10[n + 32];
  }
  const int idx = (int)qn + 9 * (n - n2);
  return max(1, min(idx, ntb));
}
KIDMP_HELPER int decade_idx_d(const KConst& ck, double x, int n2, int ntb) {
  const int n0 = decade_guess((float)x);
  const double q0 = x / (double)ck.p10[n0 + 32];
  int n = n0;
  double qn = q0;
  if (!(q0 > 1.00001 && q0 < 9.9999)) {
    n = n0 + 1;
#pragma unroll
    for (int nn = -1; nn <= 1; ++nn) {
      const double q = x / (double)ck.p10[n0 + nn + 32];
      if (q >= 1.0 && q < 10.0) { n = n0 + nn; break; }
    }
    qn = x / (double)ck.p10[n + 32];
  }
  const int idx = (int)qn + 9 * (n - n2);
  return max(1, min(idx, ntb));
}

// rain number from mass at a clamped median volume diameter, M:1452-1454
KIDMP_HELPER float nr_from_mvd(const KConst& ck, float rr, float mvd_r) {
  const double lamr = (double)((3.0f + 0.0f + 0.672f) / mvd_r);
  return (float)((double)(ck.crg[1] * ck.org3 * rr) * cube_d(lamr) / (double)ck.am_r);
}
// lamr = (am_r*crg(3)*org2*nr/rr)**obmr, M:1457
KIDMP_HELPER double rain_lam(const KConst& ck, float nr, float rr) {
  return (double)pow_f(ck.am_r * ck.crg[2] * ck.org2 * nr / rr, ck.obmr);
}
KIDMP_HELPER double ice_lam(const KConst& ck, float ni, float ri) {   // M:1429
  return (double)pow_f(ck.am_i * ck.cig[1] * ck.oig1 * ni / ri, ck.obmi);
}

// graupel intercept at one level given the running minimum from above, M:1639-1653.
// xslw1 = 0.01 and MAX(5.E-5, rg) = 5.E-5 (no supercooled rain above k_0, graupel content at most 5.E-5) make
// N0_exp the per-run constant `n0_lo` (evaluated once per thread by graupel_n0_lo with the same expressions);
// lam_exp, lamg, ilamg and N0_g (M:1649-1653) are only read where rg > R1 (M:1862, M:1921, M:2168, M:2254, M:3318).
__device__ __forceinline__ double graupel_n0_exp(float xslw1, float rg) {
  const float ygra1 = 4.31f + log10_f(fmaxf(5.E-5f, rg));
  const float zans1 = 3.1f + (100.f / (300.f * xslw1 * ygra1 / (10.f / xslw1 + 1.f + 0.25f * ygra1) + 30.f + 10.f * ygra1));
  const double N0_exp = (double)pow10_f(zans1);
  return fmax((double)KP_GONV_MIN, fmin(N0_exp, (double)KP_GONV_MAX));
}
KIDMP_HELPER double graupel_n0_lo() { return graupel_n0_exp(0.01f, R1); }
__global__ void k_n0_lo(double* n0_lo) { *n0_lo = graupel_n0_lo(); }      // KConst::n0_lo, evaluated once by kidmp_init
KIDMP_HELPER void graupel_n0(const KConst& ck, bool above_k0, bool L_qr, bool L_qg, float mvd_r, float rg, double n0_lo,
                             double& N0_min, double& ilamg, double& N0_g) {
  const bool slw = above_k0 && L_qr && mvd_r > 100.E-6f;
  double N0_exp = n0_lo;
  if (slw || rg > 5.E-5f) {
    float xslw1 = 0.01f;
    if (slw) xslw1 = 4.01f + log10_f(mvd_r);
    N0_exp = graupel_n0_exp(xslw1, rg);
  }
  N0_min = fmin(N0_exp, N0_min);
  N0_exp = N0_min;
  if (L_qg) {
    const double lam_exp = sqrt(sqrt(N0_exp * (double)ck.am_g * (double)ck.cgg[0] / (double)rg));   // **oge1, oge1 = 1/4
    const double lamg = lam_exp * (double)ck.lamg_fac;
    ilamg = (double)1.f / lamg;
    N0_g = N0_exp / ((double)ck.cgg[1] * lam_exp) * lamg;                                         // lamg**cge(2), cge(2) = 1
  }
}

enum { F_QV = 0, F_QC, F_QI, F_QR, F_QS, F_QG, F_NI, F_NR, F_T };

// ---- K0: classification (pass 0).  One thread per column reads the ten fields once, decides
// `no_micro` (M:1396-1521; the early RETURN at M:1540), writes back the species <= R1 that the
// reference zeroes in the caller's arrays before returning (M:1412-1489, U9), marks clear-sky columns
// in colflag and leaves the ballot of the cloudy lanes of every 32-column group for the work list.
// Every cell also gets its class byte: species present, ice supersaturation, below 0 C (k_cell_* sort the busy cells by it).
// A cell is BUSY (some process rate can be non-zero) when it holds a hydrometeor, or - vapour only - when nucleation
// or condensation can start (each rate is gated by a species flag or by ssati / ssatw, M:1676-2286, M:2780, M:2880).
// Both need ssati > 0: at or below 0 C ssatw > eps implies ssati > 0 because e_s(ice) <= e_s(liquid) for both polynomials
// over their whole range (tests/test_oracle_kat.py::test_saturation_over_ice_not_above_liquid), above 0 C the two are
// the same number.  The column test of M:1540 is the reference's (any ssati > 0).
// Light on registers: many warps per SM keep the HBM pipe full for the ~70 % of columns that need nothing else.
__device__ __forceinline__ int cell_kernel_class(unsigned sp, bool cold, bool iiwarm) {
  const bool icephase = (sp & (CLS_QI | CLS_QS | CLS_QG)) != 0;
  if (iiwarm) return icephase ? KC_FULL : KC_WARM;       // S3/S4/S6/S10 are switched off as a whole (M:1545, M:1749)
  if (!cold && !icephase) return KC_WARM;
  if (cold && !(sp & (CLS_QC | CLS_QR | CLS_QG))) return KC_ICE;
  return (sp & CLS_QR) ? KC_FULL : KC_MIXNR;
}
// Sort key of a busy cell: its five species bits and whether it is below 0 C (64 keys, kidmp_cells.cuh).
__device__ __forceinline__ unsigned cell_key(unsigned c) { return (c & 31u) | ((c >> CLS_COLD_SHIFT) & 1u) << 5; }

__global__ void __launch_bounds__(128, 8) k_classify(StepArgs a) {
  __shared__ int s_cnt[4][64];                              // busy cells of every sort key in the 32 columns of every warp
  const long col = (long)blockIdx.x * blockDim.x + threadIdx.x;
  const bool in_range = col < a.ncol;
  const int nz = a.nz;
  const long ncol = a.ncol, ld = a.ld;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  s_cnt[warp][lane] = 0; s_cnt[warp][lane + 32] = 0;
  __syncwarp();
  bool active = false;
  if (in_range) {
    const long c = col;
    const float* __restrict__ Gp = a.p + c;
    float* Gqv = a.f[F_QV] + c; float* Gqc = a.f[F_QC] + c; float* Gqi = a.f[F_QI] + c;
    float* Gqr = a.f[F_QR] + c; float* Gqs = a.f[F_QS] + c; float* Gqg = a.f[F_QG] + c;
    float* Gni = a.f[F_NI] + c; float* Gnr = a.f[F_NR] + c; float* Gt = a.f[F_T] + c;
    unsigned char* Gcls = a.cls + c;
    bool no_micro = true, graupel = false, zeroed = false;
#pragma unroll 4
    for (int k = 0; k < nz; ++k) {
      const long o = (long)k * ld;
      const float qc = Gqc[o], qi = Gqi[o], qr = Gqr[o], qs = Gqs[o], qg = Gqg[o];
      const float ni = Gni[o], nr = Gnr[o];
      const float t = Gt[o], pr = Gp[o], qv = fmaxf(1.E-10f, Gqv[o]);
      unsigned sp = 0;
      if (qc > R1) sp |= CLS_QC;
      if (qi > R1) sp |= CLS_QI;
      if (qr > R1) sp |= CLS_QR;
      if (qs > R1) sp |= CLS_QS;
      if (qg > R1) { sp |= CLS_QG; graupel = true; }
      if (in_range) {
        if (!(qc > R1) && qc != 0.0f) { Gqc[o] = 0.0f; zeroed = true; }
        if (!(qi > R1) && (qi != 0.0f || ni != 0.0f)) { Gqi[o] = 0.0f; Gni[o] = 0.0f; zeroed = true; }
        if (!(qr > R1) && (qr != 0.0f || nr != 0.0f)) { Gqr[o] = 0.0f; Gnr[o] = 0.0f; zeroed = true; }
        if (!(qs > R1) && qs != 0.0f) { Gqs[o] = 0.0f; zeroed = true; }
        if (!(qg > R1) && qg != 0.0f) { Gqg[o] = 0.0f; zeroed = true; }
      }
      const float tempc = t - 273.15f;
      unsigned c8 = sp;
      // (a screening test that skips the two divisions for clearly sub-saturated cells was measured: 8 % slower, the
      // polynomial and the divisions hide behind the loads)
      const float qvsi = (tempc <= 0.0f) ? rsif(pr, t) : rslf(pr, t);
      float ssati = qv / qvsi - 1.f;
      if (fabsf(ssati) < EPSF) ssati = 0.0f;
      if (ssati > 0.0f) {
        no_micro = false;                                     // the reference's test, M:1540
        if (!sp) {
          // Vapour only.  Without a hydrometeor two things can happen: Cooper nucleation below 0 C at ssati >= 0.25, or at ssatw >
          // eps below 253.15 K (M:2090), and condensation at ssatw > eps (M:2780: the state at tau+1 is the input when every
          // other rate is zero).  Every other rate is gated by a species flag: a cell that meets neither is idle.
          float ssatw = ssati;                                // above 0 C the two are the same number (qvsi = qvs, M:1505)
          if (tempc <= 0.0f) {
            ssatw = qv / rslf(pr, t) - 1.f;
            if (fabsf(ssatw) < EPSF) ssatw = 0.0f;
          }
          if ((t < T_0 && ssati >= 0.25f) || ssatw > EPSF) c8 |= CLS_VAP;
        }
      }
      if (sp) no_micro = false;
      if (t < T_0) c8 |= 1u << CLS_COLD_SHIFT;
      if (in_range) Gcls[(long)k * ncol] = (unsigned char)c8;
      // key histogram of the busy cells of this warp's 32 columns (k_cell_fill turns it into list positions): a shared-memory
      // reduction per busy cell, no warp-wide step in the loop - the loads of the next levels stay in flight
      if (in_range && (c8 & CLS_BUSY) != 0u) atomicAdd(&s_cnt[warp][cell_key(c8)], 1);
    }
    active = in_range && !no_micro;
    if (in_range) {
      a.colflag[col] = active ? (graupel ? 1 : 0) : (zeroed ? -2 : -1);     // -1: the step leaves this column bit for bit as it was
      if (!active) {                                 // clear-sky column: nothing left to do
        a.ppt[col] = 0.f; a.ppt[ld + col] = 0.f; a.ppt[2 * ld + col] = 0.f; a.ppt[3 * ld + col] = 0.f;   // I:55-58
      }
    }
  }
  // ballot of the cloudy lanes of this 32-column group; k_list_scan / k_list_fill turn the ballots into the
  // compacted work list IN COLUMN ORDER (neighbouring lanes of the column kernels are neighbouring columns: coalesced
  // accesses, similar branches)
  const unsigned mask = __ballot_sync(0xffffffffu, active);
  if (lane == 0 && in_range) a.work_mask[col >> 5] = mask;
  // first entry of this warp's cells inside the segment of every key (the segments are laid out by k_cell_offsets)
  __syncthreads();
  if (threadIdx.x < 64) {
    const int key = threadIdx.x;
    const int n0 = s_cnt[0][key], n1 = s_cnt[1][key], n2 = s_cnt[2][key], n3 = s_cnt[3][key];
    const int total = n0 + n1 + n2 + n3;
    if (total) {
      const int run = atomicAdd(&a.cell_hist[key], total);
      int* base = a.cell_base + (size_t)blockIdx.x * 4 * 64 + key;
      base[0] = run; base[64] = run + n0; base[128] = run + n0 + n1; base[192] = run + n0 + n1 + n2;
    }
  }
}

// exclusive prefix sum of the per-group cloudy-column counts (one block; ngroups is at most 2^19: 16 777 216 columns per launch).
// 4096 groups per round: every thread takes four neighbouring ballots (the array is padded to a multiple of four by its allocation).
__global__ void __launch_bounds__(1024) k_list_scan(const unsigned* __restrict__ mask, int ngroups, int* __restrict__ offset,
                                                    int* __restrict__ count) {
  __shared__ int s_warp[32];
  __shared__ int s_run;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) s_run = 0;
  __syncthreads();
  for (int g0 = 0; g0 < ngroups; g0 += 4096) {
    const int g = g0 + threadIdx.x * 4;
    int n[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) n[j] = g + j < ngroups ? __popc(mask[g + j]) : 0;
    const int mine = n[0] + n[1] + n[2] + n[3];
    int v = mine;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) v += u; }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
      int w = s_warp[lane];
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += u; }
      s_warp[lane] = w;
    }
    __syncthreads();
    const int run = s_run;
    const int incl = v + (warp ? s_warp[warp - 1] : 0);
    int e = run + incl - mine;
#pragma unroll
    for (int j = 0; j < 4; ++j) { if (g + j < ngroups) offset[g + j] = e; e += n[j]; }
    __syncthreads();
    if (threadIdx.x == 1023) s_run = run + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) *count = s_run;
}

__global__ void __launch_bounds__(256) k_list_fill(const unsigned* __restrict__ mask, const int* __restrict__ offset, int ngroups,
                                                   int* __restrict__ list) {
  const int g = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (g >= ngroups) return;
  const unsigned m = mask[g];
  if ((m >> lane) & 1u) list[offset[g] + __popc(m & ((1u << lane) - 1u))] = g * 32 + lane;
}

// ---- the last (or only) sedimentation sub-step of the four species at one level (M:3365-3578), the instant melting /
// freezing of cloud ice and cloud water (S15, M:3584-3606), the tendencies applied with the final clamps (S16,
// M:3623-3686), the nine output stores and the water paths of the new state.  Walked top-down: the fluxes of the level
// above come in `c`.  Used by k_finish (kidmp_cells.cuh) after the extra sub-steps.
struct SedParams {            // per column, fixed over the sweep
  float DT, odt, on_r, on_i, on_s, on_g, Nt_c;
  int top_r, top_i, top_s, top_g;   // ksed1(1..4): top sedimenting level of rain, ice, snow, graupel (M:3208)
  bool sedi, iiwarm;
};
struct SedCarry {             // carried down the column
  float sr_up, snr_up, si_up, sni_up, ss_up, sg_up;     // fluxes leaving the level above
  float ppt_r, ppt_i, ppt_s, ppt_g;
  double lwp, iwp;
};
struct HandOff {              // what S1..S13 leave for a level (SC_* order)
  float tt, qvt, qct, qit, qrt, qst, qgt, nit, nrt, nct, rr, nr, ri, ni, rs, rg, v_r, v_nr, v_i, v_ni, v_s, v_g, rho, s15;
  float nwfat, nifat;           // aerosol-aware runs only (M:2398-2408, M:2863, M:2952)
};
// AERO: is_aerosol_aware = .true.: the droplet number and the two aerosol numbers are state (a.nc, a.nwfa, a.nifa, M:3626-3647)
template <bool AERO = false>
__device__ __forceinline__ void finish_level(const KConst& ck, const StepArgs& a, const SedParams& p, SedCarry& c, const HandOff& h,
                                             int k, int nz, long g, float dzk, float t1d, float qv1d, float qc1d, float qi1d, float qr1d,
                                             float qs1d, float qg1d, float ni1d, float nr1d, float pres) {
  float tt = h.tt, qvt = h.qvt, qct = h.qct, qit = h.qit, qrt = h.qrt, qst = h.qst, qgt = h.qgt, nit = h.nit, nrt = h.nrt, nct = h.nct;
  const float rho = h.rho, s15 = h.s15, rr = h.rr, nr = h.nr, ri = h.ri, ni = h.ni, rs = h.rs, rg = h.rg;
  const float odzq = 1.f / dzk, orho = 1.f / rho;
  const float sr = h.v_r * rr, snr = h.v_nr * nr;
  const float si = p.sedi ? h.v_i * ri : 0.f, sni = p.sedi ? h.v_ni * ni : 0.f;
  const float ssn = p.sedi ? h.v_s * rs : 0.f, sg = p.sedi ? h.v_g * rg : 0.f;
  float rr_n = rr, ri_n = ri, rs_n = rs, rg_n = rg;
  if (k == nz - 1) {
    qrt = qrt - sr * odzq * p.on_r * orho;   nrt = nrt - snr * odzq * p.on_r * orho;
    rr_n = fmaxf(KP_R1, rr - sr * odzq * p.DT * p.on_r);
    qit = qit - si * odzq * p.on_i * orho;   nit = nit - sni * odzq * p.on_i * orho;
    ri_n = fmaxf(KP_R1, ri - si * odzq * p.DT * p.on_i);
    qst = qst - ssn * odzq * p.on_s * orho;  rs_n = fmaxf(KP_R1, rs - ssn * odzq * p.DT * p.on_s);
    qgt = qgt - sg * odzq * p.on_g * orho;   rg_n = fmaxf(KP_R1, rg - sg * odzq * p.DT * p.on_g);
  } else {
    if (k + 1 <= p.top_r) {
      qrt = qrt + (c.sr_up - sr) * odzq * p.on_r * orho;   nrt = nrt + (c.snr_up - snr) * odzq * p.on_r * orho;
      rr_n = fmaxf(KP_R1, rr + (c.sr_up - sr) * odzq * p.DT * p.on_r);
    }
    if (k + 1 <= p.top_i) {
      qit = qit + (c.si_up - si) * odzq * p.on_i * orho;   nit = nit + (c.sni_up - sni) * odzq * p.on_i * orho;
      ri_n = fmaxf(KP_R1, ri + (c.si_up - si) * odzq * p.DT * p.on_i);
    }
    if (k + 1 <= p.top_s) {
      qst = qst + (c.ss_up - ssn) * odzq * p.on_s * orho;  rs_n = fmaxf(KP_R1, rs + (c.ss_up - ssn) * odzq * p.DT * p.on_s);
    }
    if (k + 1 <= p.top_g) {
      qgt = qgt + (c.sg_up - sg) * odzq * p.on_g * orho;   rg_n = fmaxf(KP_R1, rg + (c.sg_up - sg) * odzq * p.DT * p.on_g);
    }
  }
  c.sr_up = sr; c.snr_up = snr; c.si_up = si; c.sni_up = sni; c.ss_up = ssn; c.sg_up = sg;
  if (k == 0) {                                         // surface precipitation of the last sub-step, M:3391-3392
    if (rr_n > KP_R1 * 10.f) c.ppt_r = c.ppt_r + sr * p.DT * p.on_r;
    if (ri_n > KP_R1 * 10.f) c.ppt_i = c.ppt_i + si * p.DT * p.on_i;
    if (rs_n > KP_R1 * 10.f) c.ppt_s = c.ppt_s + ssn * p.DT * p.on_s;
    if (rg_n > KP_R1 * 10.f) c.ppt_g = c.ppt_g + sg * p.DT * p.on_g;
  }

  // ---- S15 + S16 for this level ----------------------------------------------------------------
  float nc1d = AERO ? a.nc[g] : p.Nt_c / (0.622f * pres / (KP_R * t1d * (qv1d + 0.622f)));   // U1
  if (!(qc1d > KP_R1)) { qc1d = 0.f; nc1d = 0.f; }
  if (!(qi1d > KP_R1)) { qi1d = 0.f; ni1d = 0.f; }
  if (!(qr1d > KP_R1)) { qr1d = 0.f; nr1d = 0.f; }
  if (!(qs1d > KP_R1)) qs1d = 0.f;
  if (!(qg1d > KP_R1)) qg1d = 0.f;
  if (!p.iiwarm) {
    const float xri = fmaxf(0.0f, qi1d + qit * p.DT);
    if ((s15 > 0.f) && (xri > 0.0f)) {                  // temp > T_0
      qct = qct + xri * p.odt;
      nct = nct + ni1d * p.odt;
      qit = qit - xri * p.odt;
      nit = -ni1d * p.odt;
      tt = tt - s15 * xri * p.odt * 1.0f;
    }
    const float xrc = fmaxf(0.0f, qc1d + qct * p.DT);
    if ((s15 < 0.f) && (xrc > 0.0f)) {                  // temp < HGFR
      const float xnc = nc1d + nct * p.DT;
      qit = qit + xrc * p.odt;
      nit = nit + xnc * p.odt;
      qct = qct - xrc * p.odt;
      nct = nct - xnc * p.odt;
      tt = tt + (-s15) * xrc * p.odt * 1.0f;
    }
  }
  t1d = t1d + tt * p.DT;
  qv1d = fmaxf(1.E-10f, qv1d + qvt * p.DT);
  qc1d = qc1d + qct * p.DT;
  if (AERO) {                                  // M:3626-3647
    nc1d = fmaxf(2.f / rho, nc1d + nct * p.DT);
    a.nwfa[g] = fmaxf(11.1E6f / rho, fminf(9999.E6f / rho, (a.nwfa[g] + h.nwfat * p.DT)));
    a.nifa[g] = fmaxf(0.5E6f * 0.01f, fminf(9999.E6f / rho, (a.nifa[g] + h.nifat * p.DT)));
    if (qc1d <= KP_R1) {
      nc1d = 0.0f;
    } else {
      const int nu = min(15, nint_f(1000.E6f / (nc1d * rho)) + 2);
      double lc = (double)pow_f(ck.am_r * ck.ccg[1][nu - 1] * ck.ocg1[nu - 1] * nc1d / qc1d, ck.obmr);
      const float xD = (float)((double)(3.f + (float)nu + 1.f) / lc);
      if (xD < KP_D0C) lc = (double)(ck.cce[1][nu - 1] / KP_D0C);
      else if (xD > KP_D0R * 2.f) lc = (double)(ck.cce[1][nu - 1] / (KP_D0R * 2.f));
      nc1d = (float)fmin((double)(ck.ccg[0][nu - 1] * ck.ocg2[nu - 1] * qc1d / ck.am_r) * cube_d(lc), (double)KP_NT_C_MAX / (double)rho);
    }
    a.nc[g] = nc1d;
  }
  if (qc1d <= KP_R1) qc1d = 0.0f;              // (not aerosol aware: nc1d is not returned to the host, I:143-152, I:198-245)
  qi1d = qi1d + qit * p.DT;
  ni1d = fmaxf(KP_R2 / rho, ni1d + nit * p.DT);
  if (qi1d <= KP_R1) {
    qi1d = 0.0f; ni1d = 0.0f;
  } else {
    double lami = ice_lam(ck, ni1d, qi1d);
    const double ilami = (double)1.f / lami;
    const float xDi = (float)((double)(3.f + 0.f + 1.f) * ilami);
    if (xDi < 5.E-6f) lami = (double)(ck.cie[1] / 5.E-6f);
    else if (xDi > 300.E-6f) lami = (double)(ck.cie[1] / 300.E-6f);
    ni1d = (float)fmin((double)(ck.cig[0] * ck.oig2 * qi1d / ck.am_i) * cube_d(lami), 499.E3 / (double)rho);
  }
  qr1d = qr1d + qrt * p.DT;
  nr1d = fmaxf(KP_R2 / rho, nr1d + nrt * p.DT);
  if (qr1d <= KP_R1) {
    qr1d = 0.0f; nr1d = 0.0f;
  } else {
    const double lamr = rain_lam(ck, nr1d, qr1d);
    float mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr);
    if (mvd_r > 2.5E-3f) mvd_r = 2.5E-3f;
    else if (mvd_r < KP_D0R * 0.75f) mvd_r = KP_D0R * 0.75f;
    nr1d = nr_from_mvd(ck, qr1d, mvd_r);
  }
  qs1d = qs1d + qst * p.DT;
  if (qs1d <= KP_R1) qs1d = 0.0f;
  qg1d = qg1d + qgt * p.DT;
  if (qg1d <= KP_R1) qg1d = 0.0f;
  a.f[F_T][g] = t1d; a.f[F_QV][g] = qv1d; a.f[F_QC][g] = qc1d; a.f[F_QI][g] = qi1d; a.f[F_QR][g] = qr1d; a.f[F_QS][g] = qs1d; a.f[F_QG][g] = qg1d;
  a.f[F_NI][g] = ni1d; a.f[F_NR][g] = nr1d;
  // domain diagnostics: liquid / ice water paths of the new state
  const float rho_new = 0.622f * pres / (KP_R * t1d * (qv1d + 0.622f));
  c.lwp += (double)((qc1d + qr1d) * rho_new * dzk);
  c.iwp += (double)((qi1d + qs1d + qg1d) * rho_new * dzk);
}

// Domain sums in COLUMN order, whatever order the work list had: bitwise reproducible run to run and across
// different work-list orders.  Fixed grid: block b sums the columns [b*chunk, (b+1)*chunk) (thread-strided, then a
// tree), the per-block partials are added up by k_diag_reduce.
__global__ void __launch_bounds__(256) k_diag_columns(StepArgs a, long chunk) {
  __shared__ double s[256];
  const long c0 = (long)blockIdx.x * chunk, c1 = min(c0 + chunk, a.ncol);
  const long ncol = a.ncol, ld = a.ld;
  double v[KIDMP_NDIAG] = {0., 0., 0., 0., 0., 0., 0., 0.};
  for (long c = c0 + threadIdx.x; c < c1; c += blockDim.x) {
    v[7] += 1.0;
    if (a.colflag[c] < 0) continue;                         // clear sky: ppt = 0, no condensate
    v[0] += (double)a.ppt[c]; v[1] += (double)a.ppt[ld + c]; v[2] += (double)a.ppt[2 * ld + c]; v[3] += (double)a.ppt[3 * ld + c];
    v[4] += a.coldiag[c]; v[5] += a.coldiag[ncol + c];
    v[6] += 1.0;
  }
  for (int q = 0; q < KIDMP_NDIAG; ++q) {
    s[threadIdx.x] = v[q];
    __syncthreads();
    for (int st = 128; st > 0; st >>= 1) {
      if ((int)threadIdx.x < st) s[threadIdx.x] += s[threadIdx.x + st];
      __syncthreads();
    }
    if (threadIdx.x == 0) a.diag_partial[(size_t)blockIdx.x * KIDMP_NDIAG + q] = s[0];
    __syncthreads();
  }
}

// fixed-order reduction of the block partials into diag[8] (accumulates: kidmp_diag reads and clears)
__global__ void k_diag_reduce(const double* __restrict__ partial, int nblocks, double* __restrict__ diag) {
  __shared__ double s[256];
  const int q = blockIdx.x;
  double x = 0.0;
  for (int b = threadIdx.x; b < nblocks; b += blockDim.x) x += partial[(size_t)b * KIDMP_NDIAG + q];
  s[threadIdx.x] = x;
  __syncthreads();
  for (int st = blockDim.x >> 1; st > 0; st >>= 1) {
    if ((int)threadIdx.x < st) s[threadIdx.x] += s[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) diag[q] += s[0];
}

// mp_gt_driver after the column call of an aerosol-aware run, M:1001: nwfa1d(kts) = nwfa1d(kts) + nwfa2d(i,j)*dt_in
__global__ void k_nwfa_surface(float* __restrict__ nwfa, const float* __restrict__ nwfa2d, long ncol, float dt) {
  const long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (c < ncol) nwfa[c] = nwfa[c] + nwfa2d[c] * dt;
}

// The columns that the step changed, written straight into the caller's PINNED host arrays over PCIe (zero copy): a clear-sky
// column comes back bit for bit as it went in (the early RETURN of M:1540), so only the cloudy columns - and the rare
// clear one in which a species <= R1 was zeroed - need to travel.  One thread per column, lanes = neighbouring columns:
// runs of changed columns become full 128-byte writes.
struct HostFields { float* f[KIDMP_NFIELDS]; };
__global__ void __launch_bounds__(128) k_scatter_host(StepArgs a, HostFields hf, long hld) {
  const long col = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= a.ncol || a.colflag[col] == -1) return;
  const int nz = a.nz;
#pragma unroll 2
  for (int k = 0; k < nz; ++k) {
    const long o = (long)k * a.ld + col, ho = (long)k * hld + col;
#pragma unroll
    for (int q = 0; q < KIDMP_NFIELDS; ++q) hf.f[q][ho] = a.f[q][o];
  }
}
// The same return path of an aerosol-aware step: the nine fields, then nc, nwfa, nifa (written by finish_level of the active
// columns only, so an untouched column is unchanged in all twelve).  nwfa_row0: the surface emission (M:1001) added level 0 of
// nwfa in every column after the step, so that row goes back for the untouched columns too.
struct HostFieldsAero { float* f[KIDMP_NFIELDS + 3]; };
__global__ void __launch_bounds__(128) k_scatter_host_aero(StepArgs a, HostFieldsAero hf, long hld, int nwfa_row0) {
  const long col = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= a.ncol) return;
  if (a.colflag[col] == -1) {
    if (nwfa_row0) hf.f[KIDMP_NFIELDS + 1][col] = a.nwfa[col];
    return;
  }
  const float* const src[KIDMP_NFIELDS + 3] = {a.f[0], a.f[1], a.f[2], a.f[3], a.f[4], a.f[5], a.f[6], a.f[7], a.f[8],
                                               a.nc, a.nwfa, a.nifa};
  const int nz = a.nz;
#pragma unroll 2
  for (int k = 0; k < nz; ++k) {
    const long o = (long)k * a.ld + col, ho = (long)k * hld + col;
#pragma unroll
    for (int q = 0; q < KIDMP_NFIELDS + 3; ++q) hf.f[q][ho] = src[q][o];
  }
}

// layout conversion between KiD's (k,i) arrays [col][nz] and the device layout [nz][ncol]
__global__ void k_transpose(const float* __restrict__ src, float* __restrict__ dst, long ncol, int nz, int to_col_fastest) {
  __shared__ float tile[32][33];
  // src is [R][C] row-major, dst is [C][R]
  // blockIdx.x tiles the columns, blockIdx.y the levels
  const long R = to_col_fastest ? ncol : nz, Cn = to_col_fastest ? nz : ncol;
  const long tc = (long)blockIdx.x * 32, tk = (long)blockIdx.y * 32;
  const long r0 = to_col_fastest ? tc : tk, c0 = to_col_fastest ? tk : tc;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const long r = r0 + j, c = c0 + threadIdx.x;
    if (r < R && c < Cn) tile[j][threadIdx.x] = src[r * Cn + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const long c = c0 + j, r = r0 + threadIdx.x;
    if (r < R && c < Cn) dst[c * R + r] = tile[threadIdx.x][j];
  }
}

#undef R1
#undef R2
#undef EPSF
#undef T_0
#undef D0r
#undef D0c
#undef D0s
#undef D0g

}  // namespace kidmp
