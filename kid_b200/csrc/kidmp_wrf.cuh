// kidmp_wrf.cuh - the WRF / MPAS-shaped entry around the column step, on the device.
// Replaces mp_gt_driver (M:806-1143): 3-D (i,k,j) arrays in, theta -> T with the Exner function (M:941), per-column
// layer depths dz(i,k,j) (M:944), the column step, T -> theta (M:1022), the precipitation accumulators
// RAINNC / RAINNCV / SNOWNC / SNOWNCV / GRAUPELNC / GRAUPELNCV / SR (M:991-1003) and the effective radii of cloud
// water, cloud ice and snow (calc_effectRad, M:4834-4935; clamps M:1118-1122).
//
// A WRF array a(i,k,j) of the caller's memory box (ni_m x nk_m x nj_m, halo and spare levels included) sits at
// a[i + ni_m*(k + nk_m*j)], a 2-D one at a[i + ni_m*j].  A call steps one tile of it: tile cell (i,k,j) is memory cell
// (i0+i, k0+k, j0+j) and column i + ni*j of the step's [k][col] planes, so a row of ni floats moves as a whole and both
// sides of every copy are coalesced.  Nothing outside the tile is read or written.
//
// The is_aerosol_aware branches (M:950-956, M:999-1007, M:4875) are served by kidmp_mp_gt_driver_aero: nc, nwfa, nifa and w
// travel through k_ikj_planes, the surface emission is k_nwfa_surface, the cloud radius reads the prognostic droplet number.
// Not restated (dead in the reference): WRF_CHEM arguments, refl_10cm / calc_refl10cm (never called), and the negative-qv repair of
// M:1096-1107, which cannot trigger: mp_thompson returns qv1d = MAX(1.E-10, ...) (M:3629).
#pragma once
#include "kidmp_internal.h"
#include "kidmp_math.cuh"
#include "kidmp_column.cuh"

namespace kidmp {

// the tile of a call inside the memory box of its arrays (the host checks that it lies inside)
struct WrfBox {
  int ni, nk, nj;        // tile extents
  int i0, k0, j0;        // tile origin in the memory box
  int ni_m, nk_m;        // memory extents of i and k (the strides)
  __device__ long at(int i, int k, int j) const { return (long)(i0 + i) + (long)ni_m * ((long)(k0 + k) + (long)nk_m * (j0 + j)); }
  __device__ long at2(int i, int j) const { return (long)(i0 + i) + (long)ni_m * (j0 + j); }
  __device__ long plane(int i, int k, int j) const { return (long)k * ni * nj + (long)j * ni + i; }
};

struct WrfArgs {
  WrfBox t;
  float* a3[9];                 // qv qc qi qr qs qg ni nr th, (i,k,j), in state-field order
  const float *pii, *p3, *dz3;  // (i,k,j)
  float* f[KIDMP_NFIELDS];      // state [nk][ni*nj] of the tile
  float *p, *dz_col;            // [nk][ni*nj]
  const float* ppt;             // [4][ni*nj] rain, ice, snow, graupel of this step
  float *rainnc, *rainncv, *sr, *snownc, *snowncv, *graupelnc, *graupelncv;   // (i,j); the last four may be NULL
  float *re_cloud, *re_ice, *re_snow;   // (i,k,j), all three or none (has_reqc, has_reqi, has_reqs, M:1110)
  const float* nc_plane;                // [nk][ni*nj] prognostic droplet number of an aerosol-aware run, else NULL (nc = Nt_c, M:4875)
  const float* set_nc;                  // [ni*nj] set_Nc of every column of a per-column run (Nt_c = set_nc * 1e6f), else NULL
};

// one (i,k,j) array <-> one [k][col] plane of the step; x: i, y: k, z: j.  A 2-D (i,j) array is the box with nk = nk_m = 1.
__global__ void k_ikj_planes(float* a3, float* plane, WrfBox t, int to_planes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y, j = blockIdx.z;
  if (i >= t.ni) return;
  const long x = t.at(i, k, j), y = t.plane(i, k, j);
  if (to_planes) plane[y] = a3[x]; else a3[x] = plane[y];
}

// one thread per cell; x: i, y: k, z: j
__global__ void k_wrf_gather(WrfArgs a) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y, j = blockIdx.z;
  if (i >= a.t.ni) return;
  const long src = a.t.at(i, k, j), dst = a.t.plane(i, k, j);
#pragma unroll
  for (int q = 0; q < 8; ++q) a.f[q][dst] = a.a3[q][src];
  a.f[8][dst] = a.a3[8][src] * a.pii[src];                 // t1d = th*pii, M:941
  a.p[dst] = a.p3[src];
  a.dz_col[dst] = a.dz3[src];
}

// M:4857-4868 cloud droplet shape parameter and g_ratio
__device__ __constant__ float c_g_ratio[15] = {24, 60, 120, 210, 336, 504, 720, 990, 1320, 1716, 2184, 2730, 3360, 4080, 4896};

__global__ void k_wrf_scatter(WrfArgs a, const __grid_constant__ KConst ck) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x, k = blockIdx.y, j = blockIdx.z;
  if (i >= a.t.ni) return;
  const long dst = a.t.at(i, k, j), src = a.t.plane(i, k, j);
  const float qv1d = a.f[0][src], qc1d = a.f[1][src], qi1d = a.f[2][src], qs1d = a.f[4][src], ni1d = a.f[6][src];
  const float t1d = a.f[8][src];
#pragma unroll
  for (int q = 0; q < 8; ++q) a.a3[q][dst] = a.f[q][src];
  a.a3[8][dst] = t1d / a.pii[dst];                         // M:1022
  if (a.re_cloud) {
    // calc_effectRad, M:4834-4935 (the column-wide has_qc / has_qi / has_qs only skip loops whose bodies are
    // switched off cell by cell anyway), then the clamps of M:1118-1122
    const float p1d = a.p[src];
    float re_qc = 2.49E-6f, re_qi = 4.99E-6f, re_qs = 9.99E-6f;          // M:1112-1114
    const float rho = 0.622f * p1d / (KP_R * t1d * (qv1d + 0.622f));
    const float rc = fmaxf(KP_R1, qc1d * rho);
    const float nc = a.nc_plane ? fmaxf(KP_R2, a.nc_plane[src] * rho)                // M:4874-4875
                   : a.set_nc ? a.set_nc[(long)j * a.t.ni + i] * 1.e6f : ck.Nt_c;
    const float ri = fmaxf(KP_R1, qi1d * rho);
    const float ni = fmaxf(KP_R2, ni1d * rho);
    const float rs = fmaxf(KP_R1, qs1d * rho);
    if (rc > KP_R1 && nc > KP_R2) {
      int inu_c;
      if (nc < 100.f) inu_c = 15;
      else if (nc > 1.E10f) inu_c = 2;
      else inu_c = min(15, nint_f(1000.E6f / nc) + 2);
      const double lamc = (double)pow_f(nc * ck.am_r * c_g_ratio[inu_c - 1] / rc, ck.obmr);
      re_qc = fmaxf(2.51E-6f, fminf((float)(0.5 * (double)(3.f + (float)inu_c) / lamc), 50.E-6f));
    }
    if (ri > KP_R1 && ni > KP_R2) {
      const double lami = (double)pow_f(ck.am_i * ck.cig[1] * ck.oig1 * ni / ri, ck.obmi);
      re_qi = fmaxf(5.01E-6f, fminf((float)(0.5 * (double)(3.f + 0.f) / lami), 125.E-6f));    // mu_i = 0
    }
    if (rs > KP_R1) {
      const float tc0 = fminf(-0.1f, t1d - 273.15f);
      const float smob = rs * ck.oams;
      const float smo2 = smob;                               // bm_s = 2 branch of M:4907
      const float smoc = field_moment(tc0, ck.cse[0], smo2);
      re_qs = fmaxf(10.E-6f, fminf(0.5f * (smoc / smob), 999.E-6f));
    }
    a.re_cloud[dst] = fmaxf(2.49E-6f, fminf(re_qc, 50.E-6f));
    a.re_ice[dst] = fmaxf(4.99E-6f, fminf(re_qi, 125.E-6f));
    a.re_snow[dst] = fmaxf(9.99E-6f, fminf(re_qs, 999.E-6f));
  }
}

// M:986-1003, one thread per column of the tile (c = i + ni*j)
__global__ void k_wrf_accumulate(WrfArgs a) {
  const long c = (long)blockIdx.x * blockDim.x + threadIdx.x, ncol = (long)a.t.ni * a.t.nj;
  if (c >= ncol) return;
  const int j = (int)(c / a.t.ni), i = (int)(c - (long)j * a.t.ni);
  const long m = a.t.at2(i, j);
  const float pptrain = a.ppt[c], pptice = a.ppt[ncol + c], pptsnow = a.ppt[2 * ncol + c], pptgraul = a.ppt[3 * ncol + c];
  const float rncv = pptrain + pptsnow + pptgraul + pptice;
  a.rainncv[m] = rncv;
  a.rainnc[m] = a.rainnc[m] + pptrain + pptsnow + pptgraul + pptice;
  if (a.snowncv && a.snownc) { a.snowncv[m] = pptsnow + pptice; a.snownc[m] = a.snownc[m] + pptsnow + pptice; }
  if (a.graupelncv && a.graupelnc) { a.graupelncv[m] = pptgraul; a.graupelnc[m] = a.graupelnc[m] + pptgraul; }
  a.sr[m] = (pptsnow + pptgraul + pptice) / (rncv + 1.e-12f);
}

}  // namespace kidmp
