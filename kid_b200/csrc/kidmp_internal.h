// kidmp_internal.h - shared declarations of the CUDA implementation (not part of the ABI).
// Reference: M: = module_mp_thompson09n.f90.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <map>
#include "../../include/kidmp.h"

namespace kidmp {

// ---- PARAMETERs of the scheme (M:30-204) ------------------------------------------------------
#define KP_T_0 273.15f
#define KP_PI 3.1415926536f
#define KP_RHO_W 1000.0f
#define KP_RHO_G 500.0f
#define KP_RHO_I 890.0f
#define KP_NT_C_MAX 1999.E6f
#define KP_MU_S 0.6357f
#define KP_KAP0 490.6f
#define KP_KAP1 17.46f
#define KP_LAM0 20.78f
#define KP_LAM1 3.29f
#define KP_GONV_MIN 1.E4f
#define KP_GONV_MAX 3.E6f
#define KP_AM_S 0.069f
#define KP_AV_R 4854.0f
#define KP_FV_R 195.0f
#define KP_AV_S 40.0f
#define KP_BV_S 0.55f
#define KP_FV_S 100.0f
#define KP_AV_G 442.0f
#define KP_BV_G 0.89f
#define KP_AV_I 1847.5f
#define KP_C_CUBE 0.5f
#define KP_C_SQRD 0.15f
#define KP_EF_SI 0.05f
#define KP_EF_RS 0.95f
#define KP_EF_RG 0.75f
#define KP_EF_RI 0.95f
#define KP_R1 1.E-12f
#define KP_R2 1.E-6f
#define KP_EPS 1.E-15f
#define KP_TNO 5.0f
#define KP_ATO 0.304f
#define KP_HGFR 235.16f
#define KP_R 287.04f
#define KP_CP 1004.0f
#define KP_LSUB 2.834E6f
#define KP_LVAP0 2.5E6f
#define KP_XM0I 1.E-12f
#define KP_D0C 1.E-6f
#define KP_D0R 50.E-6f
#define KP_D0S 200.E-6f
#define KP_D0G 250.E-6f
#define KP_NSTEP_MAX 32767        /* U12: cap of the sedimentation sub-step count */

enum { NBINS = 100, NTB_C = 37, NTB_I = 64, NTB_R = 37, NTB_S = 28, NTB_G = 28, NTB_G1 = 28, NTB_R1 = 37,
       NTB_I1 = 55, NTB_T = 9, NTB_TC = 45 };
enum : long { N_RACG = (long)NTB_G1 * NTB_G * NTB_R1 * NTB_R, N_RACS = (long)NTB_S * NTB_T * NTB_R1 * NTB_R,
              N_QRFZ = (long)NTB_R * NTB_R1 * NTB_TC, N_QCFZ = (long)NTB_C * NTB_TC, N_IAUS = (long)NTB_I * NTB_I1,
              N_EF = (long)NBINS * NBINS };

// interleaved (array-of-structs) table records: every lookup of the step reads all members at
// one index (M:1967-1985, M:2004-2016, M:2067-2070), so one gather touches one contiguous record.
enum { G_TCG_RACG = 0, G_TMR_RACG, G_TCR_GACR, G_TMG_GACR, G_TNR_RACG, G_TNR_GACR, G_N };
enum { S_TCS_RACS1 = 0, S_TMR_RACS1, S_TCS_RACS2, S_TMR_RACS2, S_TCR_SACR1, S_TMS_SACR1, S_TCR_SACR2, S_TMS_SACR2,
       S_TNR_RACS1, S_TNR_RACS2, S_TNR_SACR1, S_TNR_SACR2, S_N };
enum { F_TPI = 0, F_TPG, F_TNI, F_TNR, F_N };        // qrfz
enum { C_TPI = 0, C_TNI, C_N };                      // qcfz
enum { I_TPS = 0, I_TNI, I_TPI_IDE, I_N };           // iaus

// constants written by the host part of init (M:381-670): one copy per handle, a __grid_constant__ parameter `ck` of
// every kernel that reads them
struct KConst {
  float Nt_c, Sc3, D0i, xm0s, xm0g, rho_not;
  float am_r, am_g, am_i, oRv, lfus, olfus;
  float cce[5][15], ccg[5][15], ocg1[15], ocg2[15];
  float cie[7], cig[7], oig1, oig2, obmi;
  float cre[13], crg[13], ore1, org1, org2, org3, obmr;
  float cse[18], csg[18], oams, obms, ocms;
  float cge[12], cgg[12], oge1, ogg1, ogg2, ogg3, oamg, obmg, ocmg;
  float t1_qr_qc, t1_qr_qi, t2_qr_qi, t1_qg_qc, t1_qs_qc, t1_qs_qi, t1_qr_ev, t2_qr_ev;
  float t1_qs_sd, t2_qs_sd, t1_qg_sd, t2_qg_sd, t1_qs_me, t2_qs_me, t1_qg_me, t2_qg_me;
  int nic1, nic2, nii2, nii3, nir2, nir3, nis2, nig2, nig3, niIN2;
  int iiwarm, l_sediment;
  float r_c1, r_i1, r_r1, r_s1, r_g1, Nt_i1;        // first axis nodes (M:215-279)
  float p10[64];                                    // 10.**n as libgcc powi builds it, n = -32..31
  // constant sub-expressions of the column step, evaluated once on the host with libm like the
  // reference evaluates them every level: (crg(3)*org2*org1)**bm_r M:1844, (cgg(3)*ogg2*ogg1)**bm_g
  // M:1888, (cgg(3)*ogg2*ogg1)**obmg M:1651, (ccg(3,nu_c)*ocg2(nu_c))**obmr M:1701
  float n0r_fac, n0g_fac, lamg_fac, dcg_fac[15];
  double Dr1, Ds1, lnDr, lnDs;                      // Dr(1), Ds(1), DLOG(Dr(nbr)/Dr(1)), DLOG(Ds(nbs)/Ds(1))
  double t_Nc1;                                     // t_Nc(1), M:668
  double n0_lo;                                     // graupel_n0_lo() as the device computes it (k_n0_lo, run by kidmp_init)
  const double* tnc_wev;                            // [NBINS][NTB_C][NBINS] (idx_d fastest), table_dropEvap M:4400-4439; NULL until an aerosol-aware step asks for it
  // device tables
  const double* racg;   // [N_RACG][G_N]
  const double* racs;   // [N_RACS][S_N]
  const double* qrfz;   // [N_QRFZ][F_N]
  const double* qcfz;   // [N_QCFZ][C_N]
  const double* iaus;   // [N_IAUS][I_N]
  const float* efrw;    // [100][100] column-major (idx_r, idx_c)
  const float* efsw;
};

// Hand-off between the cell kernels and the column kernels: one record of 32 f32 (SC_* = offset in the record) per BUSY
// cell (a hydrometeor or supersaturation; every rate of an idle cell is exactly zero), in the order of the cell list, kept
// as two arrays of 64-byte halves: floats 0-15 (what only k_finish reads) in `scratch`, floats 16-31 (everything k_carries
// reads) in `scratch_b` - DRAM moves whole 128-byte lines, so k_carries would otherwise drag the other half along.  Every
// access is a whole 32-byte sector (256-bit loads / stores), so the traffic is the records themselves whatever the order
// of the cells; cellidx[k][slot] is the record number of a cell.
//   SC_TTEN..SC_NCTEN  the ten tendencies after S12
//   SC_RR..SC_RG, SC_NR, SC_NI  contents at tau+1 (M:2602-2656 and the in-place refreshes of S11 / S12)
//   SC_VTR..SC_VTNI    the cell's own fall speeds (0 without the species: k_carries applies the rule of the level above)
//   SC_VTS, SC_VTG     written by k_carries (final snow / graupel speed of the level)
//   SC_RHO, SC_S15     air density at tau+1; signed latent-heat factor of S15
//   SC_N0A             S10's intercept without supercooled rain, negated when the level's updated temperature is >= 270.65 K
//   SC_N0B_SLW         S10's intercept with supercooled rain; SC_VTS_RAW / SC_VTS_BOOST / SC_TEMP for the snow speed rule
enum { SC_TTEN = 0, SC_QVTEN, SC_QCTEN, SC_QITEN, SC_QRTEN, SC_QSTEN, SC_QGTEN, SC_NITEN,
       SC_NRTEN = 8, SC_NCTEN, SC_NR, SC_NI, SC_VTNI,
       SC_RR = 16, SC_RI, SC_RS, SC_RG, SC_VTR, SC_VTNR, SC_VTI, SC_RHO,
       SC_S15 = 24, SC_N0A, SC_N0B_SLW, SC_VTS_RAW, SC_VTS_BOOST, SC_TEMP, SC_VTS, SC_VTG, SC_REC = 32, SC_HALF = 16 };

// Cell classes: every busy cell goes to the kernel specialised for the smallest species set that covers it
// (kidmp_cells.cuh).  The class byte of a cell: bits 0-4 qc qi qr qs qg > R1 on input, bit 5 ice supersaturation,
// bit 6 T < T_0; (bits 0-5) == 0: idle cell.
enum { KC_WARM = 0, KC_ICE = 1, KC_MIXNR = 2, KC_FULL = 3, KC_N = 4 };
enum { CLS_QC = 1, CLS_QI = 2, CLS_QR = 4, CLS_QS = 8, CLS_QG = 16, CLS_VAP = 32, CLS_BUSY = 63, CLS_COLD_SHIFT = 6 };
enum { LIST_TILE = 256 };          // columns per block of the cell-list kernels

enum { DIAG_BLOCKS = 296 };

struct StepArgs {
  long ncol;                   // columns of this launch (one chunk of the domain)
  long ld;                     // row stride of the caller's arrays (state, p, dz_col, rates: [nz][ld]; ppt: [4][ld])
  int nz;
  float dt;
  float* f[KIDMP_NFIELDS];     // qv qc qi qr qs qg ni nr t, [nz][ld], pointing at the chunk's first column
  const float* p;              // [nz][ld]
  const float* dz;             // [nz] layer depths shared by all columns (KiD, I:63) ...
  const float* dz_col;         // ... or [nz][ld] per column (WRF's dz(i,k,j), M:944); NULL when dz is used
  float* ppt;                  // [4][ld]
  float* scratch;              // [records][SC_HALF] hand-off (see SC_*): first half of the record of every busy cell, in the order of cell_list
  float* scratch_b;            // [records][SC_HALF] second half
  unsigned* cellidx;           // [nz][count] record number of every busy cell of the cloudy columns
  float* n0a;                  // [nz][count] running minimum of the graupel intercept of S4 at the graupel cells (k_n0_sweep)
  float* ws;                   // [WS_N][nz][ws_cols] SoA workspace of the columns with sedimentation sub-steps (k_substeps)
  long ws_cols;
  unsigned char* cls;          // [nz][ncol] class byte of every cell (0 = idle)
  int* colflag;                // [ncol] < 0 clear sky (the early RETURN of M:1540; -2: a species <= R1 was zeroed, -1: untouched), else bit 0 = graupel somewhere in the column
  int* work_count;             // number of cloudy columns found by the classification kernel
  int* work_list;              // their column indices, compacted in column order (slot -> column)
  unsigned* work_mask;         // [ngroups] ballot of the cloudy lanes of every 32-column group
  int* work_offset;            // [ngroups] exclusive prefix sum of the ballots' popcounts
  unsigned* cell_list;         // [<= nz*ncol] busy cells, sort key after sort key, entry = k << 24 | slot
  int* cell_hist;              // [64] busy cells of each sort key (species bits, T < T_0)
  int* cell_start;             // [64] first entry of each key
  int* cell_count;             // [KC_N] busy cells of each kernel class (+ [KC_N]: all busy cells) ...
  int* cell_kstart;            // [KC_N] ... and its first entry (the keys of a class are next to each other)
  int* cell_base;              // [32-column groups][64] first entry of a group's cells inside the segment of their key
  unsigned* busy;              // [ceil(nz/32)][count] busy bits of every cloudy column (bit k%32 of word k/32)
  int* colint;                 // [8][count] sub-step counts and top sedimenting levels of rain, ice, snow, graupel ([0] < 0: a simple column, see colvmax)
  int* colvmax;                // [2][ncol] by slot, float bits: largest fall speed any cell of the column can hand a level; largest vts / (T - T_0) of its melting snow
  int* sub_count;              // columns that need sedimentation sub-steps (nstep > 1, M:3242) ...
  int* sub_list;               // ... their slots
  float* rates;                // optional [36][nz][ld]
  double* coldiag;             // [2][ncol] liquid / ice water path of each cloudy column
  double* diag_partial;        // [DIAG_BLOCKS][KIDMP_NDIAG] block sums of k_diag_columns
  // aerosol-aware runs (is_aerosol_aware = .true., M:28): prognostic droplet number and aerosol numbers, vertical velocity
  float* nc; float* nwfa; float* nifa;   // [nz][ld] INOUT
  const float* w;                        // [nz][ld] IN
  // per-column droplet number of the plain scheme: set_Nc [cm^-3] of every column, [ld]; Nt_c = set_nc[col] * 1e6f (M:381).
  // NULL: ck.Nt_c everywhere.  Read only by the NCOL instantiations of k_cells, k_substeps and k_finish.
  const float* set_nc;
  int nsm;                     // SMs of the device
  int no_simple;               // 1: every cloudy column goes through the counts of k_carries ("simple" option off: for A/B runs)
  int no_classes;              // 1: every busy cell goes to k_cells<KC_FULL> ("classes" option off: the class kernels' reference)
};

// device tables (kidmp_tables.cuh fills them)
struct TableSet {
  double *racg, *racs, *qrfz, *qcfz, *iaus;
  float *efrw, *efsw;
};
struct HostBins {
  double Dc[NBINS], dtc[NBINS], Di[NBINS], dti[NBINS], Dr[NBINS], dtr[NBINS], Ds[NBINS], dts[NBINS], Dg[NBINS],
      dtg[NBINS], t_Nc[NBINS];
  float r_c[NTB_C], r_i[NTB_I], r_r[NTB_R], r_g[NTB_G], r_s[NTB_S], N0r_exp[NTB_R1], N0g_exp[NTB_G1], Nt_i[NTB_I1];
};

}  // namespace kidmp
