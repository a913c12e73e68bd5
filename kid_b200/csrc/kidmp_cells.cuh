// kidmp_cells.cuh - the physics of mp_thompson (S1..S13 of M:1156-3354) with ONE CELL as the unit of work, and the
// column kernels around it.
//
// Why cells: the process rates of a level depend on that level's inputs only; what runs down a column is small (the
// running minimum of the graupel intercept M:1648 / M:2731, the `k_0` test M:1635, the fall speed of a level without
// the species M:3235, the sub-step counts M:3242).  A column walk spends its time in dependent instruction chains of
// cells that mostly differ from their neighbours (profiles/r01: 19 of 32 lanes active, 45 % issue), and half of the
// cells of a cloudy column are idle.  Here
//   k_classify / k_cell_fill     turn the class bytes into one list of busy cells, sorted by species set and
//                                class, so the lanes of a warp are cells of neighbouring columns that hold the same species;
//   k_n0_sweep                   walks the columns that hold graupel top-down once: running minimum of M:1648;
//   k_cells<KC>                  one thread per busy cell, one kernel per class.  The class is a template parameter:
//                                code that cannot run for the class (every ice process for a warm cell, the collection
//                                tables without rain ...) is not compiled into its kernel, so ptxas needs neither the
//                                registers of the 35 f64 rates nor the 120 KB of instructions where they do not apply;
//   k_carries                    one thread per cloudy column that is not SIMPLE (graupel, or a fall speed that can cross a
//                                layer in one step): what runs down the column - intercept minimum of S10, fall speeds of the
//                                levels without the species, sub-step counts; columns with sub-steps go to k_substeps;
//   k_finish                     one thread per cloudy column: the only sedimentation sub-step (M:3365-3578), S15 and S16
//                                (finish_level); for a simple column also the snow speed of M:3301 and the top sedimenting
//                                levels.  Idle cells never had a hand-off record: their tendencies are zero and their
//                                contents R1 / R2 by construction.
// AERO (template parameter of k_cells, k_finish, k_substeps): is_aerosol_aware = .true., M:28 (kidmp_aero.cuh).
// Pruning rule: a block is compiled out of a class kernel only when it cannot execute for any cell of the class, so
// every class kernel computes bit for bit what the general code (KC_FULL) computes for the same cell.
#pragma once
#include "kidmp_column.cuh"
#include "kidmp_aero.cuh"

namespace kidmp {

// One sector (32 bytes, 8 floats) of a hand-off record per instruction: the 256-bit global accesses of sm_100
// (LDG.E.256 / STG.E.256).  A lane then reads or writes whole sectors of its record, never part of one.
struct Sector { float v[8]; };
// start fetching the line of a record that the next level of a column walk will read
__device__ __forceinline__ void prefetch_record(const float* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void st_sector(float* p, float a, float b, float c, float d, float e, float f, float g, float h) {
#ifdef KIDMP_EVICT_FIRST
#define KIDMP_REC_HINT ".L1::no_allocate.L2::evict_first"
#else
#define KIDMP_REC_HINT ""
#endif
  asm volatile("st.global" KIDMP_REC_HINT ".v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "f"(e),
               "f"(f), "f"(g), "f"(h) : "memory");
}
__device__ __forceinline__ Sector ld_sector(const float* p) {
  Sector s;
  asm volatile("ld.global" KIDMP_REC_HINT ".v8.f32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];" : "=f"(s.v[0]), "=f"(s.v[1]), "=f"(s.v[2]), "=f"(s.v[3]),
               "=f"(s.v[4]), "=f"(s.v[5]), "=f"(s.v[6]), "=f"(s.v[7]) : "l"(p));
  return s;
}

// First half of the hand-off record of the cell at list position `idx`: the ten tendencies and the numbers at tau+1.  A cell
// of the warm class has seven of those words that are not a constant of the class, a cell of the ice class eight (its ice
// number speed rides in the rain-number-speed word of the second half, which its class cannot use): the records of these two
// classes - four fifths of the busy cells, first in the list - keep ONE sector here, the mixed classes two.  An aerosol-aware
// run keeps two sectors everywhere (two more tendencies).  k1, k2: first list entries of the ice and of the mixed classes.
struct RecA { float tt, qvt, qct, qit, qrt, qst, qgt, nit, nrt, nct, nr, ni, v_ni, nwfat, nifat; };
template <bool AERO>
__device__ __forceinline__ float* rec_a_ptr(const StepArgs& a, unsigned idx, unsigned k2) {
  if (AERO) return a.scratch + (size_t)idx * SC_HALF;
  return idx < k2 ? a.scratch + (size_t)idx * 8 : a.scratch + ((size_t)idx * SC_HALF - (size_t)k2 * 8);
}
template <bool AERO>
__device__ __forceinline__ RecA load_rec_a(const StepArgs& a, unsigned idx, unsigned k1, unsigned k2, const Sector& s2) {
  RecA r;
  const float* q = rec_a_ptr<AERO>(a, idx, k2);
  const Sector s0 = ld_sector(q);
  r.nwfat = 0.f; r.nifat = 0.f;
  if (!AERO && idx < k2) {
    r.tt = s0.v[0]; r.qvt = s0.v[1]; r.qct = s0.v[2]; r.qgt = 0.0f;
    if (idx < k1) {          // warm: no ice-phase tendency (the zeros as S8 leaves them: nit = -ni1d * odts with ni1d = 0)
      r.qrt = s0.v[3]; r.nrt = s0.v[4]; r.nct = s0.v[5]; r.nr = s0.v[6];
      r.qit = 0.0f; r.qst = 0.0f; r.nit = -0.0f; r.ni = KP_R2; r.v_ni = 0.0f;
    } else {                 // ice: no rain (qrt = -qr1d * odts, nrt = -nr1d * odts with zero inputs), no graupel
      r.qit = s0.v[3]; r.qst = s0.v[4]; r.nit = s0.v[5]; r.nct = s0.v[6]; r.ni = s0.v[7];
      r.qrt = -0.0f; r.nrt = -0.0f; r.nr = KP_R2; r.v_ni = s2.v[5];
    }
  } else {
    const Sector s1 = ld_sector(q + 8);
    r.tt = s0.v[0]; r.qvt = s0.v[1]; r.qct = s0.v[2]; r.qit = s0.v[3]; r.qrt = s0.v[4]; r.qst = s0.v[5]; r.qgt = s0.v[6]; r.nit = s0.v[7];
    r.nrt = s1.v[0]; r.nct = s1.v[1]; r.nr = s1.v[2]; r.ni = s1.v[3]; r.v_ni = s1.v[4];
    if (AERO) { r.nwfat = s1.v[5]; r.nifat = s1.v[6]; }
  }
  return r;
}

// M:1649-1653 for a given intercept (the running minimum already taken)
__device__ __forceinline__ void graupel_slope(double N0_exp, float rg, double& ilamg, double& N0_g) {
  const double lam_exp = sqrt(sqrt(N0_exp * (double)ck.am_g * (double)ck.cgg[0] / (double)rg));   // **oge1, oge1 = 1/4
  const double lamg = lam_exp * (double)ck.lamg_fac;
  ilamg = (double)1.f / lamg;
  N0_g = N0_exp / ((double)ck.cgg[1] * lam_exp) * lamg;                                         // lamg**cge(2), cge(2) = 1
}

// What a cell of each class can hold.  Input species (S1..S8 read the input flags) and species at tau+1 (S9 on).
//   KC_WARM   no ice-phase species and (T >= T_0 or iiwarm): none can form (freezing and nucleation need T < T_0, M:2025)
//   KC_ICE    T < T_0, no cloud water, rain or graupel: liquid cannot form before S11, graupel needs liquid (M:2224, M:1964)
//   KC_MIXNR  anything without rain on input (rain may form: autoconversion, melting)
//   KC_FULL   everything
template <int KC> struct CellTraits {
  static constexpr bool C = KC != KC_ICE, R = KC == KC_WARM || KC == KC_FULL, I = KC != KC_WARM, S = KC != KC_WARM,
                        G = KC == KC_MIXNR || KC == KC_FULL;
  static constexpr bool ICEPROC = KC != KC_WARM;          // the `if (.not. iiwarm)` blocks can do something
  static constexpr bool COLD = KC == KC_ICE;              // T < T_0 is certain
  static constexpr bool C9 = KC != KC_ICE, R9 = KC != KC_ICE, I9 = KC != KC_WARM, S9 = KC != KC_WARM,
                        G9 = KC == KC_MIXNR || KC == KC_FULL;
};

#define R1 KP_R1
#define R2 KP_R2
#define EPSF KP_EPS
#define T_0 KP_T_0
#define D0r KP_D0R
#define D0c KP_D0C
#define D0s KP_D0S
#define D0g KP_D0G

// ---- lists of busy cells ------------------------------------------------------------------------------------------
// Sort key of a busy cell: its five species bits and whether it is below 0 C (64 keys).  The list holds the cells key after
// key, the keys of one kernel class next to each other, so a class kernel walks one contiguous range in which the 32
// cells of a warp hold the SAME species (same branches) and, inside a key, are the cells of 32 neighbouring columns level
// after level from the top (neighbouring columns of one or a few levels: same table entries, few cache lines per load;
// the order is the same from run to run).
// k_classify (kidmp_column.cuh) counts the keys per 32-column group and per launch while it writes the class bytes;
// k_cell_offsets: first entry of every key and class; k_cell_fill: the entries, and the busy bits of every cloudy column
// for the column kernels.
__global__ void __launch_bounds__(64) k_cell_offsets(StepArgs a) {
  __shared__ int s_n[64], s_kc[64];
  const int t = threadIdx.x;
  const bool iiwarm = ck.iiwarm != 0;
  s_n[t] = a.cell_hist[t];
  s_kc[t] = a.no_classes ? KC_FULL : cell_kernel_class((unsigned)t & 31u, (t >> 5) != 0, iiwarm);
  __syncthreads();
  int start = 0;
  for (int j = 0; j < 64; ++j) if (s_kc[j] < s_kc[t] || (s_kc[j] == s_kc[t] && j < t)) start += s_n[j];
  a.cell_start[t] = start;
  if (t < KC_N) {
    int n = 0, first = 0;
    for (int j = 0; j < 64; ++j) { if (s_kc[j] == t) n += s_n[j]; if (s_kc[j] < t) first += s_n[j]; }
    a.cell_count[t] = n; a.cell_kstart[t] = first;
  }
  if (t == 0) { int n = 0; for (int j = 0; j < 64; ++j) n += s_n[j]; a.cell_count[KC_N] = n; }
}
__global__ void __launch_bounds__(LIST_TILE) k_cell_fill(StepArgs a) {
  __shared__ int s_run[LIST_TILE / 32][64];               // next entry of every key for the cells of this warp
  const int nz = a.nz;
  const long col = (long)blockIdx.x * LIST_TILE + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool in_range = col < a.ncol;
  const unsigned gmask = in_range ? a.work_mask[col >> 5] : 0u;
  if (__shfl_sync(0xffffffffu, gmask, 0) == 0u) return;   // no cloudy column among the 32 of this warp (lane 0 is in range or the warp is empty)
  {
    const int* base = a.cell_base + ((long)blockIdx.x * (LIST_TILE / 32) + warp) * 64;
    s_run[warp][lane] = a.cell_start[lane] + base[lane];                 // (garbage for keys this warp does not hold: never read)
    s_run[warp][lane + 32] = a.cell_start[lane + 32] + base[lane + 32];
  }
  __syncwarp();
  const unsigned count = (unsigned)*a.work_count;
  const unsigned slot = (unsigned)a.work_offset[in_range ? (col >> 5) : 0] + __popc(gmask & ((1u << lane) - 1u));
  const bool cloudy = in_range && ((gmask >> lane) & 1u);
  const unsigned char* cp = a.cls + col;
  unsigned bword = 0;                                     // busy bits of 32 levels of my column, for the column kernels
  constexpr int LB = 16;                                  // class bytes of 16 levels in flight at a time
#pragma unroll 1
  for (int k0 = nz - 1; k0 >= 0; k0 -= LB) {
    unsigned cb[LB];
#pragma unroll
    for (int j = 0; j < LB; ++j) cb[j] = (in_range && k0 - j >= 0) ? cp[(long)(k0 - j) * a.ncol] : 0u;
#pragma unroll
  for (int j = 0; j < LB; ++j) {
    const int k = k0 - j;
    if (k < 0) break;
    const unsigned c = cb[j];
    const bool busy = (c & CLS_BUSY) != 0u;
    const unsigned act = __ballot_sync(0xffffffffu, busy);
    if (busy) {
      bword |= 1u << (k & 31);
      const unsigned key = cell_key(c);
      const unsigned m = __match_any_sync(act, key);
      const int leader = __ffs(m) - 1;
      int base = 0;
      if (lane == leader) { base = s_run[warp][key]; s_run[warp][key] = base + __popc(m); }
      base = __shfl_sync(m, base, leader);
      const unsigned pos = (unsigned)base + __popc(m & ((1u << lane) - 1u));
      a.cell_list[pos] = (unsigned)k << 24 | slot;          // nz <= 256 levels, at most 2^24 columns per launch
      a.cellidx[(size_t)k * count + slot] = pos;             // where the column kernels find the record of this cell
    }
    __syncwarp();
    if ((k & 31) == 0) { if (cloudy) a.busy[(size_t)(k >> 5) * count + slot] = bword; bword = 0; }
  }
  }
}

// ---- running minimum of the graupel intercept of S4 (M:1633-1648), only for columns that hold graupel: the slope and
// intercept it feeds (M:1649-1653) are read by graupel processes alone.  One thread per cloudy column, top-down; the value
// of every graupel cell goes to n0a[k][slot].  Needs the work list only: runs beside the cell-list kernels.  The rain of S1 is needed for the supercooled-drop test of M:1640.
__global__ void __launch_bounds__(128) k_n0_sweep(StepArgs a) {
  const int slot = blockIdx.x * 128 + threadIdx.x;
  const int count = *a.work_count;
  if (slot >= count || ck.iiwarm) return;
  const long col = a.work_list[slot];
  if (!(a.colflag[col] & 1)) return;
  const int nz = a.nz;
  const long ld = a.ld;
  float* const n0a = a.n0a + slot;                         // [nz][count], read by the cell kernels for graupel cells
  const double n0_empty = g_n0_lo;
  bool warm_a = false;                                    // a level at or above this one has T >= 270.65 K (k_0, M:1635)
  double n0_min = (double)KP_GONV_MAX;
  constexpr int B = 6;                                    // levels loaded per batch: the walk is a chain of dependent steps,
#pragma unroll 1                                          // so the loads of several levels are put in flight together
  for (int k0 = nz - 1; k0 >= 0; k0 -= B) {
    float tb[B], gb[B], rb[B];
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const int k = k0 - j;
      const long g = (long)(k >= 0 ? k : 0) * ld + col;
      tb[j] = a.f[F_T][g]; gb[j] = a.f[F_QG][g]; rb[j] = a.f[F_QR][g];
    }
#pragma unroll
    for (int j = 0; j < B; ++j) {
      const int k = k0 - j;
      if (k < 0) break;
      const long g = (long)k * ld + col;
      const float t1d = tb[j], qg1d = gb[j], qr1d = rb[j];
      if (t1d >= 270.65f) warm_a = true;
      const bool cold_rain = !warm_a && k > 0 && qr1d > R1;
      if (qg1d > R1 || cold_rain) {
        const float pres = a.p[g], qv = fmaxf(1.E-10f, a.f[F_QV][g]);
        const float rho = 0.622f * pres / (KP_R * t1d * (qv + 0.622f));
        const float rg = (qg1d > R1) ? qg1d * rho : R1;
        bool slw = false;
        float mvd_r = 0.f;
        if (cold_rain) {                                  // the rain of S1 (M:1445-1466) for the xslw1 of M:1640
          const float rr = qr1d * rho;
          float nr = fmaxf(R2, a.f[F_NR][g] * rho);
          if (nr <= R2) { mvd_r = 1.0E-3f; nr = nr_from_mvd(rr, mvd_r); }
          const double lamr = rain_lam(nr, rr);
          mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr);
          if (mvd_r > 2.5E-3f) mvd_r = 2.5E-3f;
          else if (mvd_r < D0r * 0.75f) mvd_r = D0r * 0.75f;
          slw = mvd_r > 100.E-6f;
        }
        double N0_exp = n0_empty;
        if (slw || rg > 5.E-5f) N0_exp = graupel_n0_exp(slw ? 4.01f + log10_f(mvd_r) : 0.01f, rg);
        n0_min = fmin(N0_exp, n0_min);
        if (qg1d > R1) n0a[(size_t)k * count] = (float)n0_min;     // values of M:1646 are f32 numbers: exact
      } else {
        n0_min = fmin(n0_empty, n0_min);
      }
    }
  }
}

// ---- K1: S1..S13 of one busy cell ---------------------------------------------------------------------------------
// LOCK: the warps of a block meet at named barriers between the stages, so they run the same straight-line code at the
// same time and share its instruction-cache lines (the full cell code is ~100 KB of SASS; profiles/r01).  Used for the
// classes with the long bodies; the short ones run free.
// AERO: is_aerosol_aware = .true. (M:28): cloud droplet number, water-friendly and ice-friendly aerosol numbers are prognostic
// (a.nc, a.nwfa, a.nifa), a.w feeds the droplet activation; every aerosol block is compiled out of the default kernels.
template <int KC, int THREADS, int MINB, int BARS, bool RATES, bool AERO>
__global__ void __launch_bounds__(THREADS, MINB) k_cells(StepArgs a) {
  using TR = CellTraits<KC>;
  constexpr bool LOCK = BARS != 0;
  const int n = a.cell_count[KC];
  const unsigned* __restrict__ list = a.cell_list + a.cell_kstart[KC];
  const int nz = a.nz;
  const long ld = a.ld;
  const unsigned count = (unsigned)*a.work_count;
  const unsigned kstart = (unsigned)a.cell_kstart[KC], k2_list = (unsigned)a.cell_kstart[KC_MIXNR];
  float* const sb_class = a.scratch_b + (size_t)kstart * SC_HALF;            // records in list order: the half that k_carries reads as well ...
  constexpr bool COMPACT = !AERO && (KC == KC_WARM || KC == KC_ICE);         // ... and the half that only k_finish reads (RecA)
  const float DT = a.dt;
  const float odt = 1.f / DT, odts = 1.f / DT;
  const float Nt_c = ck.Nt_c;
  const bool iiwarm = ck.iiwarm != 0;
  const double n0_empty = g_n0_lo;
#define LOCKBAR(i) do { if (LOCK && ((BARS >> (i)) & 1)) { __syncwarp(); asm volatile("bar.sync 1, %0;" ::"r"(lock_threads) : "memory"); } } while (0)
#pragma unroll 1
  for (int base = blockIdx.x * THREADS; base < n; base += gridDim.x * THREADS) {
    if (LOCK && base != (int)blockIdx.x * THREADS) __syncthreads();      // the stage barriers of two rounds must not mix
    const int wbase = base + (threadIdx.x & ~31);
    if (wbase >= n) { if (LOCK) continue; else return; }
    const int lock_threads = min(THREADS, ((n - base + 31) >> 5) << 5);
    const int i = base + threadIdx.x;
    const bool valid = i < n;                             // lanes past the end shadow the warp's first cell: same branches, nothing stored
    const unsigned e = list[valid ? i : wbase];
    const int k = (int)(e >> 24);
    const unsigned slot = e & 0xffffffu;
    const long col = a.work_list[slot];
    const long o = (long)k * ld + col;
    LOCKBAR(0);
    const float t1d = a.f[F_T][o], qv1d = a.f[F_QV][o], pres = a.p[o];
    float qc1d = TR::C ? a.f[F_QC][o] : 0.0f, qi1d = TR::I ? a.f[F_QI][o] : 0.0f, qr1d = TR::R ? a.f[F_QR][o] : 0.0f,
          qs1d = TR::S ? a.f[F_QS][o] : 0.0f, qg1d = TR::G ? a.f[F_QG][o] : 0.0f;
    float ni1d = TR::I ? a.f[F_NI][o] : 0.0f, nr1d = TR::R ? a.f[F_NR][o] : 0.0f;
    float nc1d_in = 0.f, nwfa1d = 0.f, nifa1d = 0.f, w1d = 0.f;
    if (AERO) { nc1d_in = TR::C ? a.nc[o] : 0.0f; nwfa1d = a.nwfa[o]; nifa1d = a.nifa[o]; w1d = a.w[o]; }
    float* const sc = rec_a_ptr<AERO>(a, kstart + (unsigned)(valid ? i : wbase), k2_list);
    float* const sb = sb_class + (size_t)(valid ? i : wbase) * SC_HALF;

    // rates, M:1184-1211 (zeroed M:1282-1363)
    double prw_vcd = 0., pnc_wcd = 0., pnc_wau = 0., pnc_rcw = 0., pnc_scw = 0., pnc_gcw = 0.;
    double prv_rev = 0., prr_wau = 0., prr_rcw = 0., prr_rcs = 0., prr_rcg = 0., prr_sml = 0., prr_gml = 0., prr_rci = 0.;
    double pnr_wau = 0., pnr_rcs = 0., pnr_rcg = 0., pnr_rci = 0., pnr_sml = 0., pnr_gml = 0., pnr_rev = 0., pnr_rcr = 0., pnr_rfz = 0.;
    double pri_inu = 0., pni_inu = 0., pri_ihm = 0., pni_ihm = 0., pri_wfz = 0., pni_wfz = 0., pri_rfz = 0., pni_rfz = 0.;
    double pri_ide = 0., pni_ide = 0., pri_rci = 0., pni_rci = 0., pni_sci = 0., pni_iau = 0.;
    double prs_iau = 0., prs_sci = 0., prs_rcs = 0., prs_scw = 0., prs_sde = 0., prs_ihm = 0., prs_ide = 0.;
    double prg_scw = 0., prg_rfz = 0., prg_gde = 0., prg_gcw = 0., prg_rci = 0., prg_rcs = 0., prg_rcg = 0., prg_ihm = 0.;
    float smo0 = 0.f, smo1 = 0.f, smob = 0.f, smoc = 0.f, smoe = 0.f, smof = 0.f;
    bool have_smoe = false;
    float mvd_r = 0.f, mvd_c = 0.f, vts_boost = 0.f;
    double ilamg = 0., N0_g = 0., ilamr = 0., N0_r = 0., lamr = 0., lamc = 0., lami = 0., ilami = 0.;
    int nu_c = 0;
    float xDc = 0.f;
    // number tendencies are summed as their terms appear (M:2417, M:2453, M:2503 add them up later): the
    // 22 individual number rates need not stay in registers until S8
    double nc_acc = 0., ni_acc = 0., nr_acc = 0.;
    double na_acc = 0., nd_acc = 0., pri_iha = 0., pni_iha = 0.;   // AERO: pna_rca + pna_sca + pna_gca (+ pni_iha at S8), pnd_rcd + pnd_scd + pnd_gcd (M:2399-2402)
    float nwfa = 0.f, nifa = 0.f;
    // lamr / lami hold rain_lam(nr, rr) / ice_lam(ni, ri) of the current nr, rr / ni, ri unless the number was
    // re-diagnosed after they were evaluated: the reference evaluates the same power again at M:1661, M:2118,
    // M:2750 and M:3227 from unchanged arguments, which is the same number
    bool lamr_stale = false, lami_stale = false;

    // ---- S1, M:1387-1493 -------------------------------------------------------------------
    float temp = t1d;
    float qv = fmaxf(1.E-10f, qv1d);
    float rho = 0.622f * pres / (KP_R * temp * (qv + 0.622f));
    float rc, nc, ri, ni, rr, nr, rs, rg;
    bool L_qc, L_qi, L_qr, L_qs, L_qg;
    if (AERO) {                                            // M:1392-1393
      nwfa = fmaxf(11.1E6f, fminf(9999.E6f, nwfa1d * rho));
      nifa = fmaxf(KP_NAIN1 * 0.01f, fminf(9999.E6f, nifa1d * rho));
    }
    if (TR::C && qc1d > R1) {
      rc = qc1d * rho;
      L_qc = true;
      nc = Nt_c;   // the lamc/xDc clamps of M:1399-1408 only feed nc, overwritten at M:1410 ...
      if (AERO) {  // ... unless the scheme is aerosol aware
        nc = fmaxf(2.f, nc1d_in * rho);
        const int nu = min(15, nint_f(1000.E6f / nc) + 2);
        double lc = (double)pow_f(nc * ck.am_r * ck.ccg[1][nu - 1] * ck.ocg1[nu - 1] / rc, ck.obmr);
        const float xD = (float)((double)(3.f + (float)nu + 1.f) / lc);
        if (xD < D0c) lc = (double)(ck.cce[1][nu - 1] / D0c);
        else if (xD > D0r * 2.f) lc = (double)(ck.cce[1][nu - 1] / (D0r * 2.f));
        nc = (float)fmin((double)KP_NT_C_MAX, (double)(ck.ccg[0][nu - 1] * ck.ocg2[nu - 1] * rc / ck.am_r) * cube_d(lc));
      }
    } else {
      qc1d = 0.0f; nc1d_in = 0.0f; rc = R1; nc = 2.f; L_qc = false;
    }
    if (TR::I && qi1d > R1) {
      ri = qi1d * rho;
      ni = fmaxf(R2, ni1d * rho);
      if (ni <= R2) {
        lami = (double)(ck.cie[1] / 25.E-6f);
        ni = (float)fmin(499.E3, (double)(ck.cig[0] * ck.oig2 * ri / ck.am_i) * cube_d(lami));
      }
      L_qi = true;
      lami = ice_lam(ni, ri);
      ilami = (double)1.f / lami;
      const float xDi = (float)((double)(3.f + 0.f + 1.f) * ilami);
      if (xDi < 5.E-6f) {
        const double l2 = (double)(ck.cie[1] / 5.E-6f);
        ni = (float)fmin(499.E3, (double)(ck.cig[0] * ck.oig2 * ri / ck.am_i) * cube_d(l2));
        lami_stale = true;
      } else if (xDi > 300.E-6f) {
        const double l2 = (double)(ck.cie[1] / 300.E-6f);
        ni = (float)((double)(ck.cig[0] * ck.oig2 * ri / ck.am_i) * cube_d(l2));
        lami_stale = true;
      }
    } else {
      qi1d = 0.0f; ni1d = 0.0f; ri = R1; ni = R2; L_qi = false;
    }
    if (TR::R && qr1d > R1) {
      rr = qr1d * rho;
      nr = fmaxf(R2, nr1d * rho);
      if (nr <= R2) { mvd_r = 1.0E-3f; nr = nr_from_mvd(rr, mvd_r); }
      L_qr = true;
      lamr = rain_lam(nr, rr);
      mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr);
      if (mvd_r > 2.5E-3f) { mvd_r = 2.5E-3f; nr = nr_from_mvd(rr, mvd_r); lamr_stale = true; }
      else if (mvd_r < D0r * 0.75f) { mvd_r = D0r * 0.75f; nr = nr_from_mvd(rr, mvd_r); lamr_stale = true; }
    } else {
      qr1d = 0.0f; nr1d = 0.0f; rr = R1; nr = R2; L_qr = false;
    }
    if (TR::S && qs1d > R1) { rs = qs1d * rho; L_qs = true; } else { qs1d = 0.0f; rs = R1; L_qs = false; }
    if (TR::G && qg1d > R1) { rg = qg1d * rho; L_qg = true; } else { qg1d = 0.0f; rg = R1; L_qg = false; }

    // ---- S2, M:1503-1533 -------------------------------------------------------------------
    float tempc = temp - 273.15f;
    float rhof = sqrtf(ck.rho_not / rho);
    float rhof2 = sqrtf(rhof);
    float qvs = rslf(pres, temp);
    const float qvsi = (tempc <= 0.0f) ? rsif(pres, temp) : qvs;
    float ssatw = qv / qvs - 1.f;
    float ssati = qv / qvsi - 1.f;
    if (fabsf(ssatw) < EPSF) ssatw = 0.0f;
    if (fabsf(ssati) < EPSF) ssati = 0.0f;
    // diffu (M:1512) is read by vapour deposition / sublimation and melting of ice, snow and graupel only (M:1896,
    // M:2126, M:2156, M:2166, M:2238, M:2255); rain evaporation evaluates its own (M:2888)
    const bool ice_any = TR::ICEPROC && !iiwarm && (L_qi || L_qs || L_qg);
    float diffu = 0.f;
    if (ice_any) diffu = 2.11E-5f * pow_f(temp / 273.15f, 1.94f) * (101325.f / pres);
    float visco = (tempc >= 0.0f) ? (1.718f + 0.0049f * tempc) * 1.0E-5f
                                  : (1.718f + 0.0049f * tempc - 1.2E-5f * tempc * tempc) * 1.0E-5f;
    float ocp = 1.f / (KP_CP * (1.f + 0.887f * qv));
    float vsc2 = sqrtf(rho / visco);
    float lvap = KP_LVAP0 + (2106.0f - 4218.0f) * tempc;
    float tcond = (5.69f + 0.0168f * tempc) * 1.0E-5f * 418.936f;

    if (TR::ICEPROC && !iiwarm) {
      // ---- S3, M:1545-1628 snow moments ----------------------------------------------------
      if (L_qs) {
        const float tc0 = fminf(-0.1f, temp - 273.15f);
        smob = rs * ck.oams;
        const float smo2 = smob;                    // bm_s = 2 branch of M:1553
        const float* sa = c_sa; const float* sb = c_sb;
        // Of the six moments of M:1555-1626 the 1st and the (1+(bv_s+1)/2)-th feed deposition, sublimation and melting
        // of every snow level.  The 0th is only read by the melting number rate (M:2242, at or above 0 C), the
        // (bm_s+1)-th by riming (M:1905, with cloud water) and the (bv_s+2)-th by riming and by the collection of
        // cloud ice (M:1910, M:2185): those three are evaluated where they are read.
        float loga_ = sa[1] + sa[2] * tc0 + sa[3] + sa[4] * tc0 + sa[5] * tc0 * tc0 + sa[6] + sa[7] * tc0 * tc0
                      + sa[8] * tc0 + sa[9] * tc0 * tc0 * tc0 + sa[10];
        float b_ = sb[1] + sb[2] * tc0 + sb[3] + sb[4] * tc0 + sb[5] * tc0 * tc0 + sb[6] + sb[7] * tc0 * tc0
                   + sb[8] * tc0 + sb[9] * tc0 * tc0 * tc0 + sb[10];
        smo1 = pow10_f(loga_) * pow_f(smo2, b_);
        smof = field_moment(tc0, ck.cse[15], smo2);
      }
      // ---- S4, M:1633-1654 graupel intercept: the running minimum of M:1648 comes from k_n0_sweep -----------
      if (TR::G && L_qg) graupel_slope((double)a.n0a[(size_t)k * count + slot], rg, ilamg, N0_g);
    }
    // M:1661-1666 rain slope and intercept.  Without rain (rr = R1, nr = R2) every reader of lamr, ilamr, N0_r
    // and mvd_r is switched off (L_qr at M:1676, M:1724, M:2880; rr >= r_r(1) at M:1818, M:1964, M:2028, M:2188)
    if (TR::R && L_qr) {
      if (lamr_stale) { lamr = rain_lam(nr, rr); mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr); }
      ilamr = (double)1.f / lamr;
      N0_r = (double)(nr * ck.org2) * lamr;                                // lamr**cre(2), cre(2) = 1
    }

    // ---- S5, M:1676-1742 warm rain -----------------------------------------------------------
    if (TR::R && L_qr && mvd_r > D0r) {
      const float Ef_rr = 1.0f - exp_f(2300.0f * (mvd_r - 1950.0E-6f));
      pnr_rcr = (double)(Ef_rr * 2.0f * nr * rr);
      nr_acc -= pnr_rcr;
    }
    mvd_c = D0c;
    if (TR::C && L_qc) {
      nu_c = min(15, nint_f(1000.E6f / nc) + 2);
      xDc = fmaxf(D0c * 1.E6f, pow_f(rc / (ck.am_r * nc), ck.obmr) * 1.E6f);
      lamc = (double)pow_f(nc * ck.am_r * ck.ccg[1][nu_c - 1] * ck.ocg1[nu_c - 1] / rc, ck.obmr);
      mvd_c = (float)((double)(3.0f + (float)nu_c + 0.672f) / lamc);
    }
    if (TR::C && rc > 0.01e-3f) {
      const float Dc_g = (float)(((double)ck.dcg_fac[nu_c - 1] / lamc) * (double)1.E6f);
      const float Dc_b = pow_f(xDc * xDc * xDc * Dc_g * Dc_g * Dc_g - xDc * xDc * xDc * xDc * xDc * xDc, 1.f / 6.f);
      const float zeta1 = 0.5f * ((6.25E-6f * xDc * Dc_b * Dc_b * Dc_b - 0.4f) + fabsf(6.25E-6f * xDc * Dc_b * Dc_b * Dc_b - 0.4f));
      const float zeta = 0.027f * rc * zeta1;
      // Below the autoconversion threshold zeta is exactly +0 (most cloudy cells) and so are the three rates: the
      // divisions are skipped there (0/x takes the slow path of the division routines: 3 x ~60 instructions for
      // nearly every cloud level, profiles/r01).  A NaN zeta (negative argument of the 6th root) takes the full path.
      if (!(zeta == 0.0f)) {
        const float taud = 0.5f * ((0.5f * Dc_b - 7.5f) + fabsf(0.5f * Dc_b - 7.5f)) + R1;
        const float tau = 3.72f / (rc * taud);
        prr_wau = (double)(zeta / tau);
        prr_wau = fmin((double)(rc * odts), prr_wau);
        pnr_wau = prr_wau / (double)(ck.am_r * (float)nu_c * D0r * D0r * D0r);
        pnc_wau = fmin((double)(nc * odts), prr_wau / (double)(ck.am_r * mvd_c * mvd_c * mvd_c));
        nr_acc += pnr_wau; nc_acc -= pnc_wau;
      }
    }
    if (TR::R && TR::C && L_qr && mvd_r > D0r && mvd_c > D0c) {
      lamr = (double)1.f / ilamr;
      int idx = 1 + (int)((double)NBINS * log((double)mvd_r / ck.Dr1) / ck.lnDr);
      idx = min(idx, (int)NBINS);
      int jc = (int)(mvd_c * 1.E6f);
      jc = max(1, min(jc, (int)NBINS));                                   // U11: bound the unbounded subscript
      const float Ef_rw = ck.efrw[(idx - 1) + NBINS * (jc - 1)];
      const double lf4 = 1.0 / sq_d(sq_d(lamr + (double)KP_FV_R));          // (lamr+fv_r)**(-cre(9)), cre(9) = 4
      prr_rcw = (double)(rhof * ck.t1_qr_qc * Ef_rw * rc) * N0_r * lf4;
      prr_rcw = fmin((double)(rc * odts), prr_rcw);
      pnc_rcw = (double)(rhof * ck.t1_qr_qc * Ef_rw * nc) * N0_r * lf4;
      pnc_rcw = fmin((double)(nc * odts), pnc_rcw);
      nc_acc -= pnc_rcw;
    }
    // M:1729-1740 rain collecting aerosols, wet scavenging
    if (AERO && TR::R && L_qr && mvd_r > D0r) {
      lamr = (double)1.f / ilamr;
      const double lf4 = 1.0 / sq_d(sq_d(lamr + (double)KP_FV_R));          // (lamr+fv_r)**(-cre(9)), cre(9) = 4
      float Ef_ra = eff_aero<'r'>(mvd_r, 0.04E-6f, visco, rho, temp);
      const double pna_rca = fmin((double)(nwfa * odts), (double)(rhof * ck.t1_qr_qc * Ef_ra * nwfa) * N0_r * lf4);
      Ef_ra = eff_aero<'r'>(mvd_r, 0.8E-6f, visco, rho, temp);
      const double pnd_rcd = fmin((double)(nifa * odts), (double)(rhof * ck.t1_qr_qc * Ef_ra * nifa) * N0_r * lf4);
      na_acc += pna_rca; nd_acc += pnd_rcd;
    }

    LOCKBAR(1);
    // ---- S6, M:1749-2286 ice-phase processes --------------------------------------------------
    if (TR::ICEPROC && !iiwarm) {
      vts_boost = 1.5f;
      tempc = temp - 273.15f;
      const int idx_tc = max(1, min(nint_f(-tempc), 45));
      int idx_t = (int)((tempc - 2.5f) / 5.f) - 1;
      idx_t = max(1, -idx_t);
      idx_t = min(idx_t, (int)NTB_T);
      const int idx_c = (TR::C && rc > ck.r_c1) ? decade_idx_f(rc, ck.nic2, NTB_C) : 1;
      const int idx_i = (ri > ck.r_i1) ? decade_idx_f(ri, ck.nii2, NTB_I) : 1;
      const int idx_i1 = (ni > ck.Nt_i1) ? decade_idx_f(ni, ck.nii3, NTB_I1) : 1;
      int idx_r = 1, idx_r1 = NTB_R1, idx_s = 1, idx_g = 1, idx_g1 = NTB_G1;
      if (TR::R && rr > ck.r_r1) {
        idx_r = decade_idx_f(rr, ck.nir2, NTB_R);
        lamr = (double)1.f / ilamr;
        const double lam_exp = lamr * (double)ck.n0r_fac;
        const double N0_exp = (double)(ck.org1 * rr / ck.am_r) * sq_d(sq_d(lam_exp));   // **cre(1), cre(1) = 4
        idx_r1 = decade_idx_d(N0_exp, ck.nir3, NTB_R1);
      }
      if (TR::R) idx_s = (rs > ck.r_s1) ? decade_idx_f(rs, ck.nis2, NTB_S) : 1;          // only the rain-snow tables read it
      if (TR::R && TR::G && rg > ck.r_g1) {                                              // only the rain-graupel tables read them
        idx_g = decade_idx_f(rg, ck.nig2, NTB_G);
        const double lamg = (double)1.f / ilamg;
        const double lam_exp = lamg * (double)ck.n0g_fac;
        const double N0_exp = (double)(ck.ogg1 * rg / ck.am_g) * sq_d(sq_d(lam_exp));   // **cge(1), cge(1) = 4
        idx_g1 = decade_idx_d(N0_exp, ck.nig3, NTB_G1);
      }

      // M:1884-1900 sublimation/deposition prefactor
      // (rvs and t1_subl are read by the deposition / sublimation rates of ice, snow and graupel only)
      float rvs = 0.f, t1_subl = 0.f;
      if (ice_any) {
        const float otemp = 1.f / temp;
        const float lsub = KP_LSUB, oRv = ck.oRv;
        rvs = rho * qvsi;
        const float rvs_p = rvs * otemp * (lsub * otemp * oRv - 1.f);
        const float rvs_pp = rvs * (otemp * (lsub * otemp * oRv - 1.f) * otemp * (lsub * otemp * oRv - 1.f)
                                    + (-2.f * lsub * otemp * otemp * otemp * oRv) + otemp * otemp);
        const float gamsc = lsub * diffu / tcond * rvs_p;
        float alphsc = 0.5f * (gamsc / (1.f + gamsc)) * (gamsc / (1.f + gamsc)) * rvs_pp / rvs_p * rvs / rvs_p;
        alphsc = fmaxf(1.E-9f, alphsc);
        float xsat = ssati;
        if (fabsf(xsat) < 1.E-9f) xsat = 0.f;
        t1_subl = 4.f * KP_PI * (1.0f - alphsc * xsat + 2.f * alphsc * alphsc * xsat * xsat
                                 - 5.f * alphsc * alphsc * alphsc * xsat * xsat * xsat) / (1.f + gamsc);
      }

      // M:1903-1935 riming of snow and graupel
      if (TR::C && L_qc && mvd_c > D0c) {
        float xDs = 0.0f;
        if (L_qs) { smoc = field_moment(fminf(-0.1f, temp - 273.15f), ck.cse[0], smob); xDs = smoc / smob; }
        if (xDs > D0s) {
          smoe = field_moment(fminf(-0.1f, temp - 273.15f), ck.cse[12], smob); have_smoe = true;
          int idx = 1 + (int)((double)NBINS * log((double)xDs / ck.Ds1) / ck.lnDs);
          idx = min(idx, (int)NBINS);
          int jc = (int)(mvd_c * 1.E6f);
          jc = max(1, min(jc, (int)NBINS));                               // U11
          const float Ef_sw = ck.efsw[(idx - 1) + NBINS * (jc - 1)];
          prs_scw = (double)(rhof * ck.t1_qs_qc * Ef_sw * rc * smoe);
          pnc_scw = (double)(rhof * ck.t1_qs_qc * Ef_sw * nc * smoe);
          pnc_scw = fmin((double)(nc * odts), pnc_scw);
          nc_acc -= pnc_scw;
        }
        if (TR::G && rg >= ck.r_g1 && mvd_c > D0c) {
          const float xDg = (float)((double)(3.f + 0.f + 1.f) * ilamg);
          const float vtg = (float)((double)(rhof * KP_AV_G * ck.cgg[5] * ck.ogg3) * pow_d(ilamg, (double)KP_BV_G));
          const float stoke_g = mvd_c * mvd_c * vtg * KP_RHO_W / (9.f * visco * xDg);
          if (xDg > D0g) {
            float Ef_gw = 0.0f;
            if (stoke_g >= 0.4f && stoke_g <= 10.f) Ef_gw = 0.55f * log10_f(2.51f * stoke_g);
            else if (stoke_g < 0.4f) Ef_gw = 0.0f;
            else if (stoke_g > 10.f) Ef_gw = 0.77f;
            const double il9 = pow_d(ilamg, (double)ck.cge[8]);
            prg_gcw = (double)(rhof * ck.t1_qg_qc * Ef_gw * rc) * N0_g * il9;
            pnc_gcw = (double)(rhof * ck.t1_qg_qc * Ef_gw * nc) * N0_g * il9;
            pnc_gcw = fmin((double)(nc * odts), pnc_gcw);
            nc_acc -= pnc_gcw;
          }
        }
      }

      // M:1938-1959 snow and graupel collecting aerosols, wet scavenging
      if (AERO && TR::S && rs > ck.r_s1) {
        const float tc0 = fminf(-0.1f, temp - 273.15f);
        const float smoc_a = field_moment(tc0, ck.cse[0], smob), smoe_a = field_moment(tc0, ck.cse[12], smob);
        const float xDs = smoc_a / smob;
        float Ef_sa = eff_aero<'s'>(xDs, 0.04E-6f, visco, rho, temp);
        const double pna_sca = fmin((double)(nwfa * odts), (double)(rhof * ck.t1_qs_qc * Ef_sa * nwfa * smoe_a));
        Ef_sa = eff_aero<'s'>(xDs, 0.8E-6f, visco, rho, temp);
        const double pnd_scd = fmin((double)(nifa * odts), (double)(rhof * ck.t1_qs_qc * Ef_sa * nifa * smoe_a));
        na_acc += pna_sca; nd_acc += pnd_scd;
      }
      if (AERO && TR::G && rg > ck.r_g1) {
        const float xDg = (float)((double)(3.f + 0.f + 1.f) * ilamg);
        const double il9 = pow_d(ilamg, (double)ck.cge[8]);
        float Ef_ga = eff_aero<'g'>(xDg, 0.04E-6f, visco, rho, temp);
        const double pna_gca = fmin((double)(nwfa * odts), (double)(rhof * ck.t1_qg_qc * Ef_ga * nwfa) * N0_g * il9);
        Ef_ga = eff_aero<'g'>(xDg, 0.8E-6f, visco, rho, temp);
        const double pnd_gcd = fmin((double)(nifa * odts), (double)(rhof * ck.t1_qg_qc * Ef_ga * nifa) * N0_g * il9);
        na_acc += pna_gca; nd_acc += pnd_gcd;
      }

      // M:1964-2019 rain-snow and rain-graupel collection tables (interleaved records)
      if (TR::R && rr >= ck.r_r1) {
        if (rs >= ck.r_s1) {
          const double* rec = ck.racs + ((size_t)(idx_s - 1) + (size_t)NTB_S * ((idx_t - 1) + (size_t)NTB_T * ((idx_r1 - 1) + (size_t)NTB_R1 * (idx_r - 1)))) * S_N;
          const double tmr2 = rec[S_TMR_RACS2], tcr2 = rec[S_TCR_SACR2], tmr1 = rec[S_TMR_RACS1], tcr1 = rec[S_TCR_SACR1];
          const double tcs1 = rec[S_TCS_RACS1], tms1 = rec[S_TMS_SACR1];
          if (temp < T_0) {
            prr_rcs = -(tmr2 + tcr2 + tmr1 + tcr1);
            prs_rcs = tmr2 + tcr2 - tcs1 - tms1;
            prg_rcs = tmr1 + tcr1 + tcs1 + tms1;
            prr_rcs = fmax((double)(-rr * odts), prr_rcs);
            prs_rcs = fmax((double)(-rs * odts), prs_rcs);
            prg_rcs = fmin((double)((rr + rs) * odts), prg_rcs);
            pnr_rcs = rec[S_TNR_RACS1] + rec[S_TNR_RACS2] + rec[S_TNR_SACR1] + rec[S_TNR_SACR2];
          } else {
            prs_rcs = -tcs1 - tms1 + tmr2 + tcr2;
            prs_rcs = fmax((double)(-rs * odts), prs_rcs);
            prr_rcs = -prs_rcs;
            pnr_rcs = rec[S_TNR_RACS2] + rec[S_TNR_SACR2];
          }
          pnr_rcs = fmin((double)(nr * odts), pnr_rcs);
          nr_acc -= pnr_rcs;
        }
        if (TR::G && rg >= ck.r_g1) {
          const double* rec = ck.racg + ((size_t)(idx_g1 - 1) + (size_t)NTB_G1 * ((idx_g - 1) + (size_t)NTB_G * ((idx_r1 - 1) + (size_t)NTB_R1 * (idx_r - 1)))) * G_N;
          if (temp < T_0) {
            prg_rcg = rec[G_TMR_RACG] + rec[G_TCR_GACR];
            prg_rcg = fmin((double)(rr * odts), prg_rcg);
            prr_rcg = -prg_rcg;
            pnr_rcg = rec[G_TNR_RACG] + rec[G_TNR_GACR];
            pnr_rcg = fmin((double)(nr * odts), pnr_rcg);
            nr_acc -= pnr_rcg;
          } else {
            prr_rcg = rec[G_TCG_RACG];
            prr_rcg = fmin((double)(rg * odts), prr_rcg);
            prg_rcg = -prr_rcg;
            pnr_rcg = (double)-5.f * rec[G_TNR_GACR];
            nr_acc -= pnr_rcg;
          }
        }
      }

      if (TR::COLD || temp < T_0) {
        // ---- below freezing, M:2025-2231 ---------------------------------------------------
        vts_boost = 1.0f;
        const float rate_max = (qv - qvsi) * rho * odts * 0.999f;
        if (TR::R && rr > ck.r_r1) {
          const double* rec = ck.qrfz + ((size_t)(idx_r - 1) + (size_t)NTB_R * ((idx_r1 - 1) + (size_t)NTB_R1 * (idx_tc - 1))) * F_N;
          prg_rfz = rec[F_TPG] * (double)odts;
          pri_rfz = rec[F_TPI] * (double)odts;
          pni_rfz = rec[F_TNI] * (double)odts;
          pnr_rfz = rec[F_TNR] * (double)odts;
          pnr_rfz = fmin((double)(nr * odts), pnr_rfz);
          nr_acc -= pnr_rfz; ni_acc += pni_rfz;
        } else if (TR::R && rr > R1 && temp < KP_HGFR) {
          pri_rfz = (double)(rr * odts);
          pnr_rfz = (double)(nr * odts);
          pni_rfz = pnr_rfz;
          nr_acc -= pnr_rfz; ni_acc += pni_rfz;
        }
        if (TR::C && rc > ck.r_c1) {
          const double* rec = ck.qcfz + ((size_t)(idx_c - 1) + (size_t)NTB_C * (idx_tc - 1)) * C_N;
          pri_wfz = rec[C_TPI] * (double)odts;
          pri_wfz = fmin((double)(rc * odts), pri_wfz);
          pni_wfz = rec[C_TNI] * (double)odts;
          pni_wfz = fmin(fmin((double)(Nt_c * odts), pri_wfz / (double)(2.f * KP_XM0I)), pni_wfz);
          ni_acc += pni_wfz; nc_acc -= pni_wfz;
        } else if (TR::C && rc > R1 && temp < KP_HGFR) {
          pri_wfz = (double)(rc * odts);
          pni_wfz = (double)(nc * odts);
          ni_acc += pni_wfz; nc_acc -= pni_wfz;
        }
        // M:2090-2101 Cooper nucleation
        if ((ssati >= 0.25f) || (ssatw > EPSF && temp < 253.15f)) {
          const float xnc = AERO ? ice_demott(tempc, rho, nifa)                       // dustyIce, M:2092-2093
                                 : fminf(250.E3f, KP_TNO * exp_f(KP_ATO * (T_0 - temp)));
          const float xni = (float)((double)ni + (pni_rfz + pni_wfz) * (double)DT);
          pni_inu = (double)(0.5f * (xnc - xni + fabsf(xnc - xni)) * odts);
          pri_inu = fmin((double)rate_max, (double)KP_XM0I * pni_inu);
          pni_inu = (pri_inu == 0.0) ? pri_inu : pri_inu / (double)KP_XM0I;      // (a zero keeps its sign either way)
          ni_acc += pni_inu;
        }
        // M:2104-2111 freezing of aqueous aerosols (Koop et al. 2001); the 0th snow moment as at M:1557-1560
        if (AERO && temp < 238.f && ssati >= 0.4f) {
          float smo0_a = 0.f;
          if (L_qs) {
            const float tc0 = fminf(-0.1f, temp - 273.15f);
            const float* sa = c_sa; const float* sb = c_sb;
            const float loga_ = sa[1] + sa[2] * tc0 + sa[5] * tc0 * tc0 + sa[9] * tc0 * tc0 * tc0;
            const float b_ = sb[1] + sb[2] * tc0 + sb[5] * tc0 * tc0 + sb[9] * tc0 * tc0 * tc0;
            smo0_a = pow10_f(loga_) * pow_f(smob, b_);
          }
          const float xni = (float)((double)(smo0_a + ni) + (pni_rfz + pni_wfz + pni_inu) * (double)DT);
          if (xni <= 500.E3f) {
            const float xnc = ice_koop(temp, qv, qvs, nwfa, DT);
            pni_iha = (double)(xnc * odts);
            pri_iha = fmin((double)rate_max, (double)(KP_XM0I * 0.1f) * pni_iha);
            pni_iha = pri_iha / (double)(KP_XM0I * 0.1f);
            ni_acc += pni_iha;
          }
        }
        // M:2116-2149 deposition / sublimation of cloud ice, ice -> snow
        float oxmi = 0.f, xDi = 0.f;
        if (L_qi) {
          if (lami_stale) lami = ice_lam(ni, ri);
          ilami = (double)1.f / lami;
          xDi = (float)fmax((double)ck.D0i, (double)(3.f + 0.f + 1.f) * ilami);
          const float xmi = ck.am_i * cube_f(xDi);
          oxmi = 1.f / xmi;
          pri_ide = (double)(KP_C_CUBE * t1_subl * diffu * ssati * rvs * ck.oig1 * ck.cig[4] * ni) * ilami;
          const double* rec = ck.iaus + ((size_t)(idx_i - 1) + (size_t)NTB_I * (idx_i1 - 1)) * I_N;
          if (pri_ide < 0.0) {
            pri_ide = fmax(fmax((double)(-ri * odts), pri_ide), (double)rate_max);
            pni_ide = pri_ide * (double)oxmi;
            pni_ide = fmax((double)(-ni * odts), pni_ide);
          } else {
            pri_ide = fmin(pri_ide, (double)rate_max);
            prs_ide = (1.0 - rec[I_TPI_IDE]) * pri_ide;
            pri_ide = rec[I_TPI_IDE] * pri_ide;
          }
          if ((idx_i == NTB_I) || (xDi > 5.0f * D0s)) {
            prs_iau = (double)(ri * .99f * odts);
            pni_iau = (double)(ni * .95f * odts);
          } else if (xDi < 0.1f * D0s) {
            prs_iau = 0.; pni_iau = 0.;
          } else {
            prs_iau = rec[I_TPS] * (double)odts;
            prs_iau = fmin((double)(ri * .99f * odts), prs_iau);
            pni_iau = rec[I_TNI] * (double)odts;
            pni_iau = fmin((double)(ni * .95f * odts), pni_iau);
          }
          ni_acc -= pni_iau;
        }
        // M:2153-2175 deposition / sublimation of snow, sublimation of graupel
        if (L_qs) {
          float C_snow = KP_C_SQRD + (tempc + 1.5f) * (KP_C_CUBE - KP_C_SQRD) / (-30.f + 1.5f);
          C_snow = fmaxf(KP_C_SQRD, fminf(C_snow, KP_C_CUBE));
          prs_sde = (double)(C_snow * t1_subl * diffu * ssati * rvs
                             * (ck.t1_qs_sd * smo1 + ck.t2_qs_sd * rhof2 * vsc2 * smof));
          if (prs_sde < 0.) prs_sde = fmax(fmax((double)(-rs * odts), prs_sde), (double)rate_max);
          else prs_sde = fmin(prs_sde, (double)rate_max);
        }
        if (TR::G && L_qg && ssati < -EPSF) {
          prg_gde = (double)(KP_C_CUBE * t1_subl * diffu * ssati * rvs) * N0_g
                    * ((double)ck.t1_qg_sd * sq_d(ilamg)
                       + (double)(ck.t2_qg_sd * vsc2 * rhof2) * pow_d(ilamg, (double)ck.cge[10]));
          if (prg_gde < 0.) prg_gde = fmax(fmax((double)(-rg * odts), prg_gde), (double)rate_max);
          else prg_gde = fmin(prg_gde, (double)rate_max);
        }
        // M:2178-2202 snow and rain collecting cloud ice (lami/xDi/oxmi as recomputed at M:2179-2183)
        if (L_qi) {
          if (rs >= ck.r_s1) {
            if (!have_smoe) smoe = field_moment(fminf(-0.1f, temp - 273.15f), ck.cse[12], smob);
            prs_sci = (double)(ck.t1_qs_qi * rhof * KP_EF_SI * ri * smoe);
            pni_sci = prs_sci * (double)oxmi;
            ni_acc -= pni_sci;
          }
          if (TR::R && rr >= ck.r_r1 && mvd_r > 4.f * xDi) {
            lamr = (double)1.f / ilamr;
            const double lf = lamr + (double)KP_FV_R;
            const double lf2 = lf * lf, lf4 = 1.0 / (lf2 * lf2), lf7 = 1.0 / (lf2 * lf2 * lf2 * lf);
            pri_rci = (double)(rhof * ck.t1_qr_qi * KP_EF_RI * ri) * N0_r * lf4;
            pnr_rci = (double)(rhof * ck.t1_qr_qi * KP_EF_RI * ni) * N0_r * lf4;
            pni_rci = pri_rci * (double)oxmi;
            nr_acc -= pnr_rci; ni_acc -= pni_rci;
            prr_rci = (double)(rhof * ck.t2_qr_qi * KP_EF_RI * ni) * N0_r * lf7;       // cre(8) = 7
            prr_rci = fmin((double)(rr * odts), prr_rci);
            prg_rci = pri_rci + prr_rci;
          }
        }
        // M:2205-2218 Hallett-Mossop
        if (TR::C && TR::G && prg_gcw > (double)EPSF && tempc > -8.0f) {
          float tf = 0.f;
          if (tempc >= -5.0f && tempc < -3.0f) tf = 0.5f * (-3.0f - tempc);
          else if (tempc > -8.0f && tempc < -5.0f) tf = 0.33333333f * (8.0f + tempc);
          pni_ihm = (double)(3.5E8f * tf) * prg_gcw;
          pri_ihm = (double)KP_XM0I * pni_ihm;
          ni_acc += pni_ihm;
          prs_ihm = prs_scw / (prs_scw + prg_gcw) * pri_ihm;
          prg_ihm = prg_gcw / (prs_scw + prg_gcw) * pri_ihm;
        }
        // M:2224-2231 rimed snow -> graupel
        if (TR::C && prs_scw > (double)2.0f * prs_sde && prs_sde > (double)EPSF) {
          const float r_frac = (float)fmin(30.0, prs_scw / prs_sde);
          const float g_frac = fminf(0.95f, 0.15f + (r_frac - 2.f) * .028f);
          vts_boost = fminf(1.5f, 1.1f + (r_frac - 2.f) * .016f);
          prg_scw = (double)g_frac * prs_scw;
          prs_scw = (double)(1.f - g_frac) * prs_scw;
        }
      } else if (!TR::COLD) {
        // ---- at or above freezing, M:2237-2281 ----------------------------------------------
        float delQvs = 0.f;                                                // M:1508, read by the melting terms only
        if (L_qs || L_qg) delQvs = fmaxf(0.0f, rslf(pres, 273.15f) - qv);
        if (L_qs) {
          prr_sml = (double)((tempc * tcond - KP_LVAP0 * diffu * delQvs)
                             * (ck.t1_qs_me * smo1 + ck.t2_qs_me * rhof2 * vsc2 * smof));
          prr_sml = prr_sml + (double)(4218.f * ck.olfus * tempc) * (prr_rcs + prs_scw);
          prr_sml = fmin((double)(rs * odts), fmax(0., prr_sml));
          {                                          // 0th moment, M:1557-1560
            const float tc0 = fminf(-0.1f, temp - 273.15f);
            const float* sa = c_sa; const float* sb = c_sb;
            const float loga_ = sa[1] + sa[2] * tc0 + sa[5] * tc0 * tc0 + sa[9] * tc0 * tc0 * tc0;
            const float b_ = sb[1] + sb[2] * tc0 + sb[5] * tc0 * tc0 + sb[9] * tc0 * tc0 * tc0;
            smo0 = pow10_f(loga_) * pow_f(smob, b_);
          }
          pnr_sml = (double)(smo0 / rs) * prr_sml * (double)pow10_f(-0.25f * tempc);
          pnr_sml = fmin((double)(smo0 * odts), pnr_sml);
          nr_acc += pnr_sml;
          if (ssati < 0.f) {
            prs_sde = (double)(KP_C_CUBE * t1_subl * diffu * ssati * rvs
                               * (ck.t1_qs_sd * smo1 + ck.t2_qs_sd * rhof2 * vsc2 * smof));
            prs_sde = fmax((double)(-rs * odts), prs_sde);
          }
        }
        if (TR::G && L_qg) {
          const double il10 = sq_d(ilamg), il11 = pow_d(ilamg, (double)ck.cge[10]);
          prr_gml = (double)(tempc * tcond - KP_LVAP0 * diffu * delQvs) * N0_g
                    * ((double)ck.t1_qg_me * il10 + (double)(ck.t2_qg_me * rhof2 * vsc2) * il11);
          prr_gml = fmin((double)(rg * odts), fmax(0., prr_gml));
          pnr_gml = N0_g * (double)ck.cgg[1] * ilamg / (double)rg * prr_gml * (double)pow10_f(-0.5f * tempc);
          nr_acc += pnr_gml;
          if (ssati < 0.f) {
            prg_gde = (double)(KP_C_CUBE * t1_subl * diffu * ssati * rvs) * N0_g
                      * ((double)ck.t1_qg_sd * il10 + (double)(ck.t2_qg_sd * vsc2 * rhof2) * il11);
            prg_gde = fmax((double)(-rg * odts), prg_gde);
          }
        }
        if (DT > 120.f) {
          prr_rcw = prr_rcw + prs_scw + prg_gcw;
          prs_scw = 0.; prg_gcw = 0.;
        }
      }
    }

    LOCKBAR(2);
    // ---- S7, M:2291-2387 conservation limiters -----------------------------------------------
    // (a group is compiled for a class only when one of its rates can be non-zero there; the flag of the species guards it)
    {
      float sump, rate_max;
      if (TR::ICEPROC) {
        sump = (float)(pri_inu + pri_ide + prs_ide + prs_sde + prg_gde + pri_iha);
        rate_max = (qv - qvsi) * odts * 0.999f;                                // U7: no rho factor here
        if ((sump > EPSF && sump > rate_max) || (sump < -EPSF && sump < rate_max)) {
          const double ratio = (double)(rate_max / sump);
          pri_inu *= ratio; pri_ide *= ratio; pni_ide *= ratio; prs_ide *= ratio; prs_sde *= ratio;
          if (TR::G) prg_gde *= ratio;
          if (AERO) pri_iha *= ratio;
        }
      }
      if (TR::C) {
        sump = (float)(-prr_wau - pri_wfz - prr_rcw - prs_scw - prg_scw - prg_gcw);
        rate_max = -rc * odts;
        if (sump < rate_max && L_qc) {
          const double ratio = (double)(rate_max / sump);
          prr_wau *= ratio;
          if (TR::R) prr_rcw *= ratio;
          if (TR::ICEPROC) { pri_wfz *= ratio; prs_scw *= ratio; prg_scw *= ratio; }
          if (TR::G) prg_gcw *= ratio;
        }
      }
      if (TR::I) {
        sump = (float)(pri_ide - prs_iau - prs_sci - pri_rci);
        rate_max = -ri * odts;
        if (sump < rate_max && L_qi) {
          const double ratio = (double)(rate_max / sump);
          pri_ide *= ratio; prs_iau *= ratio; prs_sci *= ratio;
          if (TR::R) pri_rci *= ratio;
        }
      }
      if (TR::R) {
        sump = (float)(-prg_rfz - pri_rfz - prr_rci + prr_rcs + prr_rcg);
        rate_max = -rr * odts;
        if (sump < rate_max && L_qr) {
          const double ratio = (double)(rate_max / sump);
          if (TR::ICEPROC) { prg_rfz *= ratio; pri_rfz *= ratio; prr_rci *= ratio; prr_rcs *= ratio; prr_rcg *= ratio; }
        }
      }
      if (TR::S) {
        sump = (float)(prs_sde - prs_ihm - prr_sml + prs_rcs);
        rate_max = -rs * odts;
        if (sump < rate_max && L_qs) {
          const double ratio = (double)(rate_max / sump);
          prs_sde *= ratio; prs_ihm *= ratio; prr_sml *= ratio;
          if (TR::R) prs_rcs *= ratio;
        }
      }
      if (TR::G) {
        sump = (float)(prg_gde - prg_ihm - prr_gml + prg_rcg);
        rate_max = -rg * odts;
        if (sump < rate_max && L_qg) {
          const double ratio = (double)(rate_max / sump);
          prg_gde *= ratio; prg_ihm *= ratio; prr_gml *= ratio;
          if (TR::R) prg_rcg *= ratio;
        }
      }
      pri_ihm = prs_ihm + prg_ihm;
      if (TR::R && TR::G) {
        float ratio = (float)fmin(fabs(prr_rcg), fabs(prg_rcg));
        prr_rcg = (double)(ratio * copysignf(1.0f, (float)prr_rcg));
        prg_rcg = -prr_rcg;
      }
      if (TR::R && TR::S && temp > T_0) {
        float ratio = (float)fmin(fabs(prr_rcs), fabs(prs_rcs));
        prr_rcs = (double)(ratio * copysignf(1.0f, (float)prr_rcs));
        prs_rcs = -prr_rcs;
      }
    }

    // U1 again (nc1d = 0 without cloud water, M:1409)
    const float nc1d = AERO ? nc1d_in : ((qc1d > R1) ? Nt_c / (0.622f * pres / (KP_R * t1d * (qv1d + 0.622f))) : 0.0f);
    float nwfat = 0.f, nifat = 0.f;
    // ---- S8, M:2393-2569 tendencies and number/mass balances ------------------------------------
    float tt, qvt, qct, qit, qrt, qst, qgt, nit, nrt, nct;
    {
      const float orho = 1.f / rho;
      const float lfus2 = KP_LSUB - lvap;
      if (AERO) {                                          // M:2398-2408 (dustyIce)
        nwfat = (float)((double)0.f - (na_acc + pni_iha) * (double)orho);
        nifat = (float)((double)0.f - nd_acc * (double)orho);
        nifat = (float)((double)nifat - pni_inu * (double)orho);
      }
      qvt = (float)((-pri_inu - pri_iha - pri_ide - prs_ide - prs_sde - prg_gde) * (double)orho);
      qct = (float)((-prr_wau - pri_wfz - prr_rcw - prs_scw - prg_scw - prg_gcw) * (double)orho);
      nct = (float)(nc_acc * (double)orho);
      float xrc = fmaxf(R1, (qc1d + qct * DT) * rho);
      float xnc = fmaxf(2.f, (nc1d + nct * DT) * rho);
      if (TR::C && xrc > R1) {
        const int nu = min(15, nint_f(1000.E6f / xnc) + 2);
        const double lc = (double)pow_f(xnc * ck.am_r * ck.ccg[1][nu - 1] * ck.ocg1[nu - 1] / rc, ck.obmr);
        const float xD = (float)((double)(3.f + (float)nu + 1.f) / lc);
        if (xD < D0c) {
          const double l2 = (double)(ck.cce[1][nu - 1] / D0c);
          xnc = (float)((double)(ck.ccg[0][nu - 1] * ck.ocg2[nu - 1] * xrc / ck.am_r) * cube_d(l2));
          nct = (xnc - nc1d * rho) * odts * orho;
        } else if (xD > D0r * 2.f) {
          const double l2 = (double)(ck.cce[1][nu - 1] / (D0r * 2.f));
          xnc = (float)((double)(ck.ccg[0][nu - 1] * ck.ocg2[nu - 1] * xrc / ck.am_r) * cube_d(l2));
          nct = (xnc - nc1d * rho) * odts * orho;
        }
      } else {
        nct = -nc1d * odts;
      }
      xnc = fmaxf(0.f, (nc1d + nct * DT) * rho);
      if (xnc > KP_NT_C_MAX) nct = (KP_NT_C_MAX - nc1d * rho) * odts * orho;

      qit = (float)((pri_inu + pri_iha + pri_ihm + pri_wfz + pri_rfz + pri_ide - prs_iau - prs_sci - pri_rci) * (double)orho);
      nit = (float)((ni_acc + pni_ide) * (double)orho);
      const float xri = fmaxf(R1, (qi1d + qit * DT) * rho);
      float xni = fmaxf(R2, (ni1d + nit * DT) * rho);
      if (TR::I9 && xri > R1) {
        lami = ice_lam(xni, xri);
        ilami = (double)1.f / lami;
        const float xD = (float)((double)(3.f + 0.f + 1.f) * ilami);
        if (xD < 5.E-6f) {
          lami = (double)(ck.cie[1] / 5.E-6f);
          xni = (float)fmin(499.E3, (double)(ck.cig[0] * ck.oig2 * xri / ck.am_i) * cube_d(lami));
          nit = (xni - ni1d * rho) * odts * orho;
        } else if (xD > 300.E-6f) {
          lami = (double)(ck.cie[1] / 300.E-6f);
          xni = (float)((double)(ck.cig[0] * ck.oig2 * xri / ck.am_i) * cube_d(lami));
          nit = (xni - ni1d * rho) * odts * orho;
        }
      } else {
        nit = -ni1d * odts;
      }
      xni = fmaxf(0.f, (ni1d + nit * DT) * rho);
      if (xni > 499.E3f) nit = (499.E3f - ni1d * rho) * odts * orho;

      qrt = (float)((prr_wau + prr_rcw + prr_sml + prr_gml + prr_rcs + prr_rcg - prg_rfz - pri_rfz - prr_rci) * (double)orho);
      nrt = (float)(nr_acc * (double)orho);
      const float xrr = fmaxf(R1, (qr1d + qrt * DT) * rho);
      float xnr = fmaxf(R2, (nr1d + nrt * DT) * rho);
      if (TR::R9 && xrr > R1) {
        lamr = rain_lam(xnr, xrr);
        mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr);
        if (mvd_r > 2.5E-3f) {
          mvd_r = 2.5E-3f;
          xnr = nr_from_mvd(xrr, mvd_r);
          nrt = (xnr - nr1d * rho) * odts * orho;
        } else if (mvd_r < D0r * 0.75f) {
          mvd_r = D0r * 0.75f;
          xnr = nr_from_mvd(xrr, mvd_r);
          nrt = (xnr - nr1d * rho) * odts * orho;
        }
      } else {
        qrt = -qr1d * odts;
        nrt = -nr1d * odts;
      }
      qst = (float)((prs_iau + prs_sde + prs_sci + prs_scw + prs_rcs + prs_ide - prs_ihm - prr_sml) * (double)orho);
      qgt = (float)((prg_scw + prg_rfz + prg_gde + prg_rcg + prg_gcw + prg_rci + prg_rcs - prg_ihm - prr_gml) * (double)orho);
      if (TR::COLD || temp < T_0) {
        tt = (float)(((double)(KP_LSUB * ocp) * (pri_inu + pri_ide + prs_ide + prs_sde + prg_gde + pri_iha)
                      + (double)(lfus2 * ocp) * (pri_wfz + pri_rfz + prg_rfz + prs_scw + prg_scw + prg_gcw + prg_rcs
                                                 + prs_rcs + prr_rci + prg_rcg))
                     * (double)orho * (double)1);
      } else {
        tt = (float)(((double)(ck.lfus * ocp) * (-prr_sml - prr_gml - prr_rcg - prr_rcs)
                      + (double)(KP_LSUB * ocp) * (prs_sde + prg_gde))
                     * (double)orho * (double)1);
      }
    }

    // M:2963-3120 the rates KiD saves with save_dg that are final here (optional buffer [36][nz][ld]); the three of S11 /
    // S12 follow below
    if (RATES && valid) {
      float* rp = a.rates + o;
      const long st = (long)nz * ld;
      const double rv[30] = {pri_inu, pri_ide, prs_ide, prs_sde, prg_gde, pri_wfz, prs_scw, prg_scw, prg_gcw, pri_ihm,
                             pri_rfz, prs_iau, prs_sci, pri_rci, pni_inu, pni_ihm, pni_wfz, pni_rfz, pni_ide, pni_iau,
                             pni_sci, pni_rci, prr_sml, prr_gml, pnr_rcs, pnr_rcg, pnr_rci, pnr_sml, pnr_gml, pnr_rfz};
#pragma unroll
      for (int q = 0; q < 30; ++q) rp[q * st] = (float)rv[q];
      rp[30 * st] = (float)prr_wau; rp[31 * st] = (float)prr_rcw; rp[33 * st] = (float)pnr_wau; rp[35 * st] = (float)pnr_rcr;
    }
    const bool melted_graupel = TR::G && prr_gml > 0.0;      // M:2940 reads prr_gml after the limiters

    LOCKBAR(3);
    // ---- S9, M:2574-2656 state at tau+1 -------------------------------------------------------
    float lvt2;
    {
      temp = t1d + DT * tt;
      const float otemp = 1.f / temp;
      tempc = temp - 273.15f;
      qv = fmaxf(1.E-10f, qv1d + DT * qvt);
      rho = 0.622f * pres / (KP_R * temp * (qv + 0.622f));
      qvs = rslf(pres, temp);
      ssatw = qv / qvs - 1.f;
      if (fabsf(ssatw) < EPSF) ssatw = 0.0f;
      // rhof, rhof2, diffu, visco, vsc2, tcond of M:2588-2600 are read by rain evaporation (which evaluates them
      // again from the post-condensation state here, S12) and the fall speeds (rhof, S13) only
      lvap = KP_LVAP0 + (2106.0f - 4218.0f) * tempc;
      ocp = 1.f / (KP_CP * (1.f + 0.887f * qv));
      lvt2 = lvap * lvap * ocp * ck.oRv * otemp * otemp;

      if (AERO) nwfa = fmaxf(11.1E6f, (nwfa1d + nwfat * DT) * rho);                          // M:2597
      if (TR::C9 && (qc1d + qct * DT) > R1) { rc = (qc1d + qct * DT) * rho; nc = AERO ? fmaxf(2.f, (nc1d + nct * DT) * rho) : Nt_c; L_qc = true; }
      else { rc = R1; nc = 2.f; L_qc = false; }
      if (TR::I9 && (qi1d + qit * DT) > R1) { ri = (qi1d + qit * DT) * rho; ni = fmaxf(R2, (ni1d + nit * DT) * rho); L_qi = true; }
      else { ri = R1; ni = R2; L_qi = false; }
      if (TR::R9 && (qr1d + qrt * DT) > R1) {
        rr = (qr1d + qrt * DT) * rho;
        nr = fmaxf(R2, (nr1d + nrt * DT) * rho);
        L_qr = true;
        lamr = rain_lam(nr, rr);
        lamr_stale = false;
        mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr);
        if (mvd_r > 2.5E-3f) { mvd_r = 2.5E-3f; nr = nr_from_mvd(rr, mvd_r); lamr_stale = true; }
        else if (mvd_r < D0r * 0.75f) { mvd_r = D0r * 0.75f; nr = nr_from_mvd(rr, mvd_r); lamr_stale = true; }
      } else { rr = R1; nr = R2; L_qr = false; }
      if (TR::S9 && (qs1d + qst * DT) > R1) { rs = (qs1d + qst * DT) * rho; L_qs = true; } else { rs = R1; L_qs = false; }
      if (TR::G9 && (qg1d + qgt * DT) > R1) { rg = (qg1d + qgt * DT) * rho; L_qg = true; } else { rg = R1; L_qg = false; }
    }

    // ---- S10, M:2662-2750 snow moments and intercepts again -------------------------------------
    bool warm9 = false;
    double n0b_lo = n0_empty, n0b_slw = n0_empty;
    if (!iiwarm) {
      if (TR::S9 && L_qs) {
        const float tc0 = fminf(-0.1f, temp - 273.15f);
        smob = rs * ck.oams;
        smoc = field_moment(tc0, ck.cse[0], smob);
        // smod (M:2706-2717) is not read again by any live code
      }
      // M:2721-2731: whether this level lies above k_0 depends on the updated temperatures of the levels above,
      // which k_finish knows: both values of the intercept are handed to it (they differ only with supercooled rain),
      // and it evaluates the slope, which only the graupel fall speed of S13 reads
      warm9 = temp >= 270.65f;
      if (TR::G9) n0b_lo = (rg > 5.E-5f) ? graupel_n0_exp(0.01f, rg) : n0_empty;
      // (k_finish only reads the second one above k_0, i.e. where no level from here up has reached 270.65 K)
      n0b_slw = (TR::R9 && !warm9 && L_qr && mvd_r > 100.E-6f) ? graupel_n0_exp(4.01f + log10_f(mvd_r), rg) : n0b_lo;
    }
    if (TR::R9 && L_qr) {                                                   // M:2750-2755, as at M:1661
      if (lamr_stale) { lamr = rain_lam(nr, rr); mvd_r = (float)((double)(3.0f + 0.f + 0.672f) / lamr); lamr_stale = false; }
      ilamr = (double)1.f / lamr;
      N0_r = (double)(nr * ck.org2) * lamr;
    }

    LOCKBAR(4);
    // ---- S11, M:2780-2874 cloud condensation / evaporation ---------------------------------------
    if ((ssatw > EPSF) || (ssatw < -EPSF && L_qc)) {
      const float orho = 1.f / rho;
      float clap = (qv - qvs) / (1.f + lvt2 * qvs);
#pragma unroll
      for (int it = 0; it < 3; ++it) {
        const float ex = exp_f(lvt2 * clap);
        const float fcd = qvs * ex - qv + clap;
        const float dfcd = qvs * lvt2 * ex + 1.f;
        clap = clap - fcd / dfcd;
      }
      const float xrc = rc + clap * rho;
      if (xrc > R1) {
        prw_vcd = (double)(clap * odt);
        if (clap > EPSF) {
          const float xnc = AERO ? fmaxf(2.f, activ_ncloud(temp, w1d, nwfa)) : Nt_c;
          pnc_wcd = (double)(0.5f * (xnc - nc + fabsf(xnc - nc)) * odts * orho);
        } else if (AERO && clap < -EPSF && ssatw < -1.E-6f) {
          // M:2804-2851 the droplets smaller than Dc_star evaporate (table_dropEvap); diffu, tcond of S9 (M:2588-2593)
          const float tc9 = temp - 273.15f, otemp = 1.f / temp, oRv = ck.oRv;
          const float diffu9 = 2.11E-5f * pow_f(temp / 273.15f, 1.94f) * (101325.f / pres);
          const float tcond9 = (5.69f + 0.0168f * tc9) * 1.0E-5f * 418.936f;
          const float rvs = rho * qvs;
          const float rvs_p = rvs * otemp * (lvap * otemp * oRv - 1.f);
          const float rvs_pp = rvs * (otemp * (lvap * otemp * oRv - 1.f) * otemp * (lvap * otemp * oRv - 1.f)
                                      + (-2.f * lvap * otemp * otemp * otemp * oRv) + otemp * otemp);
          const float gamsc = lvap * diffu9 / tcond9 * rvs_p;
          float alphsc = 0.5f * (gamsc / (1.f + gamsc)) * (gamsc / (1.f + gamsc)) * rvs_pp / rvs_p * rvs / rvs_p;
          alphsc = fmaxf(1.E-9f, alphsc);
          float xsat = ssatw;
          if (fabsf(xsat) < 1.E-9f) xsat = 0.f;
          const float t1_evap = 2.f * KP_PI * (1.0f - alphsc * xsat + 2.f * alphsc * alphsc * xsat * xsat
                                               - 5.f * alphsc * alphsc * alphsc * xsat * xsat * xsat) / (1.f + gamsc);
          const double Dc_star = sqrt(-2.0 * (double)DT * (double)t1_evap / (double)(2.f * KP_PI) * 4.0 * (double)diffu9 * (double)ssatw
                                      * (double)rvs / (double)KP_RHO_W);
          const int idx_d = max(1, min((int)(1.E6 * Dc_star), (int)NBINS));
          int idx_n = nint_d(1.0 + (double)(float)NBINS * dlog((double)nc / ck.t_Nc1) / (double)ck.nic1);
          idx_n = max(1, min(idx_n, (int)NBINS));
          const int idx_c = (rc > ck.r_c1) ? decade_idx_f(rc, ck.nic2, NTB_C) : 1;
          prw_vcd = fmax((double)(-rc * 0.99f * orho * odt), prw_vcd);
          const double tnc = ck.tnc_wev[(size_t)(idx_d - 1) + (size_t)NBINS * ((idx_c - 1) + (size_t)NTB_C * (idx_n - 1))];
          pnc_wcd = fmax((double)(-nc * 0.99f * orho * odt), (double)(-tnc * (double)orho * (double)odt));
        }
      } else {
        prw_vcd = (double)(-rc * orho * odt);
        pnc_wcd = (double)(-nc * orho * odt);
      }
      qvt = (float)((double)qvt - prw_vcd);
      qct = (float)((double)qct + prw_vcd);
      nct = (float)((double)nct + pnc_wcd);
      if (AERO) nwfat = (float)((double)nwfat - pnc_wcd);
      tt = (float)((double)tt + (double)(lvap * ocp) * prw_vcd * (double)1);
      rc = fmaxf(R1, (qc1d + DT * qct) * rho);
      nc = AERO ? fmaxf(2.f, (nc1d + DT * nct) * rho) : Nt_c;
      qv = fmaxf(1.E-10f, qv1d + DT * qvt);
      temp = t1d + DT * tt;
      rho = 0.622f * pres / (KP_R * temp * (qv + 0.622f));
      qvs = rslf(pres, temp);
      ssatw = qv / qvs - 1.f;
    }

    // ---- S12, M:2880-2960 rain evaporation -------------------------------------------------------
    if (TR::R9 && (ssatw < -EPSF) && L_qr && (!(prw_vcd > 0.))) {
      tempc = temp - 273.15f;
      const float otemp = 1.f / temp;
      const float orho = 1.f / rho;
      rhof = sqrtf(ck.rho_not * orho);
      rhof2 = sqrtf(rhof);
      diffu = 2.11E-5f * pow_f(temp / 273.15f, 1.94f) * (101325.f / pres);
      visco = (tempc >= 0.0f) ? (1.718f + 0.0049f * tempc) * 1.0E-5f
                              : (1.718f + 0.0049f * tempc - 1.2E-5f * tempc * tempc) * 1.0E-5f;
      vsc2 = sqrtf(rho / visco);
      lvap = KP_LVAP0 + (2106.0f - 4218.0f) * tempc;
      tcond = (5.69f + 0.0168f * tempc) * 1.0E-5f * 418.936f;
      ocp = 1.f / (KP_CP * (1.f + 0.887f * qv));
      const float oRv = ck.oRv;
      const float rvs = rho * qvs;
      const float rvs_p = rvs * otemp * (lvap * otemp * oRv - 1.f);
      const float rvs_pp = rvs * (otemp * (lvap * otemp * oRv - 1.f) * otemp * (lvap * otemp * oRv - 1.f)
                                  + (-2.f * lvap * otemp * otemp * otemp * oRv) + otemp * otemp);
      const float gamsc = lvap * diffu / tcond * rvs_p;
      float alphsc = 0.5f * (gamsc / (1.f + gamsc)) * (gamsc / (1.f + gamsc)) * rvs_pp / rvs_p * rvs / rvs_p;
      alphsc = fmaxf(1.E-9f, alphsc);
      const float xsat = fminf(-1.E-9f, ssatw);
      const float t1_evap = 2.f * KP_PI * (1.0f - alphsc * xsat + 2.f * alphsc * alphsc * xsat * xsat
                                           - 5.f * alphsc * alphsc * alphsc * xsat * xsat * xsat) / (1.f + gamsc);
      const double lamr_ev = (double)1.f / ilamr;
      if (qv / qvs < 0.95f && rr * orho <= 1.E-8f) {
        prv_rev = (double)(rr * orho * odts);
      } else {
        const double lh = lamr_ev + (double)(0.5f * KP_FV_R);
        prv_rev = (double)(t1_evap * diffu * (-ssatw)) * N0_r * (double)rvs
                  * ((double)ck.t1_qr_ev * sq_d(ilamr)                                     // ilamr**cre(10), = 2
                     + (double)(ck.t2_qr_ev * vsc2 * rhof2) * (1.0 / (lh * lh * lh)));      // **(-cre(11)), = 3
        const float rate_max = fminf((rr * orho * odts), (qvs - qv) * odts);
        prv_rev = fmin((double)rate_max, prv_rev * (double)orho);
        if (melted_graupel) {
          const float eva_factor = fminf(1.0f, 0.01f + (0.99f - 0.01f) * (tempc / 20.0f));
          prv_rev = prv_rev * (double)eva_factor;
        }
      }
      pnr_rev = fmin((double)(nr * 0.99f * orho * odts), prv_rev * (double)nr / (double)rr);
      qrt = (float)((double)qrt - prv_rev);
      qvt = (float)((double)qvt + prv_rev);
      nrt = (float)((double)nrt - pnr_rev);
      if (AERO) nwfat = (float)((double)nwfat + pnr_rev);                                   // M:2952
      tt = (float)((double)tt - (double)(lvap * ocp) * prv_rev * (double)1);
      rr = fmaxf(R1, (qr1d + DT * qrt) * rho);
      qv = fmaxf(1.E-10f, qv1d + DT * qvt);
      nr = fmaxf(R2, (nr1d + DT * nrt) * rho);
      lamr_stale = true;
      temp = t1d + DT * tt;
      rho = 0.622f * pres / (KP_R * temp * (qv + 0.622f));
    }
    if (RATES && valid) {
      float* rp = a.rates + o;
      const long st = (long)nz * ld;
      rp[32 * st] = (float)prv_rev; rp[34 * st] = (float)pnr_rev;
    }

    LOCKBAR(5);
    // ---- S13, M:3206-3354 the cell's own fall speeds (k_finish applies what runs down the column) -------
    rhof = sqrtf(ck.rho_not / rho);
    float v_r = 0.f, v_nr = 0.f, v_i = 0.f, v_ni = 0.f, vts_h = 0.f;
    if (TR::R9 && rr > R1) {
      if (!L_qr || lamr_stale) lamr = rain_lam(nr, rr);                   // M:3227: same nr, rr as at M:2750 otherwise
      const double lf = lamr + (double)KP_FV_R;
      const double l2 = lamr * lamr, lf2 = lf * lf;
      // lamr**cre(3) * (lamr+fv_r)**(-cre(6)), cre(3) = 4, cre(6) = 5
      v_r = (float)((double)(rhof * KP_AV_R * ck.crg[5] * ck.org3) * (l2 * l2) * (1.0 / (lf2 * lf2 * lf)));
      // lamr**cre(12) * (lamr+fv_r)**(-cre(7)), cre(12) = 2.5, cre(7) = 3.5
      v_nr = (float)((double)(rhof * KP_AV_R * ck.crg[6] / ck.crg[11]) * (l2 * sqrt(lamr)) * (1.0 / (lf2 * lf * sqrt(lf))));
    }
    if (TR::ICEPROC && !iiwarm) {
      if (TR::I9 && ri > R1) {
        lami = ice_lam(ni, ri);
        ilami = (double)1.f / lami;
        v_i = (float)((double)(rhof * KP_AV_I * ck.cig[2] * ck.oig2) * ilami);               // ilami**bv_i, bv_i = 1
        v_ni = (float)((double)(rhof * KP_AV_I * ck.cig[5] / ck.cig[6]) * ilami);
      }
      if (TR::S9 && rs > R1) {
        const float xDs = smoc / smob;
        const float Mrat = 1.f / xDs;
        float ils1 = 1.f / (Mrat * KP_LAM0 + KP_FV_S);
        float ils2 = 1.f / (Mrat * KP_LAM1 + KP_FV_S);
        const float mm = pow_f(Mrat, KP_MU_S);
        const float t1_vts = KP_KAP0 * ck.csg[3] * pow_f(ils1, ck.cse[3]);
        const float t2_vts = KP_KAP1 * mm * ck.csg[9] * pow_f(ils2, ck.cse[9]);
        ils1 = 1.f / (Mrat * KP_LAM0);
        ils2 = 1.f / (Mrat * KP_LAM1);
        const float t3_vts = KP_KAP0 * ck.csg[0] * pow_f(ils1, ck.cse[0]);
        const float t4_vts = KP_KAP1 * mm * ck.csg[6] * pow_f(ils2, ck.cse[6]);
        vts_h = rhof * KP_AV_S * (t1_vts + t2_vts) / (t3_vts + t4_vts);   // M:3301 needs the rain speed after the rule of M:3235: k_finish
      }
    }

    // hand-off.  S15 (M:3584-3606) needs lfus*ocp where the level ends above T_0 and lfus2*ocp where it ends
    // below HGFR (never both): one signed value carries the product and the case.
    if (valid) {
      float s15 = 0.0f;
      if (temp > T_0) s15 = ck.lfus * ocp;
      else if (temp < KP_HGFR) s15 = -((KP_LSUB - lvap) * ocp);
      // the sign of the first intercept carries the k_0 test of this level's updated temperature (intercepts are > 0)
      const float n0a_out = warm9 ? -(float)n0b_lo : (float)n0b_lo;
      // two 64-byte half records, four whole sectors, SC_* order
      if (COMPACT && KC == KC_WARM) {
        st_sector(sc, tt, qvt, qct, qrt, nrt, nct, nr, 0.f);
        st_sector(sb, rr, ri, rs, rg, v_r, v_nr, v_i, rho);
      } else if (COMPACT) {
        st_sector(sc, tt, qvt, qct, qit, qst, nit, nct, ni);
        st_sector(sb, rr, ri, rs, rg, v_r, v_ni, v_i, rho);     // (no rain in this class: the word of its number speed carries v_ni)
      } else {
        st_sector(sc, tt, qvt, qct, qit, qrt, qst, qgt, nit);
        st_sector(sc + 8, nrt, nct, nr, ni, v_ni, nwfat, nifat, 0.f);
        st_sector(sb, rr, ri, rs, rg, v_r, v_nr, v_i, rho);
      }
      st_sector(sb + 8, s15, n0a_out, (float)n0b_slw, vts_h, vts_boost, temp, 0.f, 0.f);
      // An upper bound of every fall speed this cell can hand a level of its column, for the test "no species of this column
      // needs a second sedimentation sub-step" (k_carries): its own speeds (a level without the species inherits them, M:3235);
      // melting snow (M:3301) through the factor vts / (T - T_0) that multiplies the inherited rain speed.  Graupel takes its
      // speed from the running intercept minimum of the column (M:2731, M:3328): a column with graupel is never simple.
      float vb = fmaxf(fmaxf(v_r, v_nr), v_i);
      if (TR::S9 && rs > R1) {
        vb = fmaxf(vb, vts_h * vts_boost);
        if (temp > (T_0 + 0.1f)) atomicMax(a.colvmax + a.ncol + slot, __float_as_int(vts_h / (temp - T_0)));
      }
      if (TR::G9 && rg > R1) vb = __int_as_float(0x7f800000);
      if (vb > 1.E-3f) atomicMax(a.colvmax + slot, __float_as_int(vb));
    }
  }
#undef LOCKBAR
}

// ---- K2: what runs down the column, then S14 sedimentation (M:3365-3578), S15 instant melt / freeze (M:3584-3606) and
// S16 (M:3623-3686).  One thread per cloudy column (slot), one warp per block.
// (SoA workspace of the columns with sub-steps: plane [nz][ws_cols], lane = column)
__device__ __forceinline__ void sed_substeps(float* __restrict__ r, float* __restrict__ rten, const float* __restrict__ v,
                                             float* __restrict__ n, float* __restrict__ nten, const float* __restrict__ vn,
                                             const float* __restrict__ rhoa, const float* __restrict__ dz, long dzs, int nz, long cs,
                                             int nsub, int ksed, float onstep, float DT, bool on, float nfloor, float& ppt) {
  for (int it = 0; it < nsub; ++it) {
    float sr_up = 0.f, sn_up = 0.f, sr_k = 0.f, r0 = 0.f;
#pragma unroll 1
    for (int k = nz - 1; k >= 0; --k) {
      const long o = (long)k * cs;
      const float rk = r[o];
      const float sr = on ? v[o] * rk : 0.f;
      const float odzq = 1.f / dz[k * dzs], orho = 1.f / rhoa[o];
      float nk = 0.f, sn = 0.f;
      if (n) { nk = n[o]; sn = on ? vn[o] * nk : 0.f; }
      if (k == nz - 1) {
        rten[o] = rten[o] - sr * odzq * onstep * orho;
        r0 = fmaxf(KP_R1, rk - sr * odzq * DT * onstep);
        r[o] = r0;
        if (n) { nten[o] = nten[o] - sn * odzq * onstep * orho; n[o] = fmaxf(nfloor, nk - sn * odzq * DT * onstep); }
      } else if (k + 1 <= ksed) {
        rten[o] = rten[o] + (sr_up - sr) * odzq * onstep * orho;
        r0 = fmaxf(KP_R1, rk + (sr_up - sr) * odzq * DT * onstep);
        r[o] = r0;
        if (n) { nten[o] = nten[o] + (sn_up - sn) * odzq * onstep * orho; n[o] = fmaxf(nfloor, nk + (sn_up - sn) * odzq * DT * onstep); }
      } else {
        r0 = rk;
      }
      sr_up = sr; sn_up = sn; sr_k = sr;
    }
    if (r0 > KP_R1 * 10.f) ppt = ppt + sr_k * DT * onstep;
  }
}

// busy bit of level k from the words loaded so far (words of 32 levels, [nwords][count])
#define BUSY_WORD(w) a.busy[(size_t)(w) * count + slot]

// ---- K2a: what runs down the column after the cell kernels: the intercept minimum of S10 (M:2721-2731), the fall speed of a
// level without the species (M:3235, M:3267, M:3307, M:3333), snow above 0 C and graupel (they need the rain speed after
// that rule, M:3301, M:3328), the sub-step counts and top sedimenting levels (M:3242, M:3208).  One thread per cloudy
// column; all the values of a busy cell are loaded in one batch (one memory round trip per level).  Leaves colint
// [8][count] and the list of the columns that need sedimentation sub-steps.
__global__ void __launch_bounds__(64, 16) k_carries(StepArgs a) {
  const int slot = blockIdx.x * 64 + threadIdx.x;
  const int count = *a.work_count;
  if (slot >= count) return;
  const long col = a.work_list[slot];
  const int nz = a.nz;
  const long ld = a.ld;
  const long cs = count;
  const float DT = a.dt;
  const bool iiwarm = ck.iiwarm != 0;
  const double n0_empty = g_n0_lo;
  const unsigned* const cidx = a.cellidx + slot;
  const float* const dzp = a.dz_col ? a.dz_col + col : a.dz;     // one vector shared by all columns (KiD) or this column's own (WRF entry)
  const long dzs = a.dz_col ? ld : 1;
  {
    // A SIMPLE column: no fall speed of the column can cross its thinnest layer in one step (bounds left by the cell kernels),
    // so every sub-step count of M:3242 is 0 or 1 - k_finish then settles what runs down the column on its own single sweep
    // and this kernel has nothing to read.  (v DT < 0.99 dz makes INT(DT / (dz / v) + 1.) = 1 whatever the roundings.)
    const float vmax = __int_as_float(a.colvmax[slot]), sfac = __int_as_float(a.colvmax[a.ncol + slot]);
    if (vmax <= 3.0e38f && !a.no_simple) {                // (+inf: graupel in the column)
      float dzmin = dzp[0];
      for (int k = 1; k < nz; ++k) dzmin = fminf(dzmin, dzp[k * dzs]);
      if (fmaxf(vmax, sfac * vmax) * DT < 0.99f * dzmin) { a.colint[slot] = -1; return; }
    }
  }
  int nstep_r = 0, nstep_i = 0, nstep_s = 0, nstep_g = 0, ksed_r = 1, ksed_i = 1, ksed_s = 1, ksed_g = 1;
  double n0_min = (double)KP_GONV_MAX;
  bool warm_b = false;
  float v_r = 0.f, v_nr = 0.f, v_i = 0.f, v_s = 0.f, v_g = 0.f;     // speeds of the level above (the ice number speed sets no count, M:3267)
  unsigned bw = 0;
  // record numbers two levels ahead, the record of the next level on its way to L2 (the index of an idle cell is never used)
  unsigned idx_next = cidx[(size_t)(nz - 1) * cs], idx_next2 = cidx[(size_t)(nz - 2) * cs];
#pragma unroll 1
  for (int k = nz - 1; k >= 0; --k) {
    if (k == nz - 1 || (k & 31) == 31) bw = BUSY_WORD(k >> 5);
    const unsigned idx = idx_next;
    idx_next = idx_next2;
    if (k > 1) idx_next2 = cidx[(size_t)(k - 2) * cs];
    if ((k & 31) != 0 && ((bw >> ((k - 1) & 31)) & 1u)) prefetch_record(a.scratch_b + (size_t)idx_next * SC_HALF);
    float* sc = a.scratch_b + (size_t)idx * SC_HALF - 16;       // (SC_* offsets of the second half start at 16)
    const float dzq = dzp[k * dzs];
    if ((bw >> (k & 31)) & 1u) {
      // the second half of the record (two sectors) holds everything this kernel reads
      const Sector s2 = ld_sector(sc + 16);
      const float rr = s2.v[0], o_vr = s2.v[4], o_vnr = s2.v[5];
      if (!iiwarm) {
        const Sector s3 = ld_sector(sc + 24);
        const float ri = s2.v[1], rs = s2.v[2], rg = s2.v[3];
        const float x1 = s3.v[1], x2 = s3.v[2];
        const float o_vi = s2.v[6];
        const float vts = s3.v[3], vts_boost = s3.v[4], temp = s3.v[5];
        const float rho = s2.v[7], s15 = s3.v[0];
        if (rr > R1) { v_r = o_vr; v_nr = o_vnr; }
        if (x1 < 0.f) warm_b = true;
        const double N0_exp = (!warm_b && k > 0) ? (double)x2 : (double)fabsf(x1);
        n0_min = fmin(N0_exp, n0_min);
        if (ri > R1) v_i = o_vi;
        if (rs > R1) {
          if (temp > (T_0 + 0.1f)) v_s = fmaxf(vts * vts_boost, vts * ((v_r - vts * vts_boost) / (temp - T_0)));
          else v_s = vts * vts_boost;
          sc[SC_VTS] = v_s;
        }
        if (rg > R1) {
          const float rhof = sqrtf(ck.rho_not / rho);
          double ilamg = 0., N0_g = 0.;
          graupel_slope(n0_min, rg, ilamg, N0_g);
          const float vtg = (float)((double)(rhof * KP_AV_G * ck.cgg[5] * ck.ogg3) * pow_d(ilamg, (double)KP_BV_G));
          v_g = (s15 > 0.f) ? fmaxf(vtg, v_r) : vtg;         // temp > T_0 is what makes the S15 factor positive
          sc[SC_VTG] = v_g;
        }
      } else if (rr > R1) { v_r = o_vr; v_nr = o_vnr; }
    } else if (!iiwarm) {
      if (!warm_b && a.f[F_T][(long)k * ld + col] >= 270.65f) warm_b = true;      // an idle cell keeps its temperature
      n0_min = fmin(n0_empty, n0_min);
    }
    if (fmaxf(v_r, v_nr) > 1.E-3f) {
      ksed_r = max(ksed_r, k + 1);
      const float delta_tp = dzq / (fmaxf(v_r, v_nr));
      nstep_r = max(nstep_r, (int)(DT / delta_tp + 1.f));
    }
    if (!iiwarm) {
      if (v_i > 1.E-3f) { ksed_i = max(ksed_i, k + 1); const float d = dzq / v_i; nstep_i = max(nstep_i, (int)(DT / d + 1.f)); }
      if (v_s > 1.E-3f) { ksed_s = max(ksed_s, k + 1); const float d = dzq / v_s; nstep_s = max(nstep_s, (int)(DT / d + 1.f)); }
      if (v_g > 1.E-3f) { ksed_g = max(ksed_g, k + 1); const float d = dzq / v_g; nstep_g = max(nstep_g, (int)(DT / d + 1.f)); }
    }
  }
  // U12: the reference leaves the sub-step count unbounded (M:3242); on non-physical input (dt*v/dz in the
  // millions) that is a kernel that never ends, so it is capped where no real case comes near
  nstep_r = min(nstep_r, KP_NSTEP_MAX); nstep_i = min(nstep_i, KP_NSTEP_MAX);
  nstep_s = min(nstep_s, KP_NSTEP_MAX); nstep_g = min(nstep_g, KP_NSTEP_MAX);
  int* ci = a.colint + slot;
  ci[0] = nstep_r; ci[cs] = nstep_i; ci[2 * cs] = nstep_s; ci[3 * cs] = nstep_g;
  ci[4 * cs] = ksed_r; ci[5 * cs] = ksed_i; ci[6 * cs] = ksed_s; ci[7 * cs] = ksed_g;
  if (max(max(nstep_r, nstep_i), max(nstep_s, nstep_g)) > 1) a.sub_list[atomicAdd(a.sub_count, 1)] = slot;
}

// per-column sedimentation parameters out of colint (M:3208, M:3242, M:3365-3578)
struct SedCounts { int n_r, n_i, n_s, n_g, ksed_r, ksed_i, ksed_s, ksed_g; float on_r, on_i, on_s, on_g; };
__device__ __forceinline__ SedCounts sed_counts(const int* ci, long cs, int nz) {
  SedCounts s;
  const int nstep_r = ci[0], nstep_i = ci[cs], nstep_s = ci[2 * cs], nstep_g = ci[3 * cs];
  s.ksed_r = ci[4 * cs]; s.ksed_i = ci[5 * cs]; s.ksed_s = ci[6 * cs]; s.ksed_g = ci[7 * cs];
  const int kte = nz;
  if (s.ksed_r == kte) s.ksed_r = kte - 1;
  if (s.ksed_i == kte) s.ksed_i = kte - 1;
  if (s.ksed_s == kte) s.ksed_s = kte - 1;
  if (s.ksed_g == kte) s.ksed_g = kte - 1;
  s.on_r = nstep_r > 0 ? 1.f / (float)nstep_r : 1.0f; s.on_i = nstep_i > 0 ? 1.f / (float)nstep_i : 1.0f;
  s.on_s = nstep_s > 0 ? 1.f / (float)nstep_s : 1.0f; s.on_g = nstep_g > 0 ? 1.f / (float)nstep_g : 1.0f;
  s.n_r = nint_f(1.f / s.on_r); s.n_i = nint_f(1.f / s.on_i); s.n_s = nint_f(1.f / s.on_s); s.n_g = nint_f(1.f / s.on_g);
  return s;
}

// the record of an idle cell: all rates zero, state unchanged, contents R1 / R2 (speeds: those of the level above)
__device__ __forceinline__ void idle_record(float temp, float pres, float qv1d, float& rho, float& s15) {
  const float qv = fmaxf(1.E-10f, qv1d);
  const float tempc = temp - 273.15f;
  const float ocp = 1.f / (KP_CP * (1.f + 0.887f * qv));
  const float lvap = KP_LVAP0 + (2106.0f - 4218.0f) * tempc;
  rho = 0.622f * pres / (KP_R * temp * (qv + 0.622f));
  s15 = 0.0f;
  if (temp > T_0) s15 = ck.lfus * ocp;
  else if (temp < KP_HGFR) s15 = -((KP_LSUB - lvap) * ocp);
}

// ---- K2b: the columns that need sedimentation sub-steps (nstep > 1, M:3242), on their compacted list: full warps.  Such a
// column needs a record for every level (mass falls into idle cells) and is swept once per sub-step, so it is first
// gathered into an SoA workspace [WS_N][nz][ws_cols] (lane = column: every access of the sub-steps is one line per warp):
// the records of its busy cells, the zero record of its idle cells, and at every level the speeds that k_carries settled.
// Then all but the last sub-step of each species (M:3365-3578), then the last one with S15 / S16 (finish_level), as k_finish
// does for the other columns.  Runs beside k_finish on a second stream: the two kernels own different columns.
enum { WS_TTEN = 0, WS_QVTEN, WS_QCTEN, WS_QITEN, WS_QRTEN, WS_QSTEN, WS_QGTEN, WS_NITEN, WS_NRTEN, WS_NCTEN,
       WS_RR, WS_NR, WS_RI, WS_NI, WS_RS, WS_RG, WS_VTR, WS_VTNR, WS_VTI, WS_VTNI, WS_VTS, WS_VTG, WS_RHO, WS_S15, WS_NWFAT, WS_NIFAT, WS_N };
template <bool RATES, bool AERO>
__global__ void __launch_bounds__(32, 16) k_substeps(StepArgs a) {
  const int n = *a.sub_count, count = *a.work_count;
  const unsigned k1_list = (unsigned)a.cell_kstart[KC_ICE], k2_list = (unsigned)a.cell_kstart[KC_MIXNR];
  const int nz = a.nz;
  const long ld = a.ld, ncol = a.ncol;
  const long cs = a.ws_cols;
  const size_t ps = (size_t)nz * cs;
  const float DT = a.dt, odt = 1.f / DT;
  const bool iiwarm = ck.iiwarm != 0;
  const bool sedi = ck.l_sediment != 0;
#pragma unroll 1
  for (int j = blockIdx.x * 32 + threadIdx.x; j < n; j += gridDim.x * 32) {
    const int slot = a.sub_list[j];
    const long col = a.work_list[slot];
    const SedCounts s = sed_counts(a.colint + slot, count, nz);
    const unsigned* const cidx = a.cellidx + slot;
    const float* const dzp = a.dz_col ? a.dz_col + col : a.dz;
    const long dzs = a.dz_col ? ld : 1;
    float* const w0 = a.ws + j;
    {
      float v_r = 0.f, v_nr = 0.f, v_i = 0.f, v_ni = 0.f, v_s = 0.f, v_g = 0.f;
      unsigned bw = 0;
#pragma unroll 1
      for (int k = nz - 1; k >= 0; --k) {
        if (k == nz - 1 || (k & 31) == 31) bw = BUSY_WORD(k >> 5);
        float* w = w0 + (size_t)k * cs;
        if ((bw >> (k & 31)) & 1u) {
          const unsigned idx = cidx[(size_t)k * count];
          const float* qb = a.scratch_b + (size_t)idx * SC_HALF;
          const Sector s2 = ld_sector(qb), s3 = ld_sector(qb + 8);
          const RecA ra = load_rec_a<AERO>(a, idx, k1_list, k2_list, s2);
          w[WS_TTEN * ps] = ra.tt; w[WS_QVTEN * ps] = ra.qvt; w[WS_QCTEN * ps] = ra.qct; w[WS_QITEN * ps] = ra.qit;
          w[WS_QRTEN * ps] = ra.qrt; w[WS_QSTEN * ps] = ra.qst; w[WS_QGTEN * ps] = ra.qgt; w[WS_NITEN * ps] = ra.nit;
          w[WS_NRTEN * ps] = ra.nrt; w[WS_NCTEN * ps] = ra.nct; w[WS_NR * ps] = ra.nr; w[WS_NI * ps] = ra.ni;
          w[WS_RR * ps] = s2.v[0]; w[WS_RI * ps] = s2.v[1]; w[WS_RS * ps] = s2.v[2]; w[WS_RG * ps] = s2.v[3];
          w[WS_RHO * ps] = s2.v[7]; w[WS_S15 * ps] = s3.v[0];
          if (AERO) { w[WS_NWFAT * ps] = ra.nwfat; w[WS_NIFAT * ps] = ra.nifat; }
          if (s2.v[0] > R1) { v_r = s2.v[4]; v_nr = s2.v[5]; }
          if (!iiwarm) {
            if (s2.v[1] > R1) { v_i = s2.v[6]; v_ni = ra.v_ni; }
            if (s2.v[2] > R1) v_s = s3.v[6];
            if (s2.v[3] > R1) v_g = s3.v[7];
          }
        } else {
          const long o = (long)k * ld + col;
          float rho, s15;
          idle_record(a.f[F_T][o], a.p[o], a.f[F_QV][o], rho, s15);
#pragma unroll
          for (int q = WS_TTEN; q <= WS_NCTEN; ++q) w[q * ps] = 0.0f;
          w[WS_RR * ps] = R1; w[WS_NR * ps] = R2; w[WS_RI * ps] = R1; w[WS_NI * ps] = R2; w[WS_RS * ps] = R1; w[WS_RG * ps] = R1;
          w[WS_RHO * ps] = rho; w[WS_S15 * ps] = s15;
          if (AERO) { w[WS_NWFAT * ps] = 0.0f; w[WS_NIFAT * ps] = 0.0f; }
        }
        w[WS_VTR * ps] = v_r; w[WS_VTNR * ps] = v_nr; w[WS_VTI * ps] = v_i; w[WS_VTNI * ps] = v_ni;
        w[WS_VTS * ps] = v_s; w[WS_VTG * ps] = v_g;
      }
    }
    const float* rhoa = w0 + WS_RHO * ps;
    float ppt_r = 0.f, ppt_i = 0.f, ppt_s = 0.f, ppt_g = 0.f;
    // all but the last sub-step (rain is never gated by l_sediment, U6; the cloud-water stub M:3414-3425 is a no-op, U2)
    if (s.n_r > 1) sed_substeps(w0 + WS_RR * ps, w0 + WS_QRTEN * ps, w0 + WS_VTR * ps, w0 + WS_NR * ps, w0 + WS_NRTEN * ps,
                                w0 + WS_VTNR * ps, rhoa, dzp, dzs, nz, cs, s.n_r - 1, s.ksed_r, s.on_r, DT, true, KP_R2, ppt_r);
    if (s.n_i > 1) sed_substeps(w0 + WS_RI * ps, w0 + WS_QITEN * ps, w0 + WS_VTI * ps, w0 + WS_NI * ps, w0 + WS_NITEN * ps,
                                w0 + WS_VTNI * ps, rhoa, dzp, dzs, nz, cs, s.n_i - 1, s.ksed_i, s.on_i, DT, sedi, KP_R2, ppt_i);
    if (s.n_s > 1) sed_substeps(w0 + WS_RS * ps, w0 + WS_QSTEN * ps, w0 + WS_VTS * ps, nullptr, nullptr, nullptr, rhoa, dzp, dzs,
                                nz, cs, s.n_s - 1, s.ksed_s, s.on_s, DT, sedi, 0.f, ppt_s);
    if (s.n_g > 1) sed_substeps(w0 + WS_RG * ps, w0 + WS_QGTEN * ps, w0 + WS_VTG * ps, nullptr, nullptr, nullptr, rhoa, dzp, dzs,
                                nz, cs, s.n_g - 1, s.ksed_g, s.on_g, DT, sedi, 0.f, ppt_g);
    // last sub-step of every species + S15 + S16, one top-down sweep
    SedParams sp;
    sp.DT = DT; sp.odt = odt; sp.on_r = s.on_r; sp.on_i = s.on_i; sp.on_s = s.on_s; sp.on_g = s.on_g; sp.Nt_c = ck.Nt_c;
    sp.top_r = s.ksed_r; sp.top_i = s.ksed_i; sp.top_s = s.ksed_s; sp.top_g = s.ksed_g; sp.sedi = sedi; sp.iiwarm = iiwarm;
    SedCarry c;
    c.sr_up = 0.f; c.snr_up = 0.f; c.si_up = 0.f; c.sni_up = 0.f; c.ss_up = 0.f; c.sg_up = 0.f;
    c.ppt_r = ppt_r; c.ppt_i = ppt_i; c.ppt_s = ppt_s; c.ppt_g = ppt_g; c.lwp = 0.0; c.iwp = 0.0;
    unsigned bw = 0;
#pragma unroll 1
    for (int k = nz - 1; k >= 0; --k) {
      if (k == nz - 1 || (k & 31) == 31) bw = BUSY_WORD(k >> 5);
      const long o = (long)k * ld + col;
      const float* q = w0 + (size_t)k * cs;
      HandOff h;
      h.tt = q[WS_TTEN * ps]; h.qvt = q[WS_QVTEN * ps]; h.qct = q[WS_QCTEN * ps]; h.qit = q[WS_QITEN * ps];
      h.qrt = q[WS_QRTEN * ps]; h.qst = q[WS_QSTEN * ps]; h.qgt = q[WS_QGTEN * ps]; h.nit = q[WS_NITEN * ps];
      h.nrt = q[WS_NRTEN * ps]; h.nct = q[WS_NCTEN * ps];
      h.rho = q[WS_RHO * ps]; h.s15 = q[WS_S15 * ps];
      h.nwfat = AERO ? q[WS_NWFAT * ps] : 0.f; h.nifat = AERO ? q[WS_NIFAT * ps] : 0.f;
      h.rr = q[WS_RR * ps]; h.nr = q[WS_NR * ps]; h.ri = q[WS_RI * ps]; h.ni = q[WS_NI * ps]; h.rs = q[WS_RS * ps]; h.rg = q[WS_RG * ps];
      h.v_r = q[WS_VTR * ps]; h.v_nr = q[WS_VTNR * ps]; h.v_i = q[WS_VTI * ps]; h.v_ni = q[WS_VTNI * ps];
      h.v_s = q[WS_VTS * ps]; h.v_g = q[WS_VTG * ps];
      if (RATES && !((bw >> (k & 31)) & 1u)) {           // an idle cell: every process rate is zero
        float* rp = a.rates + o;
        const long st = (long)nz * ld;
        for (int r = 0; r < KIDMP_NRATES; ++r) rp[r * st] = 0.0f;
      }
      finish_level<AERO>(a, sp, c, h, k, nz, o, dzp[k * dzs], a.f[F_T][o], a.f[F_QV][o], a.f[F_QC][o], a.f[F_QI][o], a.f[F_QR][o],
                   a.f[F_QS][o], a.f[F_QG][o], a.f[F_NI][o], a.f[F_NR][o], a.p[o]);
    }
    // ppt is overwritten with this step's amounts: rain, ice, snow, graupel (I:55-58, I:162-177)
    a.ppt[col] = c.ppt_r; a.ppt[ld + col] = c.ppt_i; a.ppt[2 * ld + col] = c.ppt_s; a.ppt[3 * ld + col] = c.ppt_g;
    a.coldiag[col] = c.lwp; a.coldiag[ncol + col] = c.iwp;      // summed in column order by k_diag_columns
  }
}

// ---- K2c: the columns without sub-steps: the only sub-step of every species (M:3365-3578) + S15 instant melt / freeze
// (M:3584-3606) + S16 (M:3623-3686), one top-down sweep per column, one warp per block.  The ten inputs and the record of a busy
// level are loaded in one batch; an idle level has no record: its tendencies are zero and its contents R1 / R2.
#ifndef K2_MINB
#define K2_MINB 20
#endif
template <bool RATES, bool AERO>
__global__ void __launch_bounds__(32, K2_MINB) k_finish(StepArgs a) {
  const int slot = blockIdx.x * 32 + threadIdx.x;
  const int count = *a.work_count;
  if (slot >= count) return;
  const unsigned k1_list = (unsigned)a.cell_kstart[KC_ICE], k2_list = (unsigned)a.cell_kstart[KC_MIXNR];
  const int nz = a.nz;
  const long cs = count;
  // A simple column (k_carries: no graupel, every sub-step count 0 or 1) has no counts: what runs down the column - the speed
  // of snow above 0 C (M:3301), the top sedimenting levels (M:3208) - is settled level by level on this sweep, with the
  // expressions of k_carries.
  const bool simple = a.colint[slot] < 0;
  SedCounts s;
  if (simple) {
    s.n_r = s.n_i = s.n_s = s.n_g = 1; s.on_r = s.on_i = s.on_s = s.on_g = 1.0f;
    s.ksed_r = s.ksed_i = s.ksed_s = s.ksed_g = 1;                    // (M:3208: ksed1 starts at 1; raised below as the sweep meets the species)
  } else {
    s = sed_counts(a.colint + slot, cs, nz);
    if (s.n_r > 1 || s.n_i > 1 || s.n_s > 1 || s.n_g > 1) return;    // k_substeps has this column
  }
  const long col = a.work_list[slot];
  const long ld = a.ld, ncol = a.ncol;
  const float DT = a.dt, odt = 1.f / DT;
  const bool iiwarm = ck.iiwarm != 0;
  const unsigned* const cidx = a.cellidx + slot;
  const float* const dzp = a.dz_col ? a.dz_col + col : a.dz;
  const long dzs = a.dz_col ? ld : 1;
  SedParams sp;
  sp.DT = DT; sp.odt = odt; sp.on_r = s.on_r; sp.on_i = s.on_i; sp.on_s = s.on_s; sp.on_g = s.on_g; sp.Nt_c = ck.Nt_c;
  sp.top_r = s.ksed_r; sp.top_i = s.ksed_i; sp.top_s = s.ksed_s; sp.top_g = s.ksed_g; sp.sedi = ck.l_sediment != 0; sp.iiwarm = iiwarm;
  SedCarry c;
  c.sr_up = 0.f; c.snr_up = 0.f; c.si_up = 0.f; c.sni_up = 0.f; c.ss_up = 0.f; c.sg_up = 0.f;
  c.ppt_r = 0.f; c.ppt_i = 0.f; c.ppt_s = 0.f; c.ppt_g = 0.f; c.lwp = 0.0; c.iwp = 0.0;
  float v_r = 0.f, v_nr = 0.f, v_i = 0.f, v_ni = 0.f, v_s = 0.f, v_g = 0.f;       // speeds of the level above
  unsigned bw = 0;
  // record numbers two levels ahead, the record of the next level on its way to L2 (the index of an idle cell is never used)
  unsigned idx_next = cidx[(size_t)(nz - 1) * cs], idx_next2 = cidx[(size_t)(nz - 2) * cs];
#pragma unroll 1
  for (int k = nz - 1; k >= 0; --k) {
    if (k == nz - 1 || (k & 31) == 31) bw = BUSY_WORD(k >> 5);
    const long o = (long)k * ld + col;
    const unsigned idx = idx_next;
    const float* qb = a.scratch_b + (size_t)idx * SC_HALF;
    idx_next = idx_next2;
    if (k > 1) idx_next2 = cidx[(size_t)(k - 2) * cs];
    if ((k & 31) != 0 && ((bw >> ((k - 1) & 31)) & 1u)) {
      prefetch_record(rec_a_ptr<AERO>(a, idx_next, k2_list)); prefetch_record(a.scratch_b + (size_t)idx_next * SC_HALF);
    }
    const bool busy = ((bw >> (k & 31)) & 1u) != 0;
    const float t1d = a.f[F_T][o], qv1d = a.f[F_QV][o], qc1d = a.f[F_QC][o], qi1d = a.f[F_QI][o], qr1d = a.f[F_QR][o],
                qs1d = a.f[F_QS][o], qg1d = a.f[F_QG][o], ni1d = a.f[F_NI][o], nr1d = a.f[F_NR][o], pres = a.p[o];
    HandOff h;
    if (busy) {
      const Sector s2 = ld_sector(qb), s3 = ld_sector(qb + 8);   // the two half records
      const RecA ra = load_rec_a<AERO>(a, idx, k1_list, k2_list, s2);
      h.tt = ra.tt; h.qvt = ra.qvt; h.qct = ra.qct; h.qit = ra.qit; h.qrt = ra.qrt; h.qst = ra.qst; h.qgt = ra.qgt; h.nit = ra.nit;
      h.nrt = ra.nrt; h.nct = ra.nct; h.nr = ra.nr; h.ni = ra.ni;
      h.rr = s2.v[0]; h.ri = s2.v[1]; h.rs = s2.v[2]; h.rg = s2.v[3];
      h.rho = s2.v[7]; h.s15 = s3.v[0];
      h.nwfat = ra.nwfat; h.nifat = ra.nifat;
      if (h.rr > R1) { v_r = s2.v[4]; v_nr = s2.v[5]; }
      if (!iiwarm) {
        if (h.ri > R1) { v_i = s2.v[6]; v_ni = ra.v_ni; }
        if (!simple) {
          if (h.rs > R1) v_s = s3.v[6];                   // (written by k_carries where the species is present)
          if (h.rg > R1) v_g = s3.v[7];
        } else if (h.rs > R1) {                           // (a simple column holds no graupel)
          const float vts = s3.v[3], vts_boost = s3.v[4], temp = s3.v[5];
          if (temp > (T_0 + 0.1f)) v_s = fmaxf(vts * vts_boost, vts * ((v_r - vts * vts_boost) / (temp - T_0)));
          else v_s = vts * vts_boost;
        }
      }
    } else {
      h.tt = 0.f; h.qvt = 0.f; h.qct = 0.f; h.qit = 0.f; h.qrt = 0.f; h.qst = 0.f; h.qgt = 0.f; h.nit = 0.f; h.nrt = 0.f; h.nct = 0.f;
      h.rr = R1; h.nr = R2; h.ri = R1; h.ni = R2; h.rs = R1; h.rg = R1;
      h.nwfat = 0.f; h.nifat = 0.f;
      idle_record(t1d, pres, qv1d, h.rho, h.s15);
      if (RATES) {                                        // an idle cell: every process rate is zero
        float* rp = a.rates + o;
        const long st = (long)nz * ld;
        for (int r = 0; r < KIDMP_NRATES; ++r) rp[r * st] = 0.0f;
      }
    }
    h.v_r = v_r; h.v_nr = v_nr; h.v_i = v_i; h.v_ni = v_ni; h.v_s = v_s; h.v_g = v_g;
    if (simple) {                                         // M:3208: the highest level with a fall speed, this level included
      if (fmaxf(v_r, v_nr) > 1.E-3f) sp.top_r = nz;
      if (!iiwarm) {
        if (v_i > 1.E-3f) sp.top_i = nz;
        if (v_s > 1.E-3f) sp.top_s = nz;
      }
    }
    finish_level<AERO>(a, sp, c, h, k, nz, o, dzp[k * dzs], t1d, qv1d, qc1d, qi1d, qr1d, qs1d, qg1d, ni1d, nr1d, pres);
  }
  // ppt is overwritten with this step's amounts: rain, ice, snow, graupel (I:55-58, I:162-177)
  a.ppt[col] = c.ppt_r; a.ppt[ld + col] = c.ppt_i; a.ppt[2 * ld + col] = c.ppt_s; a.ppt[3 * ld + col] = c.ppt_g;
  a.coldiag[col] = c.lwp; a.coldiag[ncol + col] = c.iwp;      // summed in column order by k_diag_columns
}
#undef BUSY_WORD

#undef R1
#undef R2
#undef EPSF
#undef T_0
#undef D0r
#undef D0c
#undef D0s
#undef D0g

}  // namespace kidmp
