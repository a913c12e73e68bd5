// device_probe.cu - test-only probe of the device helpers, point by point (tests/test_device_math.py).
//
// Includes the product headers unchanged and compiles with the library's flags (kid_b200/build.py BASE_FLAGS), so every
// helper below is the code the step kernels run: the same __constant__ coefficients, the same node tables (built on the
// host by kfm_build_tables and uploaded exactly as kidmp_init does), the same KConst (hostinit::compute), passed as a
// __grid_constant__ launch parameter like the step passes it.  One elementwise kernel: function id, up to five f64
// input arrays (f32 functions take their arguments rounded to f32, which is exact for f32 inputs), one f64 output array.
#include "kidmp_column.cuh"
#include "kidmp_aero.cuh"
#include "kidmp_hostinit.h"
#include <cstring>

using namespace kidmp;

enum {
  P_DEXP = 0, P_DLOG, P_DPOW, P_POW_F, P_EXP_F, P_LOG10_F, P_POW10_F, P_LOG_F, P_RSLF, P_RSIF,
  P_DECADE_F = 10, P_DECADE_D, P_FIELD_MOMENT, P_FIELD_LOGA, P_FIELD_B, P_GRAUPEL_N0, P_RAIN_LAM, P_ICE_LAM,
  P_EFF_R = 18, P_EFF_S, P_EFF_G, P_ICE_DEMOTT, P_ICE_KOOP, P_ACTIV_NCLOUD, P_N
};

__global__ void k_probe(const __grid_constant__ KConst ck, int fn, long n, const double* __restrict__ a,
                        const double* __restrict__ b, const double* __restrict__ c, const double* __restrict__ d,
                        const double* __restrict__ e, int i0, int i1, double* __restrict__ out) {
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const double A = a[t];
  const double B = b ? b[t] : 0.0, C = c ? c[t] : 0.0, D = d ? d[t] : 0.0, E = e ? e[t] : 0.0;
  const float fa = (float)A, fb = (float)B, fc = (float)C, fd = (float)D, fe = (float)E;
  double r = 0.0;
  switch (fn) {
    case P_DEXP: r = dexp(A); break;
    case P_DLOG: r = dlog(A); break;
    case P_DPOW: r = pow_d(A, B); break;
    case P_POW_F: r = pow_f(fa, fb); break;
    case P_EXP_F: r = exp_f(fa); break;
    case P_LOG10_F: r = log10_f(fa); break;
    case P_POW10_F: r = pow10_f(fa); break;
    case P_LOG_F: r = log_f(fa); break;
    case P_RSLF: r = rslf(fa, fb); break;
    case P_RSIF: r = rsif(fa, fb); break;
    case P_DECADE_F: r = decade_idx_f(ck, fa, i0, i1); break;
    case P_DECADE_D: r = decade_idx_d(ck, A, i0, i1); break;
    case P_FIELD_MOMENT: r = field_moment(fa, fb, fc); break;
    case P_FIELD_LOGA: { float la, bb; field_ab(fa, fb, la, bb); r = la; } break;
    case P_FIELD_B: { float la, bb; field_ab(fa, fb, la, bb); r = bb; } break;
    case P_GRAUPEL_N0: r = graupel_n0_exp(fa, fb); break;
    case P_RAIN_LAM: r = rain_lam(ck, fa, fb); break;
    case P_ICE_LAM: r = ice_lam(ck, fa, fb); break;
    case P_EFF_R: r = eff_aero<'r'>(fa, fb, fc, fd, fe); break;
    case P_EFF_S: r = eff_aero<'s'>(fa, fb, fc, fd, fe); break;
    case P_EFF_G: r = eff_aero<'g'>(fa, fb, fc, fd, fe); break;
    case P_ICE_DEMOTT: r = ice_demott(fa, fb, fc); break;
    case P_ICE_KOOP: r = ice_koop(fa, fb, fc, fd, fe); break;
    case P_ACTIV_NCLOUD: r = activ_ncloud(fa, fb, fc); break;
    default: r = __longlong_as_double(0x7ff8dead0000beefLL); break;
  }
  out[t] = r;
}

extern "C" {

long probe_kconst_size(void) { return (long)sizeof(KConst); }

// hostinit::compute into *out and the node tables of kidmp_fastmath.h into this module's g_exp_tab / g_log_tab, as
// kidmp_init does.  Returns a cudaError_t.
int probe_init(float set_Nc, int iiwarm, KConst* out) {
  kidmp_config cfg;
  memset(&cfg, 0, sizeof cfg);
  cfg.set_Nc = set_Nc;
  cfg.iiwarm = iiwarm;
  cfg.l_sediment = 1;
  memset(out, 0, sizeof *out);
  static HostBins hb;
  memset(&hb, 0, sizeof hb);
  hostinit::Prep pp;
  hostinit::compute(cfg, *out, hb, pp);
  static double et[KFM_N];
  static LogNode lt[KFM_N];
  kfm_build_tables(et, lt);
  cudaError_t e = cudaMemcpyToSymbol(g_exp_tab, et, sizeof et);
  if (e == cudaSuccess) e = cudaMemcpyToSymbol(g_log_tab, lt, sizeof lt);
  return (int)e;
}

// scalars of a KConst by name (the exponents and decade offsets the kernels pass); NaN for an unknown name
double probe_kconst(const KConst* k, const char* name) {
  struct { const char* n; double v; } t[] = {
      {"nic2", (double)k->nic2}, {"nii2", (double)k->nii2}, {"nii3", (double)k->nii3}, {"nir2", (double)k->nir2},
      {"nir3", (double)k->nir3}, {"nis2", (double)k->nis2}, {"nig2", (double)k->nig2}, {"nig3", (double)k->nig3},
      {"obmr", (double)k->obmr}, {"obmi", (double)k->obmi}, {"Sc3", (double)k->Sc3}, {"am_r", (double)k->am_r},
      {"am_i", (double)k->am_i}, {"crg2", (double)k->crg[2]}, {"org2", (double)k->org2}, {"cig1", (double)k->cig[1]},
      {"oig1", (double)k->oig1}, {"cse0", (double)k->cse[0]}, {"cse12", (double)k->cse[12]},
      {"cse15", (double)k->cse[15]}};
  for (auto& x : t) if (!strcmp(x.n, name)) return x.v;
  return __builtin_nan("");
}

// out[i] = f(a[i], b[i], ...) on `stream`; b..e may be NULL.  Returns a cudaError_t (launch errors only).
int probe_run(int fn, long n, const double* a, const double* b, const double* c, const double* d, const double* e,
              int i0, int i1, const KConst* k, double* out, void* stream) {
  if (fn < 0 || fn >= P_N || n < 0) return (int)cudaErrorInvalidValue;
  if (n == 0) return 0;
  const int bs = 256;
  k_probe<<<(unsigned)((n + bs - 1) / bs), bs, 0, (cudaStream_t)stream>>>(*k, fn, n, a, b, c, d, e, i0, i1, out);
  return (int)cudaGetLastError();
}

}  // extern "C"
