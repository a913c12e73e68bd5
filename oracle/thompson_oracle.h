// ORACLE — TEST INFRASTRUCTURE ONLY.
// CPU restatement of the reference Thompson scheme driven by KiD:
//   M: = /root/reference/module_mp_thompson09n.f90   I: = /root/reference/mphys_thompson09n.f90
// Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may
// load this library.  The product (kid_b200/) never includes, links or calls anything here.
//
// PARITY UNPINNED: the reference ships no tests, golden vectors or fixtures (SURVEY.md §4/§8c)
// and no Fortran compiler exists in the build container, so this restatement is pinned only by
// the source-derived known-answer values in tests/test_oracle_kat.py.
#pragma once
#ifdef __cplusplus
extern "C" {
#endif

typedef struct kor_handle kor_handle;

// M:374-797 thompson_init.  wp_double: kind of DFLOAT() at M:8 (0 = f32 default, U5).
// cache_path: optional binary cache for the two 4-D collection tables (may be NULL).
kor_handle* kor_create(float set_Nc, int iiwarm, int l_sediment, int wp_double,
                       const char* cache_path, int nthreads);
void kor_destroy(kor_handle*);
double kor_init_seconds(const kor_handle*);

// named access to constants and tables (column-major, Fortran order), returns element count or -1
long kor_table_size(const kor_handle*, const char* name);
long kor_get_table(const kor_handle*, const char* name, double* out, long n);

// M:1156-3688 mp_thompson for one column (arrays of nz, index 0 = kts).  nc may be NULL: then
// nc1d = Nt_c/rho as mp_gt_driver does (M:957-964, decision U1).  rates (optional) receives
// [36][nz] doubles in the order of kor_rate_names().
int kor_mp_thompson(const kor_handle*, int nz, float dt,
                    float* qv, float* qc, float* qi, float* qr, float* qs, float* qg,
                    float* ni, float* nr, float* nc, float* t,
                    const float* p, const float* dz, float* ppt4, double* rates);

// I:54-246 loop over columns.  layout 0: K_FASTEST a[col*nz+k] (KiD (k,i)); 1: COL_FASTEST
// a[k*ncol+col].  ppt is [4][ncol] (rain, ice, snow, graupel).  dz is one shared nz vector.
int kor_step(const kor_handle*, long ncol, int nz, float dt, int layout,
             float* qv, float* qc, float* qi, float* qr, float* qs, float* qg,
             float* ni, float* nr, float* t, const float* p, const float* dz,
             float* ppt, int nthreads);

// mp_thompson with is_aerosol_aware = .true. (M:28) and mp_gt_driver's handling of the aerosol arrays around it (M:950-956,
// M:999-1007), COL_FASTEST arrays a[k*ncol+col]: nc, nwfa, nifa INOUT, w IN, nwfa2d [ncol] or NULL.
int kor_step_aero(const kor_handle*, long ncol, int nz, float dt, float* qv, float* qc, float* qi, float* qr, float* qs,
                  float* qg, float* ni, float* nr, float* t, float* nc, float* nwfa, float* nifa, const float* p,
                  const float* w, const float* dz, const float* nwfa2d, float* ppt, int nthreads);
// M:4354-4390 Eff_aero, M:4720-4756 iceDeMott, M:4764-4789 iceKoop, M:4451-4526 activ_ncloud
float kor_eff_aero(float D, float Da, float visc, float rhoa, float temp, char species);
float kor_ice_demott(float tempc, float rho, float nifa);
float kor_ice_koop(float temp, float qv, float qvs, float naero, float dt);
float kor_activ_ncloud(float Tt, float Ww, float NCCN);

// I:28-246 mphys_thompson09_interfacen (gather, mp_thompson per column, tendencies back) without
// save_dg.  KiD (k,i) arrays a[i*nz+k]; hyd planes: qc, qr, nr, qi, ni, qs, qg; ppt [4][nx].
int kor_kid_interface(const kor_handle*, long nx, int nz, float dt, float p0, float r_on_cp,
                      const float* theta, const float* dtheta_adv, const float* dtheta_div,
                      const float* exner, const float* qv, const float* dqv_adv, const float* dqv_div,
                      const float* dz, const float* const* hyd, const float* const* dhyd_adv,
                      const float* const* dhyd_div, float* dtheta_mphys, float* dqv_mphys,
                      float* const* dhyd_mphys, float* ppt);

// M:4834-4935 calc_effectRad, one column; re_* INOUT (preset by the caller, M:1112-1114); nc1d may be NULL.
int kor_calc_effect_rad(const kor_handle*, int nz, const float* t1d, const float* p1d, const float* qv1d,
                        const float* qc1d, const float* nc1d, const float* qi1d, const float* ni1d, const float* qs1d,
                        float* re_qc1d, float* re_qi1d, float* re_qs1d);

int kor_calc_effect_rad_aero(const kor_handle*, int nz, const float* t1d, const float* p1d, const float* qv1d,
                             const float* qc1d, const float* nc1d, const float* qi1d, const float* ni1d, const float* qs1d,
                             float* re_qc1d, float* re_qi1d, float* re_qs1d);   // is_aerosol_aware = .true.: nc1d is read (M:4874)

// M:806-1143 mp_gt_driver over ni x nj columns; 3-D arrays a[i + ni*(k + nk*j)], 2-D a[i + ni*j]; the snow / graupel
// accumulators and the three radii may be NULL.
int kor_mp_gt_driver(const kor_handle*, int ni, int nk, int nj, float dt, float* qv, float* qc, float* qr, float* qi,
                     float* qs, float* qg, float* ni_, float* nr, float* th, const float* pii, const float* p,
                     const float* dz, float* rainnc, float* rainncv, float* snownc, float* snowncv, float* graupelnc,
                     float* graupelncv, float* sr, float* re_cloud, float* re_ice, float* re_snow);

const char* kor_rate_names(void);   // comma-separated, 36 names (M:2963-3120)

// M:4598-4717 helpers, exposed for known-answer tests
float kor_rslf(float p, float t);
float kor_rsif(float p, float t);
float kor_gammln(float x);
float kor_wgamma(float x);
float kor_gammp(float a, float x);
int   kor_decade_index(float x, int n2, int ntb);   // M:1762-1774 pattern
int   kor_decade_index_d(double x, int n2, int ntb);   // M:1824-1833 (f64 argument)

// array forms of the helpers above (out[i] = f(x[i], ...), i < n): one call for a sweep of millions of points
void kor_rslf_array(const float* p, const float* t, float* out, long n);
void kor_rsif_array(const float* p, const float* t, float* out, long n);
void kor_decade_index_array(const float* x, int n2, int ntb, int* out, long n);
void kor_decade_index_d_array(const double* x, int n2, int ntb, int* out, long n);
void kor_eff_aero_array(const float* D, const float* Da, const float* visc, const float* rhoa, const float* temp,
                        char species, float* out, long n);
void kor_ice_demott_array(const float* tempc, const float* rho, const float* nifa, float* out, long n);
void kor_ice_koop_array(const float* temp, const float* qv, const float* qvs, const float* naero, const float* dt,
                        float* out, long n);
void kor_activ_ncloud_array(const float* Tt, const float* Ww, const float* NCCN, float* out, long n);

#ifdef __cplusplus
}
#endif
