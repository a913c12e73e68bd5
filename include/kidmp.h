/* kidmp.h - C ABI of the B200-native Thompson microphysics step for the KiD kinematic driver.
 *
 * Reference files (read-only upstream):
 *   M: = module_mp_thompson09n.f90      I: = mphys_thompson09n.f90
 * The Fortran host keeps `module mphys_thompson09n` / `mphys_thompson09_interfacen` (I:9, I:28) and
 * binds these entry points through iso_c_binding (kid_b200/fortran/mphys_thompson09n.f90,
 * INTEGRATION.md).  Plain pointers and sizes only; no C++/torch types cross this boundary.
 *
 * Conventions
 *   - all reals are IEEE f32 (the reference's default REAL), sums returned by kidmp_diag are f64
 *   - nine prognostic fields, always in this order (M:1168-1170 minus the aerosol/nc inputs):
 *       0 qv  1 qc  2 qi  3 qr  4 qs  5 qg  6 ni  7 nr  8 t      (t = temperature in K, I:60)
 *   - layouts of a field holding ncol columns of nz levels (level 0 = lowest, kts):
 *       KIDMP_K_FASTEST   a[col*nz + k]   KiD's (k,i) arrays (I:33-35, column_variables)
 *       KIDMP_COL_FASTEST a[k*ncol + col] WRF/MPAS (i,k,j) order (M:806-853); the device layout
 *   - precipitation ppt is [4][ncol]: 0 rain, 1 ice, 2 snow, 3 graupel  (I:162-177); it is
 *     OVERWRITTEN with this step's amounts (the reference zeroes its accumulators per call, I:55-58)
 *   - every function returns 0 on success, non-zero on error; kidmp_last_error() has the text.
 *     Nothing here prints, exits or throws.  No CPU fallback exists: without a CUDA device
 *     kidmp_init fails.
 */
#ifndef KIDMP_H
#define KIDMP_H
#ifdef __cplusplus
extern "C" {
#endif

#define KIDMP_NFIELDS 9
#define KIDMP_K_FASTEST 0
#define KIDMP_COL_FASTEST 1
#define KIDMP_NDIAG 8
#define KIDMP_NRATES 36

typedef struct kidmp_handle kidmp_handle;

/* Host switches read by the reference at init (M:20-22, M:381, M:773) */
typedef struct kidmp_config {
  float set_Nc;            /* namelists:set_Nc, cloud droplets per cm^3 (M:381)                  */
  int iiwarm;              /* namelists:iiwarm, warm-rain only (M:773, M:1545, M:1749 ...)       */
  int l_sediment;          /* switches:l_sediment, gates ice/snow/graupel fall (M:3449,3506,3555)*/
  int wp_double;           /* kind of DFLOAT() in the bin grids (M:8, M:616); 0 = f32 (default)  */
  int device;              /* CUDA device ordinal                                                */
  int reuse_tables;        /* switches:l_reuse_thompson_lookup (M:3720): read table_cache_path   */
  const char* table_cache_path; /* binary cache of the lookup tables, may be NULL (M:3710-3728)  */
  int ndev;                /* 0 or 1: one GPU (`device`, or device_ids[0] when ndev == 1 and device_ids is set);
                              > 1: one handle over ndev GPUs of this process, columns cut into ndev contiguous ranges */
  const int* device_ids;   /* ndev CUDA device ordinals, NULL = 0 .. ndev-1                       */
} kidmp_config;

/* replaces thompson_init (M:374-797): constants on the host, every lookup table built by CUDA
 * kernels on the device (or read from the binary cache). */
int kidmp_init(const kidmp_config* cfg, kidmp_handle** out);
int kidmp_finalize(kidmp_handle* h);
const char* kidmp_last_error(const kidmp_handle* h);   /* h may be NULL: last init error */
const char* kidmp_build_id(void);                      /* hash of the sources and flags the library was built from */
double kidmp_table_build_ms(const kidmp_handle* h);    /* device time of the table-build kernels */

/* lookup tables and init constants by their reference names ("tcg_racg", "t_Efrw", "crg", ...),
 * Fortran column-major order (M:386-423).  For parity tests and the table cache. */
long kidmp_table_size(const kidmp_handle* h, const char* name);
int kidmp_get_table(const kidmp_handle* h, const char* name, double* out, long n);
int kidmp_save_tables(const kidmp_handle* h, const char* path);

/* KiD's own lookup-table cache (M:3710-3728, M:3823-3828, M:3857-3894, M:4066-4077): list-directed text, the six rain-graupel
 * tables in run_data/racg_thompson09.data and the twelve rain-snow tables in run_data/racs_thompson09.data, each written as one
 * `write(unit,*) table` record in Fortran element order.  The writer prints 17 significant digits (what gfortran prints for
 * REAL(8), exact on re-reading); the reader takes anything `read(unit,*)` takes (blanks, commas, line breaks, D/E exponents,
 * r*c repeats).  With these the Fortran reference and this library can run on the same tables. */
int kidmp_write_kid_cache(const kidmp_handle* h, const char* racg_path, const char* racs_path);
int kidmp_read_kid_cache(kidmp_handle* h, const char* racg_path, const char* racs_path);

/* exact single-column twin of mp_thompson (M:1156-1162): host arrays of nz, in place; ppt4 is
 * rain, ice, snow, graupel and is ACCUMULATED into like the reference's INOUT scalars (M:1172). */
int kidmp_column(kidmp_handle* h, int nz, float dt,
                 float* qv, float* qc, float* qi, float* qr, float* qs, float* qg,
                 float* ni, float* nr, float* t,
                 const float* p, const float* dz, float* ppt4);

/* the body of `do i = 1, nx` (I:54-246) for ncol independent columns: host arrays in, host
 * arrays out (H2D, kernels, D2H inside the call).  dz is one shared vector of nz (I:63).
 * Large KIDMP_COL_FASTEST domains flow through the device in chunks on three streams, unless process rates are kept (a
 * buffer of kidmp_set_rates_buffer, or kidmp_enable_rates): then the whole domain goes through the resident state, the rates
 * are those of the whole domain, and nothing travels back by the zero-copy path below.  When the nine field arrays are
 * PINNED host memory (cudaHostAlloc / cudaHostRegister), only the columns the step changed travel back - a clear-sky column
 * is returned bit for bit by the reference too (M:1540) - written by a kernel straight into the host arrays.
 * ncol = 0 (here, in kidmp_step_device and as kidmp_kid_columns::nx) is the empty loop of I:54: success, nothing touched. */
int kidmp_step(kidmp_handle* h, long ncol, int nz, float dt, int layout,
               float* const fields[KIDMP_NFIELDS], const float* p, const float* dz, float* ppt);

/* device-resident state: upload once, step many times, download when needed.  One resident state per handle: the entry
 * points that take HOST arrays of another size (kidmp_step and kidmp_step_aero below the pipeline threshold, kidmp_column,
 * kidmp_kid_interface, kidmp_mp_gt_driver) re-allocate it.  Calls on one handle are serialised by the caller; a step enqueued on a caller's
 * stream (kidmp_step_device) is ordered against kidmp_diag and the next step of the same handle by an event. */
int kidmp_state_alloc(kidmp_handle* h, long ncol, int nz);
int kidmp_upload(kidmp_handle* h, int layout, const float* const fields[KIDMP_NFIELDS],
                 const float* p, const float* dz);
int kidmp_step_resident(kidmp_handle* h, float dt);
int kidmp_download(kidmp_handle* h, int layout, float* const fields[KIDMP_NFIELDS], float* ppt);

/* same step on caller-owned DEVICE buffers in KIDMP_COL_FASTEST layout, enqueued on `stream`
 * (a cudaStream_t passed as void*; NULL = the handle's stream).  Does not synchronise. */
int kidmp_step_device(kidmp_handle* h, long ncol, int nz, float dt,
                      float* const d_fields[KIDMP_NFIELDS], const float* d_p, const float* d_dz,
                      float* d_ppt, void* stream);

/* Per-column cloud droplet number of the plain scheme (is_aerosol_aware = .false.).  The reference has one droplet number per
 * run, Nt_c = set_Nc * 1e6 (M:381); these entries take one set_Nc [cm^-3] per column instead: column c is stepped with
 * Nt_c = set_nc[c] * 1e6f (f32, as M:381), so it comes out bit for bit as a handle made with set_Nc = set_nc[c] would step it
 * (set_Nc feeds nothing but Nt_c, and the lookup tables do not depend on it).  One handle, one table build and one launch
 * sequence serve a domain of mixed droplet numbers (land and ocean) or a sweep of set_Nc values.  Every value must be finite
 * and > 0, as kidmp_init requires of set_Nc.  set_nc == NULL: the handle's set_Nc, exactly as the entry without _nc.
 *   kidmp_step_nc          kidmp_step with set_nc[ncol] on the host.  Every value is checked before anything is copied or
 *                          launched; a bad one fails the call and leaves every array as it was.  All of kidmp_step's paths:
 *                          both layouts, the chunk pipeline (each chunk takes its slice), multi-device handles (each device
 *                          its column range), the handle's process-rate buffer.
 *   kidmp_step_device_nc   kidmp_step_device with d_set_nc[ncol] on the device, enqueued on `stream`.  The values are not
 *                          checked (as no other device input is); they are read when the step runs, also when the step is
 *                          replayed from a captured CUDA graph. */
int kidmp_step_nc(kidmp_handle* h, long ncol, int nz, float dt, int layout, float* const fields[KIDMP_NFIELDS],
                  const float* p, const float* dz, const float* set_nc, float* ppt);
int kidmp_step_device_nc(kidmp_handle* h, long ncol, int nz, float dt, float* const d_fields[KIDMP_NFIELDS],
                         const float* d_p, const float* d_dz, const float* d_set_nc, float* d_ppt, void* stream);

/* Aerosol-aware step (is_aerosol_aware = .true., M:28, with dustyIce = homogIce = .true., M:30-31): the second half of
 * SURVEY.md section 8f-4.  Device pointers like kidmp_step_device; in addition the cloud droplet number nc and the numbers
 * of water-friendly and ice-friendly aerosols nwfa, nifa [kg^-1] are prognostic (INOUT, [nz][ncol]; mp_gt_driver's
 * nc / nwfa / nifa, M:950-956, M:1003-1007), w is the vertical velocity [m s^-1] that feeds the droplet activation
 * (activ_ncloud, M:2797), d_nwfa2d [ncol] (or NULL) the surface aerosol emission added to the lowest level after the step
 * (M:1001).  Rain, snow and graupel scavenge aerosols (Eff_aero, M:1729-1740, M:1938-1959), ice nucleates on dust (iceDeMott,
 * M:2092) and freezes homogeneously from deliquesced aerosols (iceKoop, M:2104-2111), evaporating cloud loses the droplets
 * smaller than D-star (table_dropEvap, M:2804-2851).  The evaporation table is made by the first such step.  No process-rate
 * buffer in this mode. */
int kidmp_step_device_aero(kidmp_handle* h, long ncol, int nz, float dt, float* const d_fields[KIDMP_NFIELDS], float* d_nc,
                           float* d_nwfa, float* d_nifa, const float* d_p, const float* d_w, const float* d_dz,
                           const float* d_nwfa2d, float* d_ppt, void* stream);
/* The same aerosol-aware step on HOST arrays, in place: kidmp_step with the aerosol switch on.  nc, nwfa, nifa (INOUT) and w (IN)
 * are laid out like the fields ([nz][ncol] for KIDMP_COL_FASTEST, (k,i) for KIDMP_K_FASTEST); nwfa2d is [ncol] in both layouts,
 * or NULL; ppt [4][ncol] is overwritten.  Every column comes out bit for bit as kidmp_step_device_aero makes it from device copies
 * of the same inputs (the nine fields, nc, nwfa, nifa, ppt), and kidmp_diag counts it the same way.  Every path of kidmp_step:
 * small domains and KIDMP_K_FASTEST through the resident state, large KIDMP_COL_FASTEST domains through the chunk pipeline (each
 * chunk carries the four aerosol planes and its slice of nwfa2d), only the changed columns back when the twelve INOUT arrays
 * are pinned (with nwfa2d the lowest nwfa level comes back for every column: the emission changes it everywhere), multi-device
 * handles (each device its column range).  A NULL array other than nwfa2d and ppt, nz outside [2, 256], dt <= 0, or process
 * rates kept or a rate buffer set (on any device of the handle) fail the call before anything is copied or launched, every
 * array left as it was.  ncol = 0: success, nothing touched. */
int kidmp_step_aero(kidmp_handle* h, long ncol, int nz, float dt, int layout, float* const fields[KIDMP_NFIELDS], float* nc,
                    float* nwfa, float* nifa, const float* p, const float* w, const float* dz, const float* nwfa2d, float* ppt);

/* optional per-level process-rate buffer (the 36 save_dg rates of M:2963-3120): device buffer
 * [36][nz][ncol] f32, NULL switches it off (default).  Names: kidmp_rate_names(). */
int kidmp_set_rates_buffer(kidmp_handle* h, float* d_rates);
const char* kidmp_rate_names(void);
/* The same rates for a HOST caller (the Fortran shim's save_dg calls, M:2963-3120): kidmp_enable_rates(h, 1) makes the handle
 * keep its own [36][nz][ncol] buffer for the resident state (36*nz*ncol floats of device memory).  Every entry point that steps
 * the resident state fills it, zero where no process ran: kidmp_step and kidmp_step_nc (with rates kept every kidmp_step
 * domain goes through the resident state, see kidmp_step), kidmp_step_resident, kidmp_column, kidmp_kid_interface and the
 * kidmp_mp_gt_driver entries without aerosols.  kidmp_get_rates copies the rates of the handle's LAST step to `rates`:
 * [36][nz][ncol] for KIDMP_COL_FASTEST, [36][ncol][nz] (KiD's (k,i) order, plane by plane) for KIDMP_K_FASTEST, with ncol
 * and nz of that step.  It fails when that step wrote no rates into this buffer (kidmp_step_device, a step with a buffer of
 * kidmp_set_rates_buffer, a failed step), before the first step after kidmp_enable_rates or kidmp_state_alloc, and after
 * kidmp_enable_rates(h, 0).  The aerosol-aware steps refuse to run while rates are kept or a buffer is set.
 * A multi-device handle returns KIDMP_K_FASTEST only, laid out by its last stepping call: [36][ncol][nz] of that call's columns,
 * whether it cut them over the devices or ran on the first device alone (kidmp_column, the WRF tiles, kidmp_kid_interface
 * with nx below the device count). */
int kidmp_enable_rates(kidmp_handle* h, int on);
int kidmp_get_rates(kidmp_handle* h, int layout, float* rates);

/* domain sums accumulated by the step since the last call (f64): 0 rain 1 ice 2 snow 3 graupel surface precipitation
 * [sum over columns of ppt], 4 liquid water path 5 ice water path [kg m^-2 summed over columns], 6 active columns,
 * 7 columns processed.  A handle over several devices (ndev > 1) returns the sums over ALL its devices: the per-device
 * sums are all-reduced with NCCL (ncclAllReduce of 8 f64 on a single-process communicator over NVLink), the device twin
 * of the column means of I:255-275.  With one process per GPU (torchrun) the host all-reduces the 8 numbers itself. */
int kidmp_diag(kidmp_handle* h, double out[KIDMP_NDIAG]);

/* The KiD-facing entry: everything mphys_thompson09_interfacen does for its nx columns except
 * save_dg (I:54-246).  Arrays are KiD's column_variables in (k,i) order, a[i*nz + k]:
 * state + (advective + divergence tendency)*dt goes in, theta -> T and exner -> p (I:59-97), the
 * column step runs, and the new state comes back as microphysics tendencies (I:198-245).
 * hyd / dhyd_* hold one plane per prognostic moment of hydrometeors(k,i,ih)%moments(1,im), in the
 * order qc (ih=1,im=1), qr (2,1), nr (2,2), qi (3,1), ni (3,2), qs (4,1), qg (5,1); planes 3..6 may
 * be NULL when iiwarm.  ppt is [4][nx]: pptrain_2d, pptice_2d, pptsnow_2d, pptgraul_2d (I:183-186). */
typedef struct kidmp_kid_columns {
  long nx; int nz;
  const float *theta, *dtheta_adv, *dtheta_div, *exner, *qv, *dqv_adv, *dqv_div;
  const float *dz;                       /* dz(k), nz values (I:63) */
  const float *hyd[7], *dhyd_adv[7], *dhyd_div[7];
  float *dtheta_mphys, *dqv_mphys, *dhyd_mphys[7];
  float *ppt;
} kidmp_kid_columns;
int kidmp_kid_interface(kidmp_handle* h, const kidmp_kid_columns* c, float dt, float p0, float r_on_cp);

/* The WRF / MPAS-facing entry: what mp_gt_driver (M:806-1143) does for ni x nj columns of nk levels.
 * ni, nk, nj are the MEMORY dimensions of the arrays.  3-D arrays are WRF's (i,k,j) order, a[i + ni*(k + nk*j)]; 2-D arrays
 * are (i,j), a[i + ni*j].  kidmp_mp_gt_driver steps the whole box; a host whose arrays carry halo points or spare levels
 * (WRF and MPAS allocate kme = kte + 1) names the cells to step with kidmp_mp_gt_driver_tile below.  INOUT: the nine
 * prognostic fields with potential temperature `th` (T = th*pii goes into the step, th = T/pii comes back, M:941,
 * M:1022); IN: pii (Exner function), p, dz (per-column layer depths, M:944).  RAINNC / SNOWNC / GRAUPELNC are
 * accumulated, RAINNCV / SNOWNCV / GRAUPELNCV / SR overwritten (M:991-1003); the snow and graupel pairs may be NULL
 * (OPTIONAL in the reference).  re_cloud, re_ice, re_snow receive the effective radii of calc_effectRad (M:4834-4935)
 * clamped as at M:1118-1122 when all three are non-NULL (has_reqc, has_reqi, has_reqs), else they are not touched.
 * w, nc, nwfa, nifa, nwfa2d, refl_10cm and the WRF_CHEM arguments are not part of this ABI: they are only read or
 * written under is_aerosol_aware / WRF_CHEM / do_radar_ref, none of which exists in the KiD build of the scheme. */
typedef struct kidmp_wrf_fields {
  int ni, nk, nj;
  float *qv, *qc, *qr, *qi, *qs, *qg, *ni_, *nr, *th;    /* (i,k,j) INOUT, argument order of M:806 (ni_ = ni) */
  const float *pii, *p, *dz;                               /* (i,k,j) IN                                      */
  float *rainnc, *rainncv, *sr;                            /* (i,j)                                           */
  float *snownc, *snowncv, *graupelnc, *graupelncv;        /* (i,j), optional                                 */
  float *re_cloud, *re_ice, *re_snow;                      /* (i,k,j), optional                               */
} kidmp_wrf_fields;
int kidmp_mp_gt_driver(kidmp_handle* h, const kidmp_wrf_fields* w, float dt_in);
/* the same entry with is_aerosol_aware = .true. (M:28): mp_gt_driver's optional arguments nc, nwfa, nifa (i,k,j, INOUT), the
 * vertical velocity w (i,k,j, IN) and the surface aerosol emission nwfa2d (i,j, IN, may be NULL) (M:807-832, M:950-956,
 * M:999-1007); re_cloud then follows the prognostic droplet number (M:4874).  See kidmp_step_device_aero. */
typedef struct kidmp_wrf_aerosols {
  float *nc, *nwfa, *nifa;
  const float* w;
  const float* nwfa2d;
} kidmp_wrf_aerosols;
int kidmp_mp_gt_driver_aero(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_aerosols* ae, float dt_in);

/* The same step for one tile inside the memory box of kidmp_wrf_fields, in place: w->ni, w->nk, w->nj are the memory
 * dimensions ime-ims+1, kme-kms+1, jme-jms+1, and the tile is given by 0-based offsets and extents,
 *   i0 = its-ims, ni = ite-its+1,  k0 = kts-kms, nk = kte-kts+1,  j0 = jts-jms, nj = jte-jts+1.
 * Tile cell (i,k,j) is memory cell (i0+i, k0+k, j0+j); its 2-D cell is (i0+i, j0+j).  The call reads and writes only cells
 * of the tile box: halo points, the spare top level and every other cell of every array are neither read nor written, so
 * the tiles of one patch may run at the same time (one handle each).  A tile outside the memory box, nk < 2 or an empty
 * extent is rejected (non-zero return, kidmp_last_error) before anything is copied or launched.  ae == NULL is
 * is_aerosol_aware = .false. (kidmp_mp_gt_driver), else kidmp_mp_gt_driver_aero.  Everything else as those two:
 * radii only with all three re_* given, optional snow and graupel accumulators, the handle's process-rate buffer on
 * the non-aerosol path, a multi-device handle steps the tile on its first device.
 * kidmp_mp_gt_driver_tile takes HOST arrays and returns when they hold the result; only the tile rows travel.
 * kidmp_mp_gt_driver_tile_device takes DEVICE arrays of the handle's GPU and is enqueued on `stream` (a cudaStream_t passed
 * as void*; NULL = the handle's stream) without synchronising; the step runs on the handle's resident state, ordered against
 * kidmp_diag and the next call by an event.  It needs a single-device handle. */
typedef struct kidmp_wrf_tile { int i0, ni, k0, nk, j0, nj; } kidmp_wrf_tile;
int kidmp_mp_gt_driver_tile(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t, const kidmp_wrf_aerosols* ae,
                            float dt_in);
int kidmp_mp_gt_driver_tile_device(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t,
                                   const kidmp_wrf_aerosols* ae, float dt_in, void* stream);
/* The plain-scheme tile entries with a droplet number per column (see kidmp_step_nc): set_nc2d is an (i,j) array of the memory
 * box, read only at the tile's 2-D cells (i0+i, j0+j); column (i,j) is stepped with Nt_c = set_nc2d(i0+i, j0+j) * 1e6f, and
 * re_cloud follows it.  kidmp_mp_gt_driver_tile_nc takes it on the host and checks every value it reads (finite, > 0) before
 * anything is copied or launched; kidmp_mp_gt_driver_tile_device_nc takes it on the device, unchecked.  NULL: the handle's
 * set_Nc.  Otherwise as kidmp_mp_gt_driver_tile / _device with ae = NULL. */
int kidmp_mp_gt_driver_tile_nc(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t, const float* set_nc2d,
                               float dt_in);
int kidmp_mp_gt_driver_tile_device_nc(kidmp_handle* h, const kidmp_wrf_fields* w, const kidmp_wrf_tile* t,
                                      const float* d_set_nc2d, float dt_in, void* stream);

/* Tuning knobs; results do not depend on them.
 * "chunk": columns per launch of the step kernels (default 1 048 576, or the KIDMP_CHUNK environment variable): the work
 * buffers (128-byte hand-off records, cell lists) are sized for one chunk, whatever the size of the domain.
 * "timing": 1 = run the kernels of a launch one after the other with an event after each (kidmp_last_kernel_ms), 2 = the
 *   normal schedule (second stream in use) with the same events on the main stream, 0 = normal.
 * "graphs": 1 (default, KIDMP_GRAPHS) = the launches of a step (up to 64 chunks) are captured once in a CUDA graph (a cache of eight) and replayed
 *   while the arguments stay the same (KiD's own cases of 1 to 14 400 columns are launch-bound; the 1 048 576-column step loses its
 *   launch gaps); 0 = plain launches.
 * "simple": 1 (default) = a column that holds no graupel and in which no fall speed can cross the thinnest layer in one step
 *   (every sub-step count of M:3242 is 0 or 1) skips the column kernel that settles those counts; 0 = every cloudy column
 *   goes through it.  KIDMP_SIMPLE.
 * "classes": 1 (default) = every busy cell goes to the cell kernel specialised for its species set and temperature class;
 *   0 = every busy cell goes to the general one.  The specialised kernels compute the same bits (tests/test_regimes.py): this
 *   is their reference, not a tuning choice.
 * Any other name is refused ("unknown option").
 * Environment only: KIDMP_PIPE_CHUNK (columns per chunk of kidmp_step's host pipeline; a smaller "chunk" takes its place,
 *   so that every pipeline chunk is one launch), KIDMP_ZEROCOPY=0 (copy whole chunks back instead of writing the changed
 *   columns into pinned host arrays), KIDMP_PIPE_TRACE=1 (device timeline of every chunk of kidmp_step on stderr). */
int kidmp_set_option(kidmp_handle* h, const char* name, int value);

/* Multi-device handles (kidmp_config::ndev > 1).  kidmp_step, kidmp_kid_interface and the resident-state calls cut the
 * host arrays into one contiguous column range per device (columns are independent, I:54: no exchange on the data path) and
 * run the devices side by side; results are bit-identical to a single-device handle, column by column.  So does kidmp_step_aero:
 * every device builds its own drop-evaporation table on its first aerosol-aware step.  kidmp_column and
 * kidmp_mp_gt_driver[_aero,_tile] run on the first device.  The entry points that take or return DEVICE pointers
 * (kidmp_step_device, kidmp_mp_gt_driver_tile_device, kidmp_set_rates_buffer, kidmp_device_state, kidmp_stream) need a
 * single-device handle.  NCCL (libnccl.so.2, or the file
 * named by the KIDMP_NCCL_LIB environment variable) is loaded when such a handle is created, not before. */
int kidmp_num_devices(const kidmp_handle* h);

/* bookkeeping for benchmarks */
long kidmp_gpu_launches(const kidmp_handle* h);         /* kernels launched so far          */
/* counts of the last launch of the step kernels in the last step (waits for it): 0 cloudy columns, 1 busy
 * cells, 2-5 busy cells of the warm / ice / mixed-without-rain / full cell kernels, 6 columns with sedimentation sub-steps,
 * 7 whether the last kidmp_step or kidmp_step_aero returned only the changed columns (pinned host arrays, see kidmp_step) */
int kidmp_step_stats(kidmp_handle* h, long out[8]);
/* per-kernel device times of the last launch of the step kernels, after kidmp_set_option(h, "timing", 1): in that mode the
 * kernels of a launch run one after the other on one stream with a CUDA event after each group (normally two of them run
 * beside others on a second stream), so the sum is a little above the time of a normal step.  Names, comma-separated, in
 * the order of the values: kidmp_kernel_names(). */
const char* kidmp_kernel_names(void);
int kidmp_last_kernel_ms(kidmp_handle* h, float* out, int n);
int kidmp_sync(kidmp_handle* h);                        /* wait for the handle's stream     */
int kidmp_last_step_ms(kidmp_handle* h, float* step_ms);  /* CUDA events around the last step */
int kidmp_tables_from_cache(const kidmp_handle* h);     /* 1 if init read the table cache   */
void* kidmp_stream(kidmp_handle* h);                    /* the handle's cudaStream_t        */
/* device pointers of the resident state ([nz][ncol] each), for callers that fill it on the device */
int kidmp_device_state(kidmp_handle* h, float* d_fields[KIDMP_NFIELDS], float** d_p, float** d_dz, float** d_ppt);

#ifdef __cplusplus
}
#endif
#endif
